#!/usr/bin/env python
"""bench.py — DIAL-MPC sampling core on B200.

One "step" = one MPC planning step of a BASELINE.json config: shift + Ndiffuse x reverse_once
(sample -> spline -> batched full-order rollout -> reward -> softmax update).  The headline is
configs[1] (unitree_go2_seq_jump, Nsample=2048 per GPU, Hsample=25, Hnode=5, Ndiffuse=4);
`--config i` selects another one, and the default run appends a compact block for every other
single-GPU config (and, at --gpus 8, configs[4] = 65536 samples over 8 GPUs).
Metric: sample-steps/s = Ndiffuse * Nsample_total * Hsample / seconds per step.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # CPU restatement (oracle) on the host cores
"""
from __future__ import annotations

import os

# the CPU arms run one process per core: BLAS / OpenMP pools inside each would oversubscribe the
# host (round 1: 128 procs x BLAS threads -> 5.9x spread between boxes).  Must precede `import numpy`.
for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
    os.environ[_k] = "1"

import argparse  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from baseline_configs import BASELINE, ENV_CFG, dial_config, product_env  # noqa: E402

METRIC = "sample-steps/s (Nsample*Hsample/wall-s) per MPC reverse_once, Go2"


def usable_cores() -> int:
    """Logical CPUs in this process's affinity mask (the CPU arms then look for the fastest thread
    count at or below it: hyper-threads and other tenants make the full count a poor choice)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return n


def cpu_quota():
    """cgroup CPU quota in CPUs (None: unlimited).  Reported, not enforced here: CFS throttles per
    100 ms period, so one reverse_once (< 1 s of CPU) bursts over every core of the box even under
    a 16-CPU quota (measured: 64 threads = 55x one core); a sustained loop would be held to it."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else int(q) / int(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            return q / per if q > 0 else None
        except Exception:
            return None


# --------------------------------------------------------------------------------------------
# CPU arms: the oracle (CPU restatement, NOT reference JAX) on the host cores.
#   kind "port"     fp64 NumPy oracle (oracle/*.py), batched over the rows of one worker
#   kind "port-c"   fp32 C port of the per-sample step (oracle/c), one sample at a time
# Both roll ONE reverse_once of the chosen config: its Nsample+1 rows are split over the host cores
# (NumPy oracle: pinned single-threaded processes; C port: one process, OpenMP threads with dynamic
# scheduling over the rows), the softmax update runs once on the gathered rewards.
# --------------------------------------------------------------------------------------------
_BARRIER = None     # multiprocessing.Barrier inherited by the forked workers
LAST_THREADS = 1    # threads (C port) / processes (NumPy oracle) the last cpu_reverse_once ran fastest with


def _cpu_worker(args):
    ci, rows_lo, rows_hi, core, kind, seed, n_calls, threads = args
    barrier = _BARRIER
    if threads <= 1:
        try:
            os.sched_setaffinity(0, {core})
        except (AttributeError, OSError):
            pass
    from oracle.envs_oracle import make_env
    from oracle.planner_oracle import PlannerOracle
    b = BASELINE[ci]
    env = make_env(b["env"], ENV_CFG[b["env"]])
    s = env.reset()
    for _ in range(10):
        s, _, _ = env.step(s, np.zeros((1, env.nu)))
    N, Hs, Hn = b["N"], b["Hs"], b["Hn"]
    pl = PlannerOracle(env, N, Hs, Hn, b["temp"], b["hdf"], b["tdf"])
    rng = np.random.default_rng(seed)
    Y = np.zeros((Hn + 1, env.nu))
    roll = None
    if kind == "port-c":
        from oracle.c_port import CPort
        roll = CPort(env, b).rollout_rews
        roll(s, np.zeros((4 * max(threads, 1), 2, env.nu)), threads=threads)   # spin up the OpenMP pool (untimed)
    t_in = 0.0
    best = float("inf")
    best_threads = threads
    out = None
    if barrier is not None:
        barrier.wait()       # every worker has finished its set-up (NumPy env build, 10 settle steps)
    if roll is not None and threads > 1:
        # the logical CPU count of a shared GPU box says little about the CPUs a slot really gets
        # (hyper-threads, cgroup shares, other tenants): try the thread counts cores, cores/2, ..., cores/16
        # on the same reverse_once and keep the fastest
        eps = rng.standard_normal((N, Hn + 1, env.nu))
        us = pl.node2u(pl.make_Y0s(eps, Y, pl.sigma_control))[rows_lo:rows_hi]
        th = threads
        while th >= max(1, threads // 16):
            for _ in range(n_calls):
                t0 = time.perf_counter()
                rews = roll(s, us, threads=th)
                dt = time.perf_counter() - t0
                if dt < best:
                    best, best_threads = dt, th
            out = rews
            th //= 2
        return best, out, best_threads
    for i in range(n_calls):
        eps = rng.standard_normal((N, Hn + 1, env.nu))        # same eps on every worker (same seed)
        Y0s = pl.make_Y0s(eps, Y, pl.sigma_control * b["tdf"] ** (i % b["Ndiffuse"]))
        us = pl.node2u(Y0s[rows_lo:rows_hi])
        t0 = time.perf_counter()
        if roll is not None:
            rews = roll(s, us, threads=threads)
        else:
            rews = env.rollout(s, us)[0].mean(-1)
        dt = time.perf_counter() - t0
        t_in += dt
        best = min(best, dt)
        out = rews
    # C port: best of the n_calls repetitions of the same reverse_once (thread start-up / scheduler
    # noise of a shared host); NumPy oracle (n_calls = 1): the call itself
    return (best if kind == "port-c" else t_in), out, best_threads


def cpu_reverse_once(ci: int, procs: int, kind: str, n_calls: int = 1, rows_cap=None):
    """One (or n_calls) reverse_once of config ci with its rows split over `procs` pinned workers.
    rows_cap bounds the sample (first rows_cap rows) when the whole config would take too long.
    Returns (sample-steps/s, wall seconds of the slowest worker, rows rolled)."""
    import multiprocessing as mp
    b = BASELINE[ci]
    rows = b["N"] + 1 if rows_cap is None else min(b["N"] + 1, rows_cap)
    procs = max(1, min(procs, rows))
    try:
        cores = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cores = list(range(os.cpu_count() or 1))
    threads = 1
    if kind == "port-c":
        n_calls = max(n_calls, 3)        # best of 3 (see _cpu_worker)
        if procs > 1:
            threads, procs = procs, 1    # the C port is OpenMP-parallel over the rows: one process, `procs` threads
    bounds = np.linspace(0, rows, procs + 1).astype(int)
    jobs = [(ci, int(bounds[i]), int(bounds[i + 1]), cores[i % len(cores)], kind, 0, n_calls, threads) for i in range(procs)]
    global _BARRIER
    _BARRIER = mp.get_context("fork").Barrier(procs)   # timed region = all workers rolling at the same time
    # always in child processes: the workers pin themselves to one core each, and an affinity set
    # in this process would be inherited by every later pool (round-2 bug: 128 workers on one core)
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_cpu_worker, jobs, chunksize=1)
    wall = max(r[0] for r in res)
    rews = np.concatenate([r[1] for r in res])
    global LAST_THREADS
    LAST_THREADS = res[0][2] if kind == "port-c" else procs
    t0 = time.perf_counter()                 # the one softmax on the gathered rewards (negligible)
    lp = (rews - rews[-1]) / rews.std() / b["temp"]
    w = np.exp(lp - lp.max())
    w /= w.sum()
    wall += time.perf_counter() - t0
    per_call = 1 if kind == "port-c" else n_calls
    units = (rows - 1) * b["Hs"] * per_call if rows_cap is None else rows * b["Hs"] * per_call
    return units / wall, wall, rows


def have_c_port() -> bool:
    try:
        from oracle import c_port
        return c_port.available()
    except Exception:
        return False


def run_reference(args):
    """Reference arm for this tier: the CPU restatement of the path on all host cores, SAME config
    (Nsample, Hsample, env) as the own arm; a step = one reverse_once (the own arm's step is
    Ndiffuse of them: the metric is per reverse_once, so the two are comparable)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ci = args.config
    b = BASELINE[ci]
    cores = usable_cores()
    kind = "port-c" if have_c_port() and not args.numpy_oracle else "port"
    for _ in range(1 if args.warmup else 0):
        cpu_reverse_once(ci, cores, kind)
    vals, t_all = [], 0.0
    for _ in range(args.steps):
        v, wall, rows = cpu_reverse_once(ci, cores, kind)
        vals.append(v)
        t_all += wall
    value = float(b["N"] * b["Hs"] * args.steps / t_all)
    used = LAST_THREADS
    what = ("fp32 C port of the per-sample step (oracle/c)" if kind == "port-c" else "fp64 NumPy oracle port")
    sample = (f"one reverse_once of {b['name']} per step: all {b['N']}+1 rows x (Hsample+1)={b['Hs'] + 1} env steps split over "
              f"the host's CPUs (C port: OpenMP over the rows, fastest of {cores}, {cores}/2 ... {cores}/16 threads = {used}; NumPy oracle: pinned "
              f"processes), one softmax; {what}; CPU restatement, not reference JAX")
    line = dict(impl="reference", metric=METRIC, value=value, unit="sample-steps/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * t_all / args.steps,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32" if kind == "port-c" else "f64",
                data="synthetic",
                config=dict(workload=f"{b['name']} (BASELINE configs[{ci}])", Nsample_per_gpu=b["N"], Nsample_total=b["N"],
                            Hsample=b["Hs"], Hnode=b["Hn"], Ndiffuse=b["Ndiffuse"],
                            step="one reverse_once (metric is per reverse_once)"),
                cpu_baseline=dict(value=value, unit="sample-steps/s", cores=used, logical_cpus=cores, cgroup_cpu_quota=cpu_quota(),
                                  kind=kind, sample=sample),
                e2e=dict(value=value, unit="sample-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled every 20 ms from before the warm-up; stop(t0, t1) keeps the samples that
    fall inside the timed region (falls back to the nearest ones if the region is shorter than
    the sampling period)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [t.strip() for t in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.proc.terminate()
        ok = [(t, r) for t, r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        inside = [r for t, r in ok if t0 <= t <= t1 + 0.03]
        where = "timed region"
        if not inside and ok:
            mid = 0.5 * (t0 + t1)
            inside = [r for _, r in sorted(ok, key=lambda tr: abs(tr[0] - mid))[:3]]
            where = "nearest samples (region shorter than the sampling period)"
        sm = [float(r[0]) for r in inside]
        mx = [float(r[1]) for r in inside if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in inside for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm), window=where)


# --------------------------------------------------------------------------------------------
# own arm
# --------------------------------------------------------------------------------------------
def _load_json(*path):
    try:
        return json.load(open(os.path.join(ROOT, *path)))
    except Exception:
        return {}


def issue_roofline(warp_inst_per_step, rows, steps_per_row, t_kernel, sm_mhz, n_sm, probe):
    """Achieved warp instructions per clock and SM (= ncu sm__inst_executed.avg.per_cycle_elapsed) against what
    an SM delivers from code that does not fit its instruction cache: every resident warp receives one
    instruction per `cpi` cycles (profiles/r02_icache_probe.md), so the ceiling is resident warps / cpi —
    14 warps per SM at N = 2048, 1 at N = 128 (the launch policy puts ceil(rows / SMs) <= 16 warps on an SM)."""
    if not (warp_inst_per_step and sm_mhz and t_kernel > 0):
        return None
    ipc = warp_inst_per_step * rows * steps_per_row / (t_kernel * float(sm_mhz) * 1e6 * n_sm)
    per_sm = -(-rows // n_sm)
    waves = -(-per_sm // 16)
    wpc = -(-per_sm // waves)                                  # warps per CTA of the launch policy
    resident = min(rows, n_sm * wpc) / n_sm                    # average over all SMs, like `ipc`
    cpi = (probe.get("cycles_per_instr_per_warp_128KB") or {}).get("14")
    # (below 8 warps per SM the probe's two builds disagree, 2.9 vs 5.7 cycles for a lone warp: no ceiling is claimed)
    ceiling = resident / cpi if (cpi and resident >= 8) else None
    return dict(warp_inst_per_physics_step=warp_inst_per_step, ipc_per_sm=ipc, resident_warps_per_sm=resident,
                cycles_per_instr_per_warp_streaming=cpi, ipc_ceiling_streaming_code=ceiling,
                frac=(ipc / ceiling) if ceiling else None, sm_clock_mhz=float(sm_mhz), sms=n_sm,
                source="instruction count: ncu smsp__inst_executed.sum (profiles/rollout_counts.json); ceiling: "
                       "scripts/probes/icache_probe.cu on this pool's B200 (profiles/r02_icache_probe.json)")


def dump_outputs(out_dir, arrays):
    """One ``<name>.npy`` per output of the timed path (integers and float64 as float64, the rest as
    float32), so that two builds can be compared output for output.  The largest config returns
    well under 1 MB (Nsample+1 rewards, the knots, the bars), so nothing is sampled."""
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        a = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
        a = a.astype(np.float64 if a.dtype.kind in "iu" or a.dtype == np.float64 else np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_config(ci, args, rank, world, local, steps, warmup, sampler=None, full=True, fp32_peak_tf=None,
                   dump_dir=None):
    """Time config ci on this process group.  Returns the JSON fields of the config (rank 0: all
    of them; other ranks: partial).  full=False skips the clocks / cpu arms (secondary blocks).
    dump_dir: rank 0 writes there what the last timed step returned (dump_outputs)."""
    import torch
    import torch.distributed as dist
    from dial_mpc_b200 import random as drandom
    from dial_mpc_b200.core.dial_core import MBDPI

    b = BASELINE[ci]
    cfg = dial_config(ci, world=world)       # weak scaling: b["N"] samples per GPU
    Ntotal = cfg.Nsample
    env = product_env(b["env"])
    mb = MBDPI(cfg, env, rank=rank, world_size=world)
    dev = mb.device
    # synthetic state: reset, then 10 env steps with zero action so contacts are settled
    state = env.reset(drandom.PRNGKey(0))
    for _ in range(10):
        state = env.step(state, torch.zeros(mb.nu, device=dev))
    factors = mb.schedule(cfg.Ndiffuse)
    rng = drandom.PRNGKey(cfg.seed)
    Y = torch.zeros(cfg.Hnode + 1, mb.nu, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # The timed step goes through the public device-resident loop (DeviceLoop -> C ABI dial_mpc_step):
    # shift + Ndiffuse x reverse_once replayed as ONE CUDA graph per rank, the bars of every
    # iteration on a side branch.  Sharded runs without the peer-memory exchange (no CUDA IPC) fall
    # back to the eager MBDPI.reverse_scan with NCCL collectives.
    from dial_mpc_b200.core.dial_core import DeviceLoop
    use_graph = world == 1 or mb.xch
    loop = DeviceLoop(mb, state, rng, Y) if use_graph else None
    carry = {"Y": Y, "rng": rng}

    def mpc_step():
        if use_graph:
            loop.step(cfg.Ndiffuse, env_step=2)
        else:
            carry["rng"], carry["Y"], carry["info"] = mb.reverse_scan(state, carry["rng"], mb.shift(carry["Y"]), factors)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        mpc_step()
    sync_all()
    launches0 = mb.plan.launches
    evs = []
    sync_all()
    xst0 = mb.plan.exchange_status() if (world > 1 and mb.xch) else None
    t_wall0 = time.perf_counter()
    for _ in range(steps):
        flush.zero_()                                   # L2 flush, outside the timed events
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        mpc_step()
        e1.record()
        evs.append((e0, e1))
    sync_all()
    t_wall = time.perf_counter() - t_wall0
    if dump_dir is not None and rank == 0:
        if use_graph:
            outs = dict(Y=loop.Y, rng=loop.rng_host(), **loop.info())
        else:
            outs = dict(Y=carry["Y"], rng=carry["rng"],
                        **{k: v for k, v in carry["info"].items() if k in ("rews", "qbar", "qdbar", "xbar")})
        dump_outputs(dump_dir, outs)
    xwait = None
    if xst0 is not None:
        # device-measured time this rank's update kernels spent waiting for the slowest peer's flag
        # (skew between the GPUs + NVLink latency), per reverse_once: min / mean / max over ranks
        xst1 = mb.plan.exchange_status()
        w_us = ((xst1["update_wait_ns"] - xst0["update_wait_ns"]) & 0xFFFFFFFF) / 1e3 / (steps * cfg.Ndiffuse)
        t = torch.tensor([w_us], device=dev, dtype=torch.float64)
        allw = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allw, t)
        ws = [float(a.item()) for a in allw]
        xwait = dict(min=min(ws), mean=sum(ws) / len(ws), max=max(ws))
    launches = mb.plan.launches - launches0
    clocks = sampler.stop(t_wall0, t_wall0 + t_wall) if (sampler is not None and rank == 0) else None
    t_dev = sum(a.elapsed_time(b_) for a, b_ in evs) / 1e3
    if world > 1:
        t = torch.tensor([t_dev], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev = float(t.item())
    units_per_step = cfg.Ndiffuse * Ntotal * cfg.Hsample
    value = units_per_step * steps / t_dev

    # ---- e2e: the same public call with HOST buffers (pinned): H2D of the state + knots, D2H of the
    # new knots and the plan's reward, every step, inside the timed region -------------------------------
    ps = state.pipeline_state
    h_q, h_v, h_w = (t.cpu().pin_memory() for t in (ps.qpos, ps.qvel, ps.qacc_warmstart))
    h_Y = torch.zeros(cfg.Hnode + 1, mb.nu).pin_memory()
    h_out = torch.empty(cfg.Hnode + 1, mb.nu).pin_memory()
    from dial_mpc_b200.envs.base_env import PipelineState, State
    h2d = sum(t.numel() * 4 for t in (h_q, h_v, h_w, h_Y))
    d2h = h_out.numel() * 4 + 4

    def e2e_step():
        if use_graph:
            b = loop.buf
            b["qpos"].copy_(h_q, non_blocking=True)
            b["qvel"].copy_(h_v, non_blocking=True)
            b["qacc_warmstart"].copy_(h_w, non_blocking=True)
            b["Y"].copy_(h_Y, non_blocking=True)
            loop.step(cfg.Ndiffuse, env_step=2)
            h_out.copy_(b["Y"], non_blocking=True)
            r = float(loop.info()["rews"][-1])           # D2H read of the plan's reward (syncs)
        else:
            d_state = State(PipelineState(h_q.to(dev, non_blocking=True), h_v.to(dev, non_blocking=True),
                                          h_w.to(dev, non_blocking=True)), None, 0.0, 0.0, {}, dict(state.info))
            Yd = mb.shift(h_Y.to(dev, non_blocking=True))
            carry["rng"], Yd, info = mb.reverse_scan(d_state, carry["rng"], Yd, factors)
            h_out.copy_(Yd, non_blocking=True)
            r = float(info["rews"][-1])
        h_Y.copy_(h_out)
        return r

    for _ in range(3):
        e2e_step()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    sync_all()
    t_e2e = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([t_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_e2e = float(t.item())
    e2e_value = units_per_step * steps / t_e2e
    rng = carry["rng"]

    # ---- per-phase device times of one reverse_once (CUDA events between the stages) ---------------
    phases = mb.phase_times(state, drandom.split(rng)[1], Y, factors[0], reps=10)
    if world > 1:
        keys = sorted(phases)
        t = torch.tensor([phases[k] for k in keys], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        phases = {k: float(v) for k, v in zip(keys, t.tolist())}

    # ---- roofline of the dominant kernel (rollout_kernel), timed alone with CUDA events ----------
    m = env.sys
    Y0 = torch.zeros(cfg.Hnode + 1, mb.nu, device=dev)
    key = drandom.split(rng)[1]
    reps = 20 if b["env"] != "allegro_reorient" else 4
    for _ in range(reps // 2):
        mb.plan.reverse_rollout(state, None, key, Y0, mb.sigma_control, mb._rews_local)
    torch.cuda.synchronize()
    batches = []            # median of 5 back-to-back batches (one batch of 20 launches lasts ~15 ms: too short to be
    for _ in range(5):      # immune to whatever the process did just before — r02: 0.80 vs 0.71 ms in one such batch)
        ks, ke = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ks.record()
        for _ in range(reps):
            mb.plan.reverse_rollout(state, None, key, Y0, mb.sigma_control, mb._rews_local)
        ke.record()
        torch.cuda.synchronize()
        batches.append(ks.elapsed_time(ke) / 1e3 / reps)
    t_kernel = sorted(batches)[len(batches) // 2]
    rows, H = mb.Nlocal + 1, cfg.Hsample + 1
    nfr = env._n_frames
    per_rowstep = 4 * (m.nq + m.nv + 3 * (m.nbody - 1))            # q, qd, x.pos written once per env step
    alg_bytes = rows * H * per_rowstep + rows * 4 + (m.nq + 2 * m.nv) * 4
    peaks = _load_json("MEASURED_PEAKS.json")
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_ach = alg_bytes / t_kernel / 1e9
    prof = _load_json("profiles", "rollout_counts.json").get(b["name"], {})
    traffic = prof.get("dram_bytes_per_launch")
    fpp = prof.get("flop_per_physics_step")
    hbm = dict(achieved=hbm_ach, peak=hbm_peak, unit="GB/s", frac=hbm_ach / hbm_peak, traffic=traffic,
               peak_source="MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s", algorithmic_bytes_per_launch=alg_bytes,
               bytes_per_row_step=per_rowstep)
    roofline = dict(kernel="rollout_kernel", kernel_ms=t_kernel * 1e3, kernel_ms_batches=[round(x * 1e3, 4) for x in batches],
                    kernel_share_of_step=cfg.Ndiffuse * t_kernel / (t_dev / steps),
                    physics_steps_per_s=rows * H * nfr / t_kernel, hbm=hbm)
    if fpp and fp32_peak_tf:
        ach_tf = fpp * rows * H * nfr / t_kernel / 1e12
        roofline.update(bound="fp32", achieved=ach_tf, peak=fp32_peak_tf, unit="TFLOP/s", frac=ach_tf / fp32_peak_tf,
                        traffic=traffic, flop_per_physics_step=fpp,
                        peak_source="measured in-run: dial_fp32_peak (independent FFMA chains, full occupancy, CUDA events)",
                        flop_source="ncu thread-instruction counts FADD+FMUL+2*FFMA, profiles/rollout_counts.json",
                        note=("the path has ~140 flop per algorithmic byte (SURVEY.md 8d): bound by fp32 issue / "
                              "dependent-instruction latency, not HBM; the HBM fraction is kept under `hbm`"))
    else:
        roofline.update(bound="hbm", achieved=hbm_ach, peak=hbm_peak, unit="GB/s", frac=hbm_ach / hbm_peak, traffic=traffic,
                        note="no flop count for this config under profiles/: HBM view only (the path is fp32-bound)")
    # What actually binds (DESIGN.md 5): instruction delivery.  The executed path does not fit the SM's
    # instruction caches (~136 KB per env step vs 32 KB), and a B200 SM issues at most `ipc_ceiling` warp
    # instructions per clock from such code — measured with independent FFMA chains (no data stalls at
    # all) by scripts/probes/icache_probe.cu, numbers committed under profiles/r02_icache_probe.json.
    try:
        issue = issue_roofline(prof.get("warp_inst_per_physics_step"), rows, H * nfr, t_kernel,
                               (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz"),
                               torch.cuda.get_device_properties(dev).multi_processor_count,
                               _load_json("profiles", "r02_icache_probe.json"))
    except Exception as e:      # an explanatory block must never cost the bench line
        issue = dict(error=repr(e))
    if issue:
        roofline["issue"] = issue
    out = dict(value=value, ms_per_step=1e3 * t_dev / steps, gpu_launches=int(launches), wall_s_timed_region=t_wall,
               e2e=dict(value=e2e_value, unit="sample-steps/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                        ms_per_step=1e3 * t_e2e / steps),
               roofline=roofline, phases_us_per_reverse_once=phases, exchange_wait_us_per_reverse_once=xwait, clocks=clocks,
               config=dict(workload=f"{b['name']} (BASELINE configs[{ci}])", Nsample_per_gpu=b["N"], Nsample_total=Ntotal,
                           Hsample=b["Hs"], Hnode=b["Hn"], Ndiffuse=b["Ndiffuse"], n_frames=nfr,
                           step=("shift + Ndiffuse x reverse_once (rollout, exchange, update, bars of every iteration) "
                                 + ("as one CUDA graph per rank (DeviceLoop / dial_mpc_step)" if use_graph else "eager (MBDPI.reverse_scan)")),
                           rng="in-kernel Threefry-2x32", l2="256 MiB memset between steps (outside the timed events)",
                           parallelism=f"samples sharded over {world} GPU(s), {mb.exchange_name} of rewards per reverse_once"))
    del loop, mb, flush
    torch.cuda.empty_cache()
    return out


def run_own(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as graft
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        graft.build()
    if world > 1:
        dist.barrier()
    from dial_mpc_b200 import _capi
    tf = _capi.C.c_float(0.0)
    _capi.check(_capi.lib().dial_fp32_peak(2000, _capi.C.byref(tf)))
    fp32_peak = float(tf.value)

    ci = args.config
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    head = measure_config(ci, args, rank, world, local, args.steps, args.warmup, sampler=sampler, fp32_peak_tf=fp32_peak,
                          dump_dir=args.dump_outputs)
    others = {}
    if not args.only:
        todo = [i for i in (0, 1, 2, 3) if i != ci] if world == 1 else []
        if world == 1 and ci != 4:
            todo.append(4)                  # one 8192-sample shard of configs[4]
        if world == 8 and ci != 4:
            todo = [4]                      # the real configs[4]: 65536 samples over 8 GPUs
        for i in todo:
            st = max(3, min(args.steps, 10 if i != 3 else 4))
            r = measure_config(i, args, rank, world, local, st, 3, fp32_peak_tf=fp32_peak)
            keep = {k: r[k] for k in ("value", "ms_per_step", "gpu_launches", "e2e", "roofline", "phases_us_per_reverse_once",
                                      "exchange_wait_us_per_reverse_once", "config")}
            keep.update(steps=st, warmup=3, unit="sample-steps/s")
            if i == 4 and world == 1:
                keep["note"] = "ONE 8192-sample shard of configs[4] on one GPU (the full config needs --gpus 8)"
            others[f"configs[{i}]"] = keep
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- CPU baseline (oracle port) on a bounded sample, rank 0 / N=1 only -------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = usable_cores()
        b = BASELINE[ci]
        kind = "port-c" if have_c_port() else "port"
        cap1 = 256 if kind == "port" else None
        v1, wall1, rows1 = cpu_reverse_once(ci, 1, kind, rows_cap=cap1)
        vall, wall, rows = cpu_reverse_once(ci, cores, kind)
        used = LAST_THREADS
        cpu = dict(value=vall, unit="sample-steps/s", cores=used, logical_cpus=cores, cgroup_cpu_quota=cpu_quota(), kind=kind,
                   sample=(f"one reverse_once of {b['name']}: all {rows} rows x {b['Hs'] + 1} env steps over "
                           + (f"{used} OpenMP threads of one process (fastest of {cores}, {cores}/2 ... {cores}/16 threads, best of 3)"
                              if kind == "port-c" else f"{cores} pinned single-threaded processes")
                           + f"; single core: {v1:.1f} sample-steps/s on {rows1} rows; "
                           + ("fp32 C port of the per-sample step" if kind == "port-c" else "fp64 NumPy oracle")
                           + " — CPU restatement, not reference JAX"),
                   single_core_value=v1, scaling_vs_linear=vall / (v1 * used), wall_s=wall + wall1)
        if kind == "port-c":               # the NumPy oracle beside it (bounded), for continuity with round 1
            vn, walln, rowsn = cpu_reverse_once(ci, cores, "port")
            cpu["numpy_oracle_value"] = vn
            cpu["wall_s"] += walln
    line = dict(metric=METRIC, value=head["value"], unit="sample-steps/s", n_gpus=world, steps=args.steps,
                warmup=max(args.warmup, 3), ms_per_step=head["ms_per_step"], higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", config=head["config"],
                clocks=head["clocks"], e2e=head["e2e"], gpu_launches=head["gpu_launches"],
                wall_s_timed_region=head["wall_s_timed_region"], roofline=head["roofline"],
                phases_us_per_reverse_once=head["phases_us_per_reverse_once"],
                exchange_wait_us_per_reverse_once=head["exchange_wait_us_per_reverse_once"], fp32_peak_tflops_measured=fp32_peak)
    if cpu:
        line["cpu_baseline"] = cpu
    if others:
        line["other_configs"] = others
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(BASELINE), help="BASELINE.json configs[i] (default 1: the headline)")
    ap.add_argument("--only", action="store_true", help="time only --config (no block for the other configs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--numpy-oracle", action="store_true", help="reference arm: NumPy oracle even if the C port is built")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of --config returned (knots Y, rng, rews, qbar, qdbar, xbar) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl own)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
