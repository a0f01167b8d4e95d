"""world_size-2 test of the sharded planner plumbing on CPU (gloo): sample sharding, the one
allgather of per-sample rewards, the mean-row handling and the allreduce of the bars.  The
per-rank compute is the emulated device code (tests/emul) — the NCCL/GPU run of the same host
code is covered by bench.py --gpus N on the GPU box."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.conftest import make_pair


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(rank, world, port, eps, Ybar, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    if world > 1:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from dial_mpc_b200.core.dial_config import DialConfig
    from dial_mpc_b200.core.dial_core import MBDPI
    from dial_mpc_b200.envs.base_env import PipelineState, State
    from tests.emul.emul import EmulPlan
    env, o = make_pair("unitree_go2_walk")
    s = o.reset()
    cfg = DialConfig(env_name="unitree_go2_walk", Nsample=eps.shape[0], Hsample=6, Hnode=3, temp_sample=0.05)
    mb = MBDPI(cfg, env, rank=rank, world_size=world, plan_factory=EmulPlan)
    f = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float32))
    st = State(PipelineState(f(s.qpos[0]), f(s.qvel[0]), f(s.qacc_warmstart[0])), None, 0.0, 0.0, {}, {"step": 0})
    _, Y, info = mb.reverse_once(st, np.array([0, 7], dtype=np.uint32), f(Ybar), mb.sigma_control, eps=f(eps))
    ret[rank] = dict(Y=Y.numpy().copy(), rews=info["rews"].numpy().copy(), qbar=info["qbar"].numpy().copy(),
                     xbar=info["xbar"].numpy().copy())
    if world > 1:
        dist.destroy_process_group()


def test_two_rank_sharding_matches_single_rank():
    rng = np.random.default_rng(0)
    N = 6
    eps = rng.standard_normal((N, 4, 12)).astype(np.float32)
    Ybar = (rng.standard_normal((4, 12)) * 0.3).astype(np.float32)
    single = {}
    _run(0, 1, _free_port(), eps, Ybar, single)
    # a spawned manager: forking this (multi-threaded) process leaves its OpenBLAS thread pool hung, and the
    # next threaded np.linalg call of a later test never returns
    with mp.get_context("spawn").Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_run, args=(2, _free_port(), eps, Ybar, ret), nprocs=2, join=True)
        r0, r1 = ret[0], ret[1]
    s0 = single[0]
    # per-sample rewards do not depend on the shard: bitwise identical
    assert np.array_equal(r0["rews"], s0["rews"]) and np.array_equal(r1["rews"], s0["rews"])
    # every rank holds the same control update; bars agree with the single-rank run
    assert np.array_equal(r0["Y"], r1["Y"])
    assert np.abs(r0["Y"] - s0["Y"]).max() < 1e-6
    assert np.abs(r0["qbar"] - s0["qbar"]).max() < 1e-5 and np.abs(r1["xbar"] - s0["xbar"]).max() < 1e-5
    # and the oracle agrees
    from oracle.planner_oracle import PlannerOracle
    env, o = make_pair("unitree_go2_walk")
    po = PlannerOracle(o, N, 6, 3, 0.05, 0.9, 0.5)
    Yo, io = po.reverse_once(o.reset(), eps.astype(np.float64), Ybar.astype(np.float64), po.sigma_control)
    assert np.abs(s0["rews"] - io["rews"]).max() < 5e-4
    assert np.abs(s0["Y"] - Yo).max() < 5e-3
