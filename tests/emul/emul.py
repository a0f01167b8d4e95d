"""TEST-ONLY python driver of the CPU warp emulator (tests/emul/libdial_emul.so)."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

from dial_mpc_b200 import _capi

_DIR = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_DIR, "libdial_emul.so")


def build(force=False, reward_source=None, defines=()):
    """g++ build of the device code for the lock-step warp emulator.  ``reward_source``: a custom
    reward file (include/dial_custom_reward.h) compiled in, as dial_mpc_b200.custom does with nvcc."""
    srcs = [os.path.join(_DIR, "emul_main.cpp"), os.path.join(_DIR, "warp_emul.h"),
            os.path.join(_DIR, "..", "..", "dial_mpc_b200", "csrc", "dial_device.cuh"),
            os.path.join(_DIR, "..", "..", "dial_mpc_b200", "csrc", "dial_host.h"),
            os.path.join(_DIR, "..", "..", "include", "dial_b200.h")]
    so, extra = _SO, []
    if reward_source is not None:
        reward_source = os.path.abspath(reward_source)
        tag = hashlib.sha256(open(reward_source, "rb").read()).hexdigest()[:12]
        so = os.path.join(_DIR, f"libdial_emul_custom_{tag}.so")
        extra = [f'-DDIAL_CUSTOM_REWARD_FILE="{reward_source}"']
        srcs += [reward_source, os.path.join(_DIR, "..", "..", "include", "dial_custom_reward.h")]
    if defines:
        so = so[:-3] + "_" + "_".join(d.replace("=", "-") for d in defines) + ".so"
        extra = extra + [f"-D{d}" for d in defines]
    if so not in _LIBS or force:
        # content hash, not mtimes: a copied tree need not keep them, and a built tree may be read-only
        h = hashlib.sha256()
        for s in srcs:
            h.update(open(s, "rb").read())
        h.update(" ".join(f"-D{d}" for d in defines).encode())
        digest, side = h.hexdigest(), so + ".sha256"
        if force or not (os.path.exists(so) and os.path.exists(side) and open(side).read().strip() == digest):
            subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", _DIR, "-shared", "-fPIC"] + extra +
                                  ["-o", so, os.path.join(_DIR, "emul_main.cpp")])
            with open(side, "w") as f:
                f.write(digest)
        _LIBS[so] = C.CDLL(so)
    return _LIBS[so]


_LIBS = {}


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def rollout(env, plan_desc, qpos, qvel, warm, step0=0, stage0=0, us=None, eps=None, Ybar=None,
            noise=None, key=(0, 0), mode=0, nrows=None, H=None, want_traj=True, defines=()):
    lib = build(reward_source=getattr(env, "reward_source", None) or None, defines=defines)
    md = _capi.fill_model_desc(env.sys.model)
    nq, nv, nu, nb = md.nq, md.nv, md.nu, md.nbody
    f32 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32)
    qpos, qvel, warm, us, eps, Ybar, noise = map(f32, (qpos, qvel, warm, us, eps, Ybar, noise))
    if mode == 0:
        nrows, H = us.shape[0], us.shape[1]
    out = dict(rewss=np.zeros((nrows, H), np.float32), rews=np.zeros(nrows, np.float32),
               q=np.zeros((nrows, H, nq), np.float32), qd=np.zeros((nrows, H, nv), np.float32),
               xpos=np.zeros((nrows, H, nb - 1, 3), np.float32), qpos_out=np.zeros(nq, np.float32),
               qvel_out=np.zeros(nv, np.float32), warm_out=np.zeros(nv, np.float32),
               ctrl_out=np.zeros(nu, np.float32), slab=np.zeros(8192, np.float32))
    rc = lib.emul_rollout(C.byref(md), C.byref(plan_desc), mode, nrows, H, step0, stage0, _p(qpos), _p(qvel),
                          _p(warm), _p(us), _p(eps), _p(Ybar), _p(noise), C.c_uint32(key[0]), C.c_uint32(key[1]),
                          _p(out["rewss"]), _p(out["rews"]), _p(out["q"]), _p(out["qd"]), _p(out["xpos"]),
                          _p(out["qpos_out"]), _p(out["qvel_out"]), _p(out["warm_out"]), _p(out["ctrl_out"]),
                          _p(out["slab"]))
    assert rc == 0
    return out


class EmulPlan:
    """TEST-ONLY stand-in for dial_mpc_b200.plan.Plan on CPU tensors: stage 1 runs the real
    device code through the warp emulator, stage 2/3 (weights, Ybar, bars) are NumPy.  Used by
    the gloo tests to exercise MBDPI's multi-rank plumbing without a GPU."""

    def __init__(self, env, desc):
        import torch
        self.env, self.desc = env, desc
        self.device = torch.device("cpu")
        m = env.sys
        self.nq, self.nv, self.nu, self.nbody = m.nq, m.nv, m.nu, m.nbody
        self.N, self.Ntotal, self.Hs, self.Hn = desc.Nsample, desc.Ntotal, desc.Hsample, desc.Hnode
        self.launches = 0
        self._traj = None

    def f32(self, x, shape=None):
        import torch
        t = x.to(torch.float32).contiguous() if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x, dtype=np.float32))
        if shape is not None:
            assert tuple(t.shape) == tuple(shape)
        return t

    def _np(self, t):
        return None if t is None else t.detach().cpu().numpy()

    def reverse_rollout(self, state, eps, key, Ybar, noise_scale, rews_local):
        ps = state.pipeline_state
        key = (0, 0) if key is None else (int(key[0]), int(key[1]))
        out = rollout(self.env, self.desc, self._np(ps.qpos), self._np(ps.qvel), self._np(ps.qacc_warmstart),
                      step0=int(state.info.get("step", 0)), stage0=int(state.info.get("contact_stage", 0)),
                      eps=self._np(eps), Ybar=self._np(Ybar), noise=self._np(noise_scale), key=key, mode=1,
                      nrows=self.N + 1, H=self.Hs + 1)
        self._traj = out
        rews_local.copy_(self.f32(out["rews"]))
        self.launches += 1

    def _Y0s(self, eps, Ybar, noise):
        Y0s = eps * noise[None, :, None] + Ybar
        Y0s[:, 0] = Ybar[0]
        return np.clip(np.concatenate([Y0s, Ybar[None]], 0), -1, 1)

    def reverse_update(self, eps, key, Ybar, noise_scale, rews_all, Ybar_out, weights=None):
        assert eps is not None, "EmulPlan.reverse_update needs injected eps"
        r = self._np(rews_all).astype(np.float64)
        logp = (r - r[-1]) / r.std() / self.desc.temp_sample
        w = np.exp(logp - logp.max())
        w /= w.sum()
        Y0s = self._Y0s(self._np(eps).astype(np.float64), self._np(Ybar).astype(np.float64), self._np(noise_scale).astype(np.float64))
        Ybar_out.copy_(self.f32(np.einsum("n,nij->ij", w, Y0s)))
        if weights is not None:
            weights.copy_(self.f32(w))

    def reverse_trajbar(self, weights, rank, qbar, qdbar, xbar):
        w = self._np(weights).astype(np.float64)
        off, N = self.desc.shard_offset, self.N
        wl = np.concatenate([w[off:off + N], [w[-1] if rank == 0 else 0.0]])
        t = self._traj
        qbar.copy_(self.f32(np.einsum("n,nij->ij", wl, t["q"]).ravel()))
        qdbar.copy_(self.f32(np.einsum("n,nij->ij", wl, t["qd"]).ravel()))
        xbar.copy_(self.f32(np.einsum("n,nijk->ijk", wl, t["xpos"]).ravel()))
