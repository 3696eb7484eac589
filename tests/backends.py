"""Scenario backends (see tests/golden/scenarios.py) for the CPU oracle and the CUDA product."""
from __future__ import annotations

import ctypes as C

import numpy as np

from oracle.oracle import STATE_DTYPE


class OracleBackend:
    """The C oracle (oracle/inversus_oracle.c) as a scenario backend. Checker only."""

    def __init__(self, sc, env_id_base=0, n=None, nthreads=1):
        from oracle import oracle as orc
        self.orc = orc
        self.b = orc.OracleBatch(n or sc["n"], sc["mode"], sc["difficulty"], sc["max_steps"],
                                 seed=sc["seed"], env_id_base=env_id_base, nthreads=nthreads)
        self.selfplay = sc["mode"] == "selfplay"

    def reset(self, table):
        self.b.reset(table)

    def step(self, a1, a2, table, auto_reset):
        b = self.b
        b.step(a1, a2, table, auto_reset)
        out = dict(reward=b.reward.copy(), done=b.done.copy(), flags=b.flags.copy(),
                   episode_steps=b.episode_steps.copy(), episode_return=b.episode_return.copy(),
                   obs1=b.obs1, extra1=b.extra1)
        if self.selfplay:
            out["obs2"], out["extra2"] = b.obs2, b.extra2
        return out

    def reset_envs(self, idx, table):
        L = self.orc.lib()
        for i in idx:
            e = self.b.envs[int(i)]
            if table is not None:
                row = np.ascontiguousarray(table[int(i)], np.uint32)
                e.table = row.ctypes.data_as(C.POINTER(C.c_uint32))
            L.orc_rl_reset(C.byref(e))
            e.table = None

    def state(self):
        return self.b.export_state()

    def obs(self):
        b = self.b
        L = self.orc.lib()
        o2 = np.zeros_like(b.obs1)
        e2 = np.zeros_like(b.extra1)
        for i in range(b.n):
            L.orc_build_obs(C.byref(b.envs[i]), 0, b.obs1[i].ctypes.data, b.extra1[i].ctypes.data)
            L.orc_build_obs(C.byref(b.envs[i]), 1, o2[i].ctypes.data, e2[i].ctypes.data)
        return b.obs1, b.extra1, o2, e2


class CudaBackend:
    """The CUDA product (through BatchedInversus -> C ABI) as a scenario backend."""

    def __init__(self, sc, env_id_base=0, n=None, obs_dtype="f32"):
        import torch
        from inversus_b200 import BatchedInversus
        self.torch = torch
        self.selfplay = sc["mode"] == "selfplay"
        self.sim = BatchedInversus(n or sc["n"], sc["mode"], sc["difficulty"], sc["max_steps"], seed=sc["seed"],
                                   auto_reset=(sc["resets"] == "auto"), env_id_base=env_id_base,
                                   obs_dtype=obs_dtype, p2_view=True, reward_f64=True)

    def _table(self, table):
        self.sim.set_draw_table(table)

    def reset(self, table):
        self._table(table)
        self.sim.reset()

    def step(self, a1, a2, table, auto_reset):
        assert auto_reset == self.sim.auto_reset
        self._table(table)
        s = self.sim
        s.step(self.torch.from_numpy(np.asarray(a1, np.int8)).cuda(),
               None if a2 is None else self.torch.from_numpy(np.asarray(a2, np.int8)).cuda())
        r64 = s.reward_f64.cpu().numpy()  # the unrounded binary64 reward; the f32 output must be its rounding
        assert np.array_equal(s.reward.cpu().numpy(), r64.astype(np.float32))
        out = dict(reward=r64, done=s.done.cpu().numpy(), flags=s.info.cpu().numpy(),
                   episode_steps=s.episode_steps.cpu().numpy(), episode_return=s.episode_return.cpu().numpy(),
                   obs1=s.obs.float().cpu().numpy(), extra1=s.extra.cpu().numpy())
        if self.selfplay:
            out["obs2"], out["extra2"] = s.obs_p2.float().cpu().numpy(), s.extra_p2.cpu().numpy()
        assert s.poll_status() == 0
        return out

    def reset_envs(self, idx, table):
        self._table(table)
        self.sim.reset_envs(np.asarray(idx, np.int64))

    def state(self):
        return self.sim.export_state()

    def obs(self):
        s = self.sim
        return (s.obs.float().cpu().numpy(), s.extra.cpu().numpy(),
                s.obs_p2.float().cpu().numpy(), s.extra_p2.cpu().numpy())


class PyLoopBackend:
    """The pure-Python restatement (oracle/py_loop.py) as a scenario backend. Checker only."""

    def __init__(self, sc, env_id_base=0):
        from oracle import py_loop
        self.pl = py_loop
        self.r = py_loop.PyRunner(sc["n"], sc["mode"], sc["difficulty"], sc["max_steps"], seed=sc["seed"],
                                  env_id_base=env_id_base)
        self.selfplay = sc["mode"] == "selfplay"

    def reset(self, table):
        self.r.reset(table)

    def step(self, a1, a2, table, auto_reset):
        return self.r.step(a1, a2, table, auto_reset, both_views=self.selfplay)

    def reset_envs(self, idx, table):
        for i in idx:
            self.r.envs[int(i)].reset(None if table is None else table[int(i)])

    def state(self):
        T = self.pl.Tile
        out = np.zeros(self.r.n, STATE_DTYPE)
        for i, e in enumerate(self.r.envs):
            bits = np.zeros(160, np.uint8)
            for y in range(10):
                for x in range(15):
                    bits[y * 15 + x] = 1 if e.grid[y][x] == T.WHITE else 0
            out["tiles"][i] = np.packbits(bits, bitorder="little").view(np.uint32)
            for name, p in (("p1", e.p1), ("p2", e.p2)):
                out[name][i] = (p.x, p.y, p.ammo, p.reload_counter, int(p.alive))
            out["n_bullets"][i] = len(e.bullets)
            for k, b in enumerate(e.bullets):
                out["bullets"][i, k] = (b.x, b.y, b.dir.value, b.owner)
            out["step_count"][i] = e.step_count
            out["episode"][i] = e.episode
            out["episode_return"][i] = e.episode_return
        return out

    def obs(self):
        o1, o2 = self.r.observations(0), self.r.observations(1)
        return o1[0], o1[1], o2[0], o2[1]


class HostKernelBackend:
    """The PRODUCT's own step logic (csrc/inversus_kernels.cuh: load_env, rl_step, rl_reset,
    build_row, store_env) and canonical-state conversions compiled for the host through
    tests/host_kernel/host_shim.h and driven over the same packed-state planes the GPU uses. Test harness only: it lets the CPU suite replay
    the golden fixtures through the real kernel logic without a GPU."""

    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            import os
            import subprocess
            here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_kernel")
            so = os.path.join(here, "libhost_kernel.so")
            srcs = [os.path.join(here, "harness.cpp"), os.path.join(here, "host_shim.h"),
                    os.path.join(os.path.dirname(here), "..", "inversus-reinforcement-learning_b200", "csrc",
                                 "inversus_kernels.cuh")]
            if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
                subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                                       "-Wno-unknown-pragmas", "-I", here, "-o", so, srcs[0]])
            cls._lib = C.CDLL(so)
        return cls._lib

    def __init__(self, sc, env_id_base=0):
        self.n = sc["n"]
        self.mode = {"dummy": 0, "selfplay": 1}[sc["mode"]]
        self.diff = {"easy": 0, "hard": 1}[sc["difficulty"]]
        self.max_steps, self.seed, self.base = sc["max_steps"], sc["seed"], env_id_base
        self.selfplay = sc["mode"] == "selfplay"
        n = self.n
        self.planes = np.zeros((5, n, 4), np.uint32)
        st = np.zeros(n, STATE_DTYPE)
        st["episode"] = 0xFFFFFFFF  # "no episode yet", like inv_create
        self.import_state(st)
        self.obs1 = np.zeros((n, 12, 10, 15), np.float32)
        self.obs2 = np.zeros((n, 12, 10, 15), np.float32)
        self.extra1 = np.zeros((n, 4), np.float32)
        self.extra2 = np.zeros((n, 4), np.float32)
        self.status = np.zeros(1, np.uint32)

    @staticmethod
    def _p(a):
        return None if a is None else a.ctypes.data_as(C.c_void_p)

    def _reset(self, idx, table):
        t = None if table is None else np.ascontiguousarray(table, np.uint32)
        i = None if idx is None else np.ascontiguousarray(idx, np.int64)
        self.lib().hk_reset(self._p(self.planes), C.c_int64(self.n), self._p(i), C.c_int64(0 if i is None else len(i)),
                            C.c_uint64(self.seed), C.c_uint32(self.base), self._p(t), self._p(self.obs1),
                            self._p(self.extra1), self._p(self.obs2), self._p(self.extra2), self._p(self.status))

    def reset(self, table):
        self._reset(None, table)

    def reset_envs(self, idx, table):
        self._reset(idx, table)

    def step(self, a1, a2, table, auto_reset):
        n = self.n
        a1 = np.ascontiguousarray(a1, np.int8)
        a2 = None if a2 is None else np.ascontiguousarray(a2, np.int8)
        t = None if table is None else np.ascontiguousarray(table, np.uint32)
        out = dict(reward=np.zeros(n, np.float32), done=np.zeros(n, np.uint8), flags=np.zeros(n, np.uint8),
                   episode_steps=np.zeros(n, np.int32), episode_return=np.zeros(n, np.float64))
        self.lib().hk_step(self._p(self.planes), C.c_int64(n), self._p(a1), self._p(a2), self._p(t), self.mode,
                           self.diff, self.max_steps, int(auto_reset), C.c_uint64(self.seed), C.c_uint32(self.base),
                           self._p(self.obs1), self._p(self.extra1), self._p(self.obs2), self._p(self.extra2),
                           self._p(out["reward"]), self._p(out["done"]), self._p(out["flags"]),
                           self._p(out["episode_steps"]), self._p(out["episode_return"]), self._p(self.status))
        assert self.status[0] == 0
        out["obs1"], out["extra1"] = self.obs1, self.extra1
        if self.selfplay:
            out["obs2"], out["extra2"] = self.obs2, self.extra2
        return out

    def export_state(self, first=0, count=None):
        """Canonical state of envs [first, first+count), decoded by the product's own conversion."""
        count = self.n - first if count is None else count
        out = np.zeros(count, STATE_DTYPE)
        self.lib().hk_export_state(self._p(self.planes), C.c_int64(self.n), C.c_int64(first), C.c_int64(count),
                                   self._p(out))
        return out

    def import_state(self, state, first=0):
        st = np.ascontiguousarray(state, STATE_DTYPE)
        if self.lib().hk_import_state(self._p(self.planes), C.c_int64(self.n), C.c_int64(first),
                                      C.c_int64(len(st)), self._p(st)) != 0:
            raise ValueError("hk_import_state: field out of range")

    def state(self):
        return self.export_state()

    def obs(self):
        return self.obs1, self.extra1, self.obs2, self.extra2


def check_state_import_export(export, import_):
    """Canonical state through a product's import/export: a round trip at an offset is exact, and
    every field outside the packed layout or the board is rejected. export(first=0, count=None) and
    import_(state, first=0) act on at least 11 envs after a reset."""
    import pytest
    st = export()
    st["bullets"][3, :2] = [[4, 5, 1, 0], [9, 2, 3, 1]]
    st["n_bullets"][3] = 2
    st["episode_return"][3] = -1.2345678901234567
    st["p1"][3] = (14, 9, 0, 29, 0)
    import_(st[3:4], first=10)
    back = export(10, 1)
    for f in st.dtype.names:
        assert np.array_equal(back[f][0], st[f][3]), f
    for field, bad in (("p1", (15, 0, 0, 0, 1)), ("p2", (0, 10, 0, 0, 1)), ("p1", (0, 0, 8, 0, 1)), ("p1", (0, 0, 0, 0, 2))):
        x = st[:1].copy()
        x[field][0] = bad
        with pytest.raises(ValueError):
            import_(x)
    x = st[:1].copy()
    x["n_bullets"][0] = 17
    with pytest.raises(ValueError):
        import_(x)
    x = st[:1].copy()
    x["tiles"][0][4] = 1 << 22  # bit beyond the 150 tiles
    with pytest.raises(ValueError):
        import_(x)
