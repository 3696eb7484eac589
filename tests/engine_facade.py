"""InversusEnv-shaped facades so the reference's own unit tests can be restated verbatim.

`OracleEngine` drives oracle/inversus_oracle.c one engine call at a time (core.py method names);
`CudaEngine` (tests/test_cuda_reference_kat.py) drives the CUDA product through its debug-phase
entry point with the same surface, and `HostKernelEngine` (tests/test_host_kernel.py) the same
engine functions compiled for the host. Directions/ids use the product's integer encoding:
UP, RIGHT, DOWN, LEFT = 0..3; P1, P2 = 0, 1; BLACK, WHITE = 0, 1.
"""
from __future__ import annotations

import ctypes as C
from collections import namedtuple

import numpy as np

Bullet = namedtuple("Bullet", "x y dir owner")
UP, RIGHT, DOWN, LEFT = 0, 1, 2, 3
P1, P2 = 0, 1
BLACK, WHITE = 0, 1
MAX_AMMO, RELOAD_TICKS_PER_AMMO, WIDE_SHOT_AMMO_COST = 6, 30, 3
NONE = 0


def MOVE(d):
    return 1 + d


def SHOOT(d):
    return 5 + d


def CHARGE(d):
    return 9 + d


class _PlayerView:
    def __init__(self, get, set_):
        object.__setattr__(self, "_get", get)
        object.__setattr__(self, "_set", set_)

    def __getattr__(self, k):
        v = self._get(k)
        return bool(v) if k == "alive" else v

    def __setattr__(self, k, v):
        self._set(k, int(v))


class OracleEngine:
    """oracle/inversus_oracle.c behind core.py's InversusEnv method names."""

    color = {P1: BLACK, P2: WHITE}

    def __init__(self, width=15, height=10, seed=1234):
        from oracle import oracle as orc
        self.orc, self.L = orc, orc.lib()
        self.e = orc.Env()
        self.L.orc_init(C.byref(self.e), width, height, 1, 1, 500, seed, 0)
        self.width, self.height = width, height
        self.player_color = BLACK
        self.reset()

    # --- players
    def _pv(self, i):
        names = {"x": "x", "y": "y", "ammo": "ammo", "reload_counter": "reload", "alive": "alive"}
        return _PlayerView(lambda k: getattr(self.e.p[i], names[k]),
                           lambda k, v: setattr(self.e.p[i], names[k], v))

    @property
    def player1(self):
        return self._pv(0)

    @property
    def player2(self):
        return self._pv(1)

    # legacy single-player accessors (core.py:156-181)
    @property
    def player_x(self):
        return self.e.p[0].x

    @player_x.setter
    def player_x(self, v):
        self.e.p[0].x = v

    @property
    def player_y(self):
        return self.e.p[0].y

    @player_y.setter
    def player_y(self, v):
        self.e.p[0].y = v
        self.e.n_bullets = 0  # core.py:180-181: the legacy y setter clears the bullet list

    # --- bullets
    @property
    def bullets(self):
        return [Bullet(b.x, b.y, b.dir, b.owner) for b in self.e.bullets[: self.e.n_bullets]]

    @bullets.setter
    def bullets(self, lst):
        self.e.n_bullets = len(lst)
        for i, b in enumerate(lst):
            s = self.e.bullets[i]
            s.x, s.y, s.dir, s.owner = b.x, b.y, b.dir, b.owner

    def get_bullets(self):
        return self.bullets

    # --- tiles
    def _get_tile(self, x, y):
        if not (0 <= x < self.width and 0 <= y < self.height):
            raise IndexError
        return self.e.grid[y * self.width + x]

    def _set_tile(self, x, y, c):
        if not (0 <= x < self.width and 0 <= y < self.height):
            raise IndexError
        self.e.grid[y * self.width + x] = c

    # --- engine calls
    def reset(self):
        self.L.orc_engine_reset(C.byref(self.e))

    def try_move_player(self, d, pid=P1):
        return bool(self.L.orc_try_move(C.byref(self.e), pid, d))

    def spawn_bullet(self, d, pid=P1):
        return bool(self.L.orc_spawn_bullet(C.byref(self.e), pid, d))

    def spawn_wide_shot(self, pid, d):
        return bool(self.L.orc_spawn_wide_shot(C.byref(self.e), pid, d))

    def _reload_ammo(self):
        self.L.orc_reload_ammo(C.byref(self.e))

    def update_bullets(self):
        self.L.orc_update_bullets(C.byref(self.e))

    def step_players(self, a1, a2):
        self.L.orc_step_players(C.byref(self.e), a1, a2)

    def step(self, a1):
        self.step_players(a1, NONE)

    def is_round_over(self):
        return bool(self.L.orc_is_round_over(C.byref(self.e)))

    def get_winner(self):
        return {0: None, 1: P1, 2: P2}[self.L.orc_get_winner(C.byref(self.e))]

    def observation(self, viewer=P1):
        g = np.zeros((12, self.height, self.width), np.float32)
        x = np.zeros(4, np.float32)
        self.L.orc_build_obs(C.byref(self.e), viewer, g.ctypes.data, x.ctypes.data)
        return g, x


class _StateEngine:
    """core.py's method names over one env of the product: field pokes edit the canonical state
    (STATE_DTYPE) and go through the product's import/export; each engine call runs ONE engine
    method through the debug-phase dispatch the fused step kernel is built from. Fixed 15x10 board.
    Subclasses provide _export, _import, _run_phase and _observation."""

    def __init__(self, width, height):
        from inversus_b200 import _capi
        assert width <= 15 and height <= 10
        self.capi = _capi
        self.width, self.height = 15, 10
        self.player_color = BLACK
        self._pull()

    def _pull(self):
        self._st = self._export()
        self._dirty = False

    def _push(self):
        if self._dirty:
            self._import(self._st)
            self._dirty = False

    def _call(self, phase, pid=0, arg=0, arg2=0):
        self._push()
        res = self._run_phase(phase, pid, arg, arg2)
        self._pull()
        return res

    def _pv(self, name):
        idx = {"x": 0, "y": 1, "ammo": 2, "reload_counter": 3, "alive": 4}

        def get(k):
            return int(self._st[name][0][idx[k]])

        def set_(k, v):
            self._st[name][0][idx[k]] = v
            self._dirty = True
        return _PlayerView(get, set_)

    @property
    def player1(self):
        return self._pv("p1")

    @property
    def player2(self):
        return self._pv("p2")

    @property
    def player_x(self):
        return int(self._st["p1"][0][0])

    @player_x.setter
    def player_x(self, v):
        self._st["p1"][0][0] = v
        self._dirty = True

    @property
    def player_y(self):
        return int(self._st["p1"][0][1])

    @player_y.setter
    def player_y(self, v):
        self._st["p1"][0][1] = v
        self._st["n_bullets"][0] = 0  # core.py:180-181
        self._dirty = True

    @property
    def bullets(self):
        n = int(self._st["n_bullets"][0])
        return [Bullet(*(int(v) for v in self._st["bullets"][0][i])) for i in range(n)]

    @bullets.setter
    def bullets(self, lst):
        self._st["n_bullets"][0] = len(lst)
        self._st["bullets"][0][:] = 0
        for i, b in enumerate(lst):
            self._st["bullets"][0][i] = (b.x, b.y, b.dir, b.owner)
        self._dirty = True

    def get_bullets(self):
        return self.bullets

    def _get_tile(self, x, y):
        if not (0 <= x < self.width and 0 <= y < self.height):
            raise IndexError
        i = y * 15 + x
        return int(self._st["tiles"][0][i >> 5] >> (i & 31)) & 1

    def _set_tile(self, x, y, c):
        if not (0 <= x < self.width and 0 <= y < self.height):
            raise IndexError
        i = y * 15 + x
        w = int(self._st["tiles"][0][i >> 5])
        w = (w | (1 << (i & 31))) if c else (w & ~(1 << (i & 31)))
        self._st["tiles"][0][i >> 5] = w
        self._dirty = True

    def reset(self):
        self._call(self.capi.PHASE_ENGINE_RESET)

    def try_move_player(self, d, pid=P1):
        return bool(self._call(self.capi.PHASE_TRY_MOVE, pid, d))

    def spawn_bullet(self, d, pid=P1):
        return bool(self._call(self.capi.PHASE_SPAWN_BULLET, pid, d))

    def spawn_wide_shot(self, pid, d):
        return bool(self._call(self.capi.PHASE_WIDE_SHOT, pid, d))

    def _reload_ammo(self):
        self._call(self.capi.PHASE_RELOAD)

    def update_bullets(self):
        self._call(self.capi.PHASE_UPDATE_BULLETS)

    def step_players(self, a1, a2):
        self._call(self.capi.PHASE_STEP_PLAYERS, 0, a1, a2)

    def step(self, a1):
        self.step_players(a1, NONE)

    def is_round_over(self):
        return not (self.player1.alive and self.player2.alive)

    def get_winner(self):
        a1, a2 = self.player1.alive, self.player2.alive
        if a1 and a2:
            return None
        return P2 if (a2 and not a1) else (P1 if (a1 and not a2) else None)

    def observation(self, viewer=P1):
        self._push()
        return self._observation(viewer)


class CudaEngine(_StateEngine):
    """The CUDA product: inv_debug_phase on the device, inv_export_state / inv_import_state."""

    def __init__(self, width=15, height=10, seed=1234):
        from inversus_b200 import BatchedInversus
        self.sim = BatchedInversus(1, "selfplay", "hard", 500, seed=seed, auto_reset=False)
        self.sim.reset()
        super().__init__(width, height)

    def _export(self):
        return self.sim.export_state()

    def _import(self, st):
        self.sim.import_state(st)

    def _run_phase(self, phase, pid, arg, arg2):
        res = int(self.sim.debug_phase(phase, pid, arg, arg2).cpu()[0])
        assert self.sim.poll_status() == 0
        return res

    def _observation(self, viewer):
        g, e = self.sim.obs_from_packed(self.sim.snapshot(), view=viewer, obs_dtype="f32")
        return g[0].cpu().numpy(), e[0].cpu().numpy()


class HostKernelEngine(_StateEngine):
    """The product's engine functions and state conversions compiled for the host (tests/host_kernel):
    the CPU-side twin of CudaEngine, no GPU needed."""

    def __init__(self, width=15, height=10, seed=1234):
        from backends import HostKernelBackend
        self.b = HostKernelBackend(dict(n=1, mode="selfplay", difficulty="hard", max_steps=500, seed=seed))
        self.b.reset(None)
        super().__init__(width, height)

    def _export(self):
        return self.b.export_state()

    def _import(self, st):
        self.b.import_state(st)

    def _run_phase(self, phase, pid, arg, arg2):
        b = self.b
        res = np.zeros(1, np.uint8)
        rc = b.lib().hk_debug(b._p(b.planes), C.c_int64(1), phase, pid, arg, arg2, 1, C.c_uint64(b.seed), C.c_uint32(0),
                              b._p(res), b._p(b.status))
        assert rc == 0 and b.status[0] == 0
        return int(res[0])

    def _observation(self, viewer):
        b = self.b
        g, e = np.zeros((12, 10, 15), np.float32), np.zeros(4, np.float32)
        b.lib().hk_observation(b._p(b.planes), C.c_int64(1), C.c_int64(0), viewer, b._p(g), b._p(e))
        return g, e
