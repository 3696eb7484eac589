"""Drives the LIVE Python reference with injected draws.

The reference is a checkout of the original project (Jason-Hoford/inversus-reinforcement-learning),
named by the environment variable INVERSUS_REFERENCE_ROOT; it is not part of this repository. Used
by tests/golden/make_golden.py (fixture generation) and tests/test_oracle_vs_reference_live.py
(differential fuzz, skipped when the reference is absent). Never imported by the product,
bench.py or any -m gpu test.

RNG injection seams (SURVEY.md section 8c):
  * inversus_rl.env_wrappers.random  -- module attribute used by dummy_opponent_policy
    (env_wrappers.py:96,105,106,123,138,155)
  * InversusEnv.rng                  -- per-env object with .randint (core.py:41,69-87)
Both are replaced by DrawShim objects that serve draws from the same counter-based stream
(Philox4x32-10 keyed (seed, env, episode, stream, k)) or from an explicit table.
"""
from __future__ import annotations

import os
import sys

import numpy as np

REFERENCE_ROOT = os.environ.get("INVERSUS_REFERENCE_ROOT", "")
SKIP_REASON = "original project not present (set INVERSUS_REFERENCE_ROOT to a checkout of it)"
STREAM_RESET = 0xFFFFFFFF
TABLE_STRIDE = 64
TABLE_RESET_OFF = 16
M32 = 0xFFFFFFFF


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "inversus_rl"))


def philox4x32_10(ctr, key):
    """Pure-Python Philox4x32-10 (independent of oracle/ and of the CUDA code)."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0 = 0xD2511F53 * c0
        p1 = 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & M32, p1 & M32, ((p0 >> 32) ^ c3 ^ k1) & M32, p0 & M32
        k0 = (k0 + 0x9E3779B9) & M32
        k1 = (k1 + 0xBB67AE85) & M32
    return c0, c1, c2, c3


class DrawShim:
    """Stands in for `random` / `random.Random`: random(), shuffle(), randint() from a stream."""

    def __init__(self, seed=0):
        self.seed = seed
        self.env_gid = 0
        self.episode = 0
        self.stream = 0
        self.k = 0
        self.table = None  # 1-D sequence of u32 for the current call, or None
        self._cache_key = None
        self._cache = None

    def set_context(self, env_gid, episode, stream, table=None):
        self.env_gid, self.episode, self.stream, self.k, self.table = env_gid, episode, stream, 0, table

    def _u32(self):
        k = self.k
        self.k += 1
        if self.table is not None:
            return int(self.table[k])
        ck = (self.env_gid, self.episode, self.stream, k >> 2)
        if ck != self._cache_key:
            self._cache = philox4x32_10(ck, (self.seed & M32, (self.seed >> 32) & M32))
            self._cache_key = ck
        return self._cache[k & 3]

    def random(self):
        return self._u32() / 4294967296.0

    def _below(self, n):
        return (self._u32() * n) >> 32

    def randint(self, a, b):
        n = b - a + 1
        if n <= 0:
            self._u32()
            return a
        return a + self._below(n)

    def shuffle(self, x):
        for i in reversed(range(1, len(x))):
            j = self._below(i + 1)
            x[i], x[j] = x[j], x[i]


def import_reference():
    if not reference_available():
        raise RuntimeError(SKIP_REASON)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import inversus.core  # noqa: F401
    import inversus_rl.env_wrappers as ew
    return ew


DIR_IDX = {"up": 0, "right": 1, "down": 2, "left": 3}

STATE_DTYPE = np.dtype([
    ("tiles", np.uint32, (5,)),
    ("p1", np.int32, (5,)),
    ("p2", np.int32, (5,)),
    ("n_bullets", np.int32),
    ("bullets", np.int8, (16, 4)),
    ("step_count", np.int32),
    ("episode", np.uint32),
    ("episode_return", np.float64),
], align=True)


def ref_state(rl_env, episode):
    """Canonical state of one reference SingleInversusRLEnv (15x10)."""
    from inversus.game_types import TileColor, PlayerId
    env = rl_env.env
    s = np.zeros((), STATE_DTYPE)
    bits = np.zeros(160, np.uint8)
    for y in range(env.height):
        for x in range(env.width):
            bits[y * env.width + x] = 1 if env.grid[y][x] == TileColor.WHITE else 0
    s["tiles"] = np.packbits(bits, bitorder="little").view(np.uint32)
    for name, p in (("p1", env.player1), ("p2", env.player2)):
        s[name] = (p.x, p.y, p.ammo, p.reload_counter, int(p.alive))
    assert len(env.bullets) <= 16
    s["n_bullets"] = len(env.bullets)
    for i, b in enumerate(env.bullets):
        s["bullets"][i] = (b.x, b.y, DIR_IDX[b.dir.value], 0 if b.owner == PlayerId.P1 else 1)
    s["step_count"] = rl_env.step_count
    s["episode"] = episode
    s["episode_return"] = rl_env.episode_return
    return s


class ReferenceRunner:
    """N live reference envs stepped one at a time with per-call draw contexts."""

    def __init__(self, n, mode="dummy", difficulty="hard", max_episode_steps=500, seed=0, env_id_base=0):
        self.ew = import_reference()
        self.n = n
        self.mode = mode
        self.seed = seed
        self.env_id_base = env_id_base
        self.step_shim = DrawShim(seed)
        self.reset_shim = DrawShim(seed)
        self.ew.random = self.step_shim  # seam (1)
        self.envs = [self.ew.SingleInversusRLEnv(mode, difficulty, max_episode_steps, seed=0) for _ in range(n)]
        for e in self.envs:
            e.env.rng = self.reset_shim  # seam (2)
        self.episode = [-1] * n

    def close(self):
        import random as _random
        self.ew.random = _random

    def reset_env(self, i, table_row=None):
        self.episode[i] += 1
        t = None if table_row is None else table_row[TABLE_RESET_OFF:]
        self.reset_shim.set_context(self.env_id_base + i, self.episode[i], STREAM_RESET, t)
        return self.envs[i].reset()

    def reset(self, table=None):
        obs = [self.reset_env(i, None if table is None else table[i]) for i in range(self.n)]
        return np.stack([o[0] for o in obs]), np.stack([o[1] for o in obs])

    def step(self, a1, a2=None, table=None, auto_reset=False):
        """Returns dict of per-env outputs (trainer semantics when auto_reset)."""
        n = self.n
        out = dict(reward=np.zeros(n, np.float64), done=np.zeros(n, np.uint8), flags=np.zeros(n, np.uint8),
                   episode_steps=np.zeros(n, np.int32), episode_return=np.zeros(n, np.float64),
                   obs1=np.zeros((n, 12, 10, 15), np.float32), extra1=np.zeros((n, 4), np.float32),
                   obs2=np.zeros((n, 12, 10, 15), np.float32), extra2=np.zeros((n, 4), np.float32))
        from inversus.game_types import PlayerId
        for i, env in enumerate(self.envs):
            row = None if table is None else table[i]
            self.step_shim.set_context(self.env_id_base + i, self.episode[i], env.step_count, row)
            pol = None
            if self.mode == "selfplay":
                a2i = int(a2[i])
                pol = lambda obs, a2i=a2i: a2i  # noqa: E731
            obs, reward, done, info = env.step(int(a1[i]), pol)
            out["reward"][i] = reward
            out["done"][i] = done
            out["flags"][i] = (int(info["landed_hit"]) | int(info["got_hit"]) << 1
                               | int(info["win"]) << 2 | int(info["lose"]) << 3)
            out["episode_steps"][i] = info["episode_steps"]
            out["episode_return"][i] = info["episode_return"]
            if done and auto_reset:
                obs = self.reset_env(i, row)  # training.py:148-151
            out["obs1"][i], out["extra1"][i] = obs
            o2 = self.ew.build_observation(env.env, PlayerId.P2)
            out["obs2"][i], out["extra2"][i] = o2
        return out

    def state(self):
        s = np.zeros(self.n, STATE_DTYPE)
        for i, e in enumerate(self.envs):
            s[i] = ref_state(e, self.episode[i])
        return s
