"""Seeded parity scenarios shared by the fixture generator and the parity tests.

A *backend* is anything with
    reset(table) -> None
    step(a1, a2, table, auto_reset) -> dict(reward f64|f32, done, flags, episode_steps,
                                            episode_return, obs1, extra1[, obs2, extra2])
    reset_envs(indices, table) -> None        (MultiEnvRunner.envs[i].reset(), training.py:149)
    state() -> structured array (STATE_DTYPE)
    obs() -> (obs1, extra1, obs2|None, extra2|None) of the CURRENT state
`run_scenario` drives one through a scenario and returns every observable as arrays; the golden
fixtures are exactly that output for the live Python reference (make_golden.py).
"""
from __future__ import annotations

import numpy as np

TABLE_STRIDE = 64

SCENARIOS = {
    # name: mode, difficulty, max_episode_steps, n_envs, steps, seed, action mix, draw source, reset policy
    # hard_auto holds the first 480 steps of a 620-step recording (no episode of it reaches the
    # timeout), which keeps the fixture under 1 MB; step t's actions do not depend on the step count
    "hard_auto":   dict(mode="dummy", difficulty="hard", max_steps=500, n=40, T=480, seed=11, actions="uniform", draws="philox", resets="auto"),
    "easy_auto":   dict(mode="dummy", difficulty="easy", max_steps=500, n=24, T=540, seed=12, actions="uniform", draws="philox", resets="auto"),
    "hard_charge": dict(mode="dummy", difficulty="hard", max_steps=500, n=32, T=300, seed=13, actions="charge", draws="philox", resets="auto"),
    "selfplay":    dict(mode="selfplay", difficulty="hard", max_steps=500, n=40, T=400, seed=14, actions="uniform", draws="philox", resets="auto"),
    "hard_short":  dict(mode="dummy", difficulty="hard", max_steps=40, n=32, T=200, seed=15, actions="passive", draws="philox", resets="auto"),
    "hard_manual": dict(mode="dummy", difficulty="hard", max_steps=60, n=24, T=300, seed=16, actions="uniform", draws="philox", resets="manual"),
    "hard_table":  dict(mode="dummy", difficulty="hard", max_steps=500, n=32, T=300, seed=17, actions="uniform", draws="table", resets="auto"),
    "easy_table":  dict(mode="dummy", difficulty="easy", max_steps=120, n=32, T=300, seed=18, actions="passive", draws="table", resets="auto"),
    "selfplay_shooty": dict(mode="selfplay", difficulty="hard", max_steps=500, n=32, T=300, seed=19, actions="shooty", draws="philox", resets="auto"),
}


def gen_actions(kind, rs, n):
    if kind == "uniform":
        return rs.randint(0, 13, size=n).astype(np.int8)
    if kind == "charge":  # P(9..12) = 0.5 (BASELINE config 3)
        a = rs.randint(0, 13, size=n)
        c = rs.randint(9, 13, size=n)
        return np.where(rs.rand(n) < 0.5, c, a).astype(np.int8)
    if kind == "passive":  # mostly moves, so episodes run into the timeout
        a = rs.randint(0, 5, size=n)
        b = rs.randint(0, 13, size=n)
        return np.where(rs.rand(n) < 0.9, a, b).astype(np.int8)
    if kind == "shooty":  # bullet-heavy: many simultaneous bullets, merges and cancels
        a = rs.randint(5, 13, size=n)
        b = rs.randint(0, 13, size=n)
        return np.where(rs.rand(n) < 0.7, a, b).astype(np.int8)
    raise ValueError(kind)


def gen_table(rs, n):
    """Biased draw table: a quarter of the draws are tiny (u < 1e-3), a quarter small (u < 0.03),
    the rest uniform -- so the rare dummy branches and the 20-try spawn loop are exercised."""
    t = rs.randint(0, 2**32, size=(n, TABLE_STRIDE), dtype=np.uint64)
    sel = rs.randint(0, 4, size=(n, TABLE_STRIDE))
    t = np.where(sel == 0, t >> 10, t)
    t = np.where(sel == 1, t >> 5, t)
    # every 7th env: all-zero reset draws -> 20 failed tries, P2 spawns on top of P1
    t[::7, 16:] = 0
    return t.astype(np.uint32)


def run_scenario(backend, sc, record_obs=True):
    rs = np.random.RandomState(sc["seed"] & 0xFFFFFFFF)
    n, T = sc["n"], sc["T"]
    use_table = sc["draws"] == "table"
    selfplay = sc["mode"] == "selfplay"
    auto = sc["resets"] == "auto"

    table0 = gen_table(rs, n) if use_table else None
    backend.reset(table0)
    st0 = backend.state()
    o = backend.obs()
    rec = dict(
        init_state=st0.copy(),
        init_obs1=np.packbits(o[0] != 0, axis=None), init_extra1=np.asarray(o[1], np.float32).copy(),
        a1=np.zeros((T, n), np.int8), a2=np.zeros((T, n), np.int8),
        state=np.zeros((T, n), st0.dtype),
        reward=np.zeros((T, n), np.float64), reward_f32=np.zeros((T, n), np.float32),
        done=np.zeros((T, n), np.uint8), flags=np.zeros((T, n), np.uint8),
        episode_steps=np.zeros((T, n), np.int32), episode_return=np.zeros((T, n), np.float64),
        extra1=np.zeros((T, n, 4), np.float32),
    )
    obs1_bits, obs2_bits = [], []
    if selfplay:
        rec["extra2"] = np.zeros((T, n, 4), np.float32)
    for t in range(T):
        a1 = gen_actions(sc["actions"], rs, n)
        a2 = gen_actions(sc["actions"], rs, n) if selfplay else None
        table = gen_table(rs, n) if use_table else None
        out = backend.step(a1, a2, table, auto)
        if not auto and t % 25 == 24:
            idx = np.nonzero(out["done"])[0]
            if len(idx):
                backend.reset_envs(idx, table)
                o = backend.obs()
                out["obs1"], out["extra1"] = o[0], o[1]
                if selfplay:
                    out["obs2"], out["extra2"] = o[2], o[3]
        rec["a1"][t] = a1
        if selfplay:
            rec["a2"][t] = a2
        rec["state"][t] = backend.state()
        rec["reward"][t] = out["reward"]
        rec["reward_f32"][t] = np.asarray(out["reward"]).astype(np.float32)
        rec["done"][t] = out["done"]
        rec["flags"][t] = out["flags"]
        rec["episode_steps"][t] = out["episode_steps"]
        rec["episode_return"][t] = out["episode_return"]
        rec["extra1"][t] = out["extra1"]
        if record_obs:
            vals = np.unique(out["obs1"])
            assert set(vals.tolist()) <= {0.0, 1.0}
            obs1_bits.append(np.packbits(np.asarray(out["obs1"]) != 0, axis=None))
        if selfplay:
            rec["extra2"][t] = out["extra2"]
            if record_obs:
                obs2_bits.append(np.packbits(np.asarray(out["obs2"]) != 0, axis=None))
    if record_obs:
        rec["obs1_bits"] = np.stack(obs1_bits)
        if selfplay:
            rec["obs2_bits"] = np.stack(obs2_bits)
    return rec


COMPARE_EXACT = ["init_state", "init_obs1", "init_extra1", "a1", "a2", "state", "done", "flags",
                 "episode_steps", "extra1", "extra2", "obs1_bits", "obs2_bits", "reward_f32"]


def compare(rec, gold, float_rtol=1e-6, what=""):
    """Bit-exact on every integer/obs field; rewards/returns within float_rtol relative
    (they are in fact reproduced exactly -- asserted separately where promised)."""
    for k in COMPARE_EXACT:
        if k not in gold:
            continue
        a, b = np.asarray(rec[k]), np.asarray(gold[k])
        if k in ("state", "init_state"):
            for f in b.dtype.names:
                if f == "episode_return":
                    np.testing.assert_allclose(a[f], b[f], rtol=float_rtol, atol=1e-12, err_msg=f"{what}:{k}.{f}")
                else:
                    if not np.array_equal(a[f], b[f]):
                        bad = np.argwhere(a[f] != b[f])[0]
                        raise AssertionError(f"{what}: state field {f} differs first at index {tuple(bad)}: "
                                             f"{a[f][tuple(bad[:a[f].ndim])]} vs {b[f][tuple(bad[:b[f].ndim])]}")
        else:
            if not np.array_equal(a, b):
                bad = np.argwhere(a != b)[0]
                raise AssertionError(f"{what}: {k} differs first at {tuple(bad)}: {a[tuple(bad)]} vs {b[tuple(bad)]}")
    np.testing.assert_allclose(rec["reward"], gold["reward"], rtol=float_rtol, atol=1e-12, err_msg=f"{what}:reward")
    np.testing.assert_allclose(rec["episode_return"], gold["episode_return"], rtol=float_rtol, atol=1e-12,
                               err_msg=f"{what}:episode_return")
