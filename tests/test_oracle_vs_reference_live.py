"""Checks against the LIVE Python reference (tests/ref_harness.py): skipped unless
INVERSUS_REFERENCE_ROOT names a checkout of the original project. Nothing here runs under -m gpu.

1. The restated known-answer tests (tests/reference_kat.py) are first run against the real
   `inversus.core.InversusEnv`, proving the restatements are true of the reference itself.
2. Fresh differential fuzz (seeds that are NOT in the committed fixtures): live reference vs
   the C oracle, all modes, bit-exact state/obs/flags and exact fp64 returns.
"""
import numpy as np
import pytest

import reference_kat as K
from ref_harness import SKIP_REASON, DrawShim, import_reference, reference_available
from engine_facade import Bullet, P1, P2

pytestmark = [pytest.mark.live_reference, pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)]


class ReferenceEngine:
    """inversus.core.InversusEnv behind the integer encoding of tests/engine_facade.py."""

    def __init__(self, width, height):
        import_reference()
        import inversus.core as core
        from inversus.game_types import Direction, PlayerId, TileColor
        self.core = core
        self.D = [Direction.UP, Direction.RIGHT, Direction.DOWN, Direction.LEFT]
        self.PID = [PlayerId.P1, PlayerId.P2]
        self.TC = [TileColor.BLACK, TileColor.WHITE]
        shim = DrawShim(1234)

        class _R:  # lets the constructor's random.Random(seed) survive height=1 (SURVEY.md section 4)
            @staticmethod
            def Random(seed=None):
                return shim
        old = core.random
        core.random = _R
        try:
            self.env = core.InversusEnv(width=width, height=height)
        finally:
            core.random = old
        self.width, self.height = width, height

    @property
    def player1(self):
        return self.env.player1

    @property
    def player2(self):
        return self.env.player2

    player_x = property(lambda s: s.env.player_x, lambda s, v: setattr(s.env, "player_x", v))
    player_y = property(lambda s: s.env.player_y, lambda s, v: setattr(s.env, "player_y", v))

    @property
    def bullets(self):
        return [Bullet(b.x, b.y, self.D.index(b.dir), self.PID.index(b.owner)) for b in self.env.bullets]

    @bullets.setter
    def bullets(self, lst):
        from inversus.game_types import Bullet as RB
        self.env.bullets = [RB(x=b.x, y=b.y, dir=self.D[b.dir], owner=self.PID[b.owner]) for b in lst]

    def get_bullets(self):
        return self.bullets

    def _get_tile(self, x, y):
        return self.TC.index(self.env._get_tile(x, y))

    def _set_tile(self, x, y, c):
        self.env._set_tile(x, y, self.TC[c])

    def reset(self):
        self.env.reset()

    def try_move_player(self, d, pid=P1):
        return self.env.try_move_player(self.D[d], self.PID[pid])

    def spawn_bullet(self, d, pid=P1):
        return self.env.spawn_bullet(self.D[d], self.PID[pid])

    def spawn_wide_shot(self, pid, d):
        return self.env.spawn_wide_shot(self.PID[pid], self.D[d])

    def _reload_ammo(self):
        self.env._reload_ammo()

    def update_bullets(self):
        self.env.update_bullets()

    def step_players(self, a1, a2):
        from inversus_rl.env_wrappers import discrete_to_action
        self.env.step_players(discrete_to_action(a1), discrete_to_action(a2))

    def step(self, a1):
        from inversus_rl.env_wrappers import discrete_to_action
        self.env.step(discrete_to_action(a1))

    def is_round_over(self):
        return self.env.is_round_over()

    def get_winner(self):
        w = self.env.get_winner()
        return None if w is None else self.PID.index(w)

    def observation(self, viewer=P1):
        from inversus_rl.env_wrappers import build_observation
        return build_observation(self.env, self.PID[viewer])


@pytest.mark.parametrize("name", K.ALL_KATS)
def test_restated_kats_hold_on_the_live_reference(name):
    getattr(K, name)(lambda w, h: ReferenceEngine(w, h))


@pytest.mark.parametrize("name", K.ALL_KATS)
def test_restated_kats_hold_on_the_live_reference_15x10(name):
    getattr(K, name)(lambda w, h: ReferenceEngine(15, 10))


FUZZ = {
    "fz_hard":     dict(mode="dummy", difficulty="hard", max_steps=500, n=12, T=150, seed=101, actions="uniform", draws="philox", resets="auto"),
    "fz_easy":     dict(mode="dummy", difficulty="easy", max_steps=50, n=12, T=150, seed=102, actions="shooty", draws="philox", resets="auto"),
    "fz_selfplay": dict(mode="selfplay", difficulty="hard", max_steps=90, n=12, T=150, seed=103, actions="shooty", draws="philox", resets="auto"),
    "fz_table":    dict(mode="dummy", difficulty="hard", max_steps=70, n=12, T=150, seed=104, actions="charge", draws="table", resets="manual"),
}


@pytest.mark.parametrize("name", sorted(FUZZ))
def test_fresh_differential_fuzz(name):
    from backends import OracleBackend
    from golden.make_golden import ReferenceBackend
    from golden.scenarios import compare, run_scenario
    sc = FUZZ[name]
    rb = ReferenceBackend(sc)
    try:
        gold = run_scenario(rb, sc)
    finally:
        rb.r.close()
    rec = run_scenario(OracleBackend(sc), sc)
    compare(rec, gold, what=name)
    assert np.array_equal(rec["episode_return"], gold["episode_return"])
