"""The reference's own engine unit tests, restated against an InversusEnv-shaped facade.

Each function takes `make(width, height)` and follows one test of the original project's tests/
(file:line cited). Board extents are read back from the env (`env.width`) so the same bodies
run on the oracle at the reference's board sizes and on the CUDA product's fixed 15x10 board.
Height-1 boards of the reference tests are row 0 of whatever board the facade provides.
"""
from engine_facade import (BLACK, CHARGE, DOWN, LEFT, MAX_AMMO, MOVE, NONE, P1, P2,
                           RELOAD_TICKS_PER_AMMO, RIGHT, SHOOT, UP, WHITE, WIDE_SHOT_AMMO_COST, Bullet)

# ---------------- tests/test_bullet_collision.py


def kat_bullets_cancel_each_other_on_same_tile(make):  # test_bullet_collision.py:8
    env = make(5, 1)
    env._set_tile(2, 0, BLACK)
    env.bullets = [Bullet(1, 0, RIGHT, P1), Bullet(3, 0, LEFT, P2)]
    env.update_bullets()
    assert len(env.bullets) == 0
    assert env._get_tile(2, 0) == BLACK


def kat_collision_does_not_hit_player(make):  # test_bullet_collision.py:35
    env = make(5, 1)
    env.player1.x, env.player1.y = 2, 0
    env.player1.alive = True
    env.bullets = [Bullet(1, 0, RIGHT, P2), Bullet(3, 0, LEFT, P1)]
    env.update_bullets()
    assert env.player1.alive is True
    assert len(env.bullets) == 0


def kat_same_owner_bullets_do_not_cancel(make):  # test_bullet_collision.py:59
    env = make(5, 1)
    env._set_tile(2, 0, BLACK)
    env.bullets = [Bullet(1, 0, RIGHT, P1), Bullet(0, 0, RIGHT, P1)]
    env.update_bullets()
    assert len(env.bullets) >= 1
    assert all(b.owner == P1 for b in env.bullets)
    assert env._get_tile(2, 0) == WHITE


def kat_collision_preserves_path_already_created(make):  # test_bullet_collision.py:85
    env = make(5, 1)
    for x in range(5):
        env._set_tile(x, 0, BLACK if x < 3 else WHITE)
    env.bullets = [Bullet(0, 0, RIGHT, P1), Bullet(4, 0, LEFT, P2)]
    env.update_bullets()
    assert env._get_tile(1, 0) == WHITE
    assert env._get_tile(3, 0) == BLACK
    env.update_bullets()
    assert len(env.bullets) == 0
    assert env._get_tile(1, 0) == WHITE
    assert env._get_tile(3, 0) == BLACK
    assert env._get_tile(2, 0) == BLACK


def kat_multiple_bullets_from_different_owners_cancel(make):  # test_bullet_collision.py:126
    env = make(5, 1)
    env._set_tile(2, 0, BLACK)
    env.bullets = [Bullet(1, 0, RIGHT, P1), Bullet(1, 0, RIGHT, P1), Bullet(3, 0, LEFT, P2)]
    env.update_bullets()
    assert len(env.bullets) == 0
    assert env._get_tile(2, 0) == BLACK


def kat_bullets_cancel_at_different_positions(make):  # test_bullet_collision.py:171
    env = make(7, 1)
    env._set_tile(2, 0, BLACK)
    env._set_tile(4, 0, BLACK)
    env.bullets = [Bullet(1, 0, RIGHT, P1), Bullet(3, 0, LEFT, P2),
                   Bullet(3, 0, RIGHT, P1), Bullet(5, 0, LEFT, P2)]
    env.update_bullets()
    assert len(env.bullets) == 0
    assert env._get_tile(2, 0) == BLACK
    assert env._get_tile(4, 0) == BLACK


# ---------------- tests/test_bullet_flip_rules.py


def kat_bullet_only_flips_owner_color_tiles(make):  # test_bullet_flip_rules.py:8
    env = make(5, 1)
    env._set_tile(1, 0, BLACK)
    env._set_tile(2, 0, WHITE)
    env.player1.x, env.player1.y = 0, 0
    env.bullets = [Bullet(0, 0, RIGHT, P1)]
    env.update_bullets()
    assert (env.bullets[0].x, env.bullets[0].y) == (1, 0)
    assert env._get_tile(1, 0) == WHITE
    env.update_bullets()
    assert (env.bullets[0].x, env.bullets[0].y) == (2, 0)
    assert env._get_tile(2, 0) == WHITE


def kat_bullet_from_p2_only_flips_white_tiles(make):  # test_bullet_flip_rules.py:43
    env = make(5, 1)
    env._set_tile(1, 0, WHITE)
    env._set_tile(2, 0, BLACK)
    env.player2.x, env.player2.y = 0, 0
    env.bullets = [Bullet(0, 0, RIGHT, P2)]
    env.update_bullets()
    assert env.bullets[0].x == 1
    assert env._get_tile(1, 0) == BLACK
    env.update_bullets()
    assert env.bullets[0].x == 2
    assert env._get_tile(2, 0) == BLACK


def kat_bullet_does_not_destroy_existing_path(make):  # test_bullet_flip_rules.py:76
    env = make(10, 1)
    for x in range(3, 7):
        env._set_tile(x, 0, WHITE)
    env.player1.x, env.player1.y = 2, 0
    env.player1.ammo = 6
    env.spawn_bullet(RIGHT, P1)
    for _ in range(5):
        env.update_bullets()
    for x in range(3, 7):
        assert env._get_tile(x, 0) == WHITE


def kat_bullet_opens_new_path(make):  # test_bullet_flip_rules.py:102
    env = make(10, 1)
    for x in range(3, 7):
        env._set_tile(x, 0, BLACK)
    env.player1.x, env.player1.y = 2, 0
    env.player1.ammo = 6
    env.spawn_bullet(RIGHT, P1)
    for _ in range(5):
        env.update_bullets()
    for x in range(3, 7):
        assert env._get_tile(x, 0) == WHITE


# ---------------- tests/test_charge_shot.py


def kat_charge_shot_spawns_three_bullets_and_consumes_ammo(make):  # test_charge_shot.py:9
    env = make(7, 7)
    env.player1.ammo = MAX_AMMO
    env.player1.x, env.player1.y = 3, 3
    assert env.spawn_wide_shot(P1, UP) is True
    assert env.player1.ammo == MAX_AMMO - WIDE_SHOT_AMMO_COST
    assert len(env.bullets) == 3
    assert sorted(b.x for b in env.bullets) == [2, 3, 4]
    assert {b.y for b in env.bullets} == {3}
    assert {b.dir for b in env.bullets} == {UP}
    assert {b.owner for b in env.bullets} == {P1}
    # lane order is observable downstream (core.py:359-370): centre, -1, +1
    assert [b.x for b in env.bullets] == [3, 2, 4]


def kat_charge_shot_horizontal_spawns_correctly(make):  # test_charge_shot.py:44
    env = make(7, 7)
    env.player1.ammo = MAX_AMMO
    env.player1.x, env.player1.y = 3, 3
    assert env.spawn_wide_shot(P1, RIGHT) is True
    assert len(env.bullets) == 3
    assert {b.x for b in env.bullets} == {3}
    assert sorted(b.y for b in env.bullets) == [2, 3, 4]
    assert {b.dir for b in env.bullets} == {RIGHT}


def kat_charge_shot_requires_enough_ammo(make):  # test_charge_shot.py:68
    env = make(7, 7)
    env.player1.ammo = WIDE_SHOT_AMMO_COST - 1
    env.player1.x, env.player1.y = 3, 3
    assert env.spawn_wide_shot(P1, RIGHT) is False
    assert env.player1.ammo == WIDE_SHOT_AMMO_COST - 1
    assert len(env.bullets) == 0


def kat_charge_shot_respects_bounds_for_side_lanes(make):  # test_charge_shot.py:82
    env = make(7, 7)
    env.player1.ammo = MAX_AMMO
    env.player1.x, env.player1.y = 0, 3
    assert env.spawn_wide_shot(P1, UP) is True
    assert len(env.bullets) == 2
    assert sorted(b.x for b in env.bullets) == [0, 1]
    env.bullets = []
    env.player1.x, env.player1.y = 3, 0
    env.player1.ammo = MAX_AMMO
    assert env.spawn_wide_shot(P1, RIGHT) is True
    assert len(env.bullets) == 2
    assert sorted(b.y for b in env.bullets) == [0, 1]
    # and at the far edges of whatever board this is
    env.bullets = []
    env.player1.x, env.player1.y = env.width - 1, env.height - 1
    env.player1.ammo = MAX_AMMO
    assert env.spawn_wide_shot(P1, DOWN) is True
    assert sorted(b.x for b in env.bullets) == [env.width - 2, env.width - 1]
    assert env.player1.ammo == MAX_AMMO - WIDE_SHOT_AMMO_COST  # charged in full even when clipped


def kat_charge_shot_integration_with_step_players(make):  # test_charge_shot.py:122
    env = make(7, 7)
    env.player1.ammo = MAX_AMMO
    env.player1.x, env.player1.y = 3, 3
    env.player2.x, env.player2.y = 0, env.height - 1  # out of the way on every board
    env.step_players(CHARGE(UP), NONE)
    assert len(env.bullets) == 3
    assert env.player1.ammo == MAX_AMMO - WIDE_SHOT_AMMO_COST
    for b in env.bullets:
        assert b.y == 2 and b.x in (2, 3, 4)
    env.update_bullets()
    for b in env.bullets:
        assert b.y == 1 and b.x in (2, 3, 4)


def kat_charge_shot_bullets_behave_like_normal_bullets(make):  # test_charge_shot.py:153
    env = make(7, 7)
    env.player1.ammo = MAX_AMMO
    env.player1.x, env.player1.y = 3, 3
    for y in range(env.height):
        for x in range(env.width):
            env._set_tile(x, y, BLACK)
    env.spawn_wide_shot(P1, UP)
    env.update_bullets()
    assert len(env.bullets) == 3
    for b in env.bullets:
        assert b.y == 2
        assert env._get_tile(b.x, b.y) == WHITE


def kat_charge_shot_cannot_be_used_by_dead_player(make):  # test_charge_shot.py:174
    env = make(7, 7)
    env.player1.ammo = MAX_AMMO
    env.player1.alive = False
    assert env.spawn_wide_shot(P1, UP) is False
    assert len(env.bullets) == 0


# ---------------- tests/test_combat_and_ammo.py


def kat_shoot_consumes_ammo_and_blocks_when_empty(make):  # test_combat_and_ammo.py:9
    env = make(10, 10)
    env.player1.ammo = 1
    assert env.spawn_bullet(RIGHT, P1) is True
    assert env.player1.ammo == 0
    assert env.spawn_bullet(RIGHT, P1) is False
    assert env.player1.ammo == 0


def kat_ammo_reloads_over_time(make):  # test_combat_and_ammo.py:27
    env = make(10, 10)
    env.player1.ammo = 0
    env.player1.reload_counter = 0
    for i in range(RELOAD_TICKS_PER_AMMO):
        env._reload_ammo()
        if i < RELOAD_TICKS_PER_AMMO - 1:
            assert env.player1.ammo == 0
            assert env.player1.reload_counter == i + 1
    assert env.player1.ammo == 1
    assert env.player1.reload_counter == 0
    env.player1.ammo = MAX_AMMO
    env.player1.reload_counter = 0
    for _ in range(RELOAD_TICKS_PER_AMMO * 2):
        env._reload_ammo()
        assert env.player1.ammo <= MAX_AMMO
    assert env.player1.reload_counter == 0  # frozen at full ammo (core.py:392)


def kat_bullet_kills_opponent(make):  # test_combat_and_ammo.py:56
    env = make(10, 10)
    env.player1.x, env.player1.y = 1, 5
    env.player2.x, env.player2.y = 4, 5
    assert env.player1.alive and env.player2.alive
    for x in range(1, 5):
        env._set_tile(x, 5, WHITE)
    env.player1.ammo = MAX_AMMO
    env.spawn_bullet(RIGHT, P1)
    for _ in range(3):
        env.update_bullets()
    assert not env.player2.alive
    assert env.player1.alive
    assert env.is_round_over()
    assert env.get_winner() == P1
    assert len(env.bullets) == 1  # the bullet continues after the hit (core.py:473)


def kat_step_players_integrates_move_shoot_reload_and_bullets(make):  # test_combat_and_ammo.py:97
    env = make(10, 10)
    env.player1.x, env.player1.y = 5, 5
    env.player2.x, env.player2.y = 7, 5
    env.player1.ammo = MAX_AMMO
    env.player2.ammo = MAX_AMMO
    env._set_tile(5, 5, WHITE)
    env._set_tile(6, 5, BLACK)
    env._set_tile(7, 5, BLACK)
    ammo0, reload0, nb0 = env.player1.ammo, env.player1.reload_counter, len(env.get_bullets())
    env.step_players(SHOOT(RIGHT), MOVE(LEFT))
    assert env.player1.ammo == ammo0 - 1
    after = env.get_bullets()
    assert len(after) == nb0 + 1
    assert (after[0].x, after[0].y, after[0].owner) == (6, 5, P1)
    assert env._get_tile(6, 5) == WHITE  # flipped to P2's colour
    assert env.player1.reload_counter == reload0 + 1
    assert (env.player2.x, env.player2.y) == (6, 5)
    # NB: P2 walked onto the tile the bullet lands on in the same tick and dies (core.py:468-470)
    assert not env.player2.alive
    env.player1.ammo = MAX_AMMO - 1
    env.player1.reload_counter = 0
    for _ in range(RELOAD_TICKS_PER_AMMO):
        env.step_players(NONE, NONE)
    assert env.player1.ammo == MAX_AMMO


def kat_bullet_does_not_kill_owner(make):  # test_combat_and_ammo.py:169
    env = make(10, 10)
    env.player2.x, env.player2.y = 0, env.height - 1
    env.player1.x, env.player1.y = 5, 5
    env._set_tile(5, 5, WHITE)
    env._set_tile(4, 5, WHITE)
    env.player1.ammo = MAX_AMMO
    env.spawn_bullet(LEFT, P1)
    env.update_bullets()
    env.player1.x, env.player1.y = 4, 5
    env.update_bullets()
    assert env.player1.alive
    env.player1.x, env.player1.y = 5, 5
    env.player1.ammo = MAX_AMMO
    env.bullets = []
    env.spawn_bullet(RIGHT, P1)
    env.update_bullets()
    env.player1.x, env.player1.y = 7, 5  # stand exactly where the own bullet lands next
    env.update_bullets()
    assert env.bullets[0].x == 7
    assert env.player1.alive


def kat_dead_player_cannot_move_or_shoot(make):  # test_combat_and_ammo.py:222
    env = make(10, 10)
    env.player2.alive = False
    assert env.try_move_player(RIGHT, P2) is False
    env.player2.ammo = MAX_AMMO
    assert env.spawn_bullet(RIGHT, P2) is False


def kat_is_round_over_and_get_winner(make):  # test_combat_and_ammo.py:239
    env = make(10, 10)
    assert not env.is_round_over()
    assert env.get_winner() is None
    env.player2.alive = False
    assert env.is_round_over()
    assert env.get_winner() == P1
    env.reset()
    env.player1.alive = False
    assert env.is_round_over()
    assert env.get_winner() == P2
    env.reset()
    env.player1.alive = False
    env.player2.alive = False
    assert env.is_round_over()
    assert env.get_winner() is None


# ---------------- tests/test_core_basic.py


def kat_player_can_only_move_on_opposite_color(make):  # test_core_basic.py:9
    env = make(5, 5)
    env.player_x, env.player_y = 2, 2
    env._set_tile(3, 2, WHITE)
    env._set_tile(1, 2, BLACK)
    assert env.try_move_player(RIGHT) is True
    assert (env.player_x, env.player_y) == (3, 2)
    env.player_x, env.player_y = 2, 2
    assert env.try_move_player(LEFT) is False
    assert (env.player_x, env.player_y) == (2, 2)


def kat_step_with_none_action_updates_bullets_only(make):  # test_core_basic.py:87
    env = make(10, 10)
    env.player2.x, env.player2.y = 0, env.height - 1
    env.player_x, env.player_y = 5, 5
    env.spawn_bullet(RIGHT)
    before = env.get_bullets()
    assert len(before) == 1
    dest_x, dest_y = before[0].x + 1, before[0].y
    env._set_tile(dest_x, dest_y, BLACK)
    tile_before = env._get_tile(dest_x, dest_y)
    env.step(NONE)
    assert (env.player_x, env.player_y) == (5, 5)
    after = env.get_bullets()
    assert len(after) == 1
    assert (after[0].x, after[0].y) == (dest_x, dest_y)
    assert env._get_tile(dest_x, dest_y) != tile_before


def kat_move_out_of_bounds_fails(make):  # test_core_basic.py:131
    env = make(5, 5)
    env.player_x, env.player_y = 0, 0
    assert env.try_move_player(UP) is False
    assert (env.player_x, env.player_y) == (0, 0)
    assert env.try_move_player(LEFT) is False
    assert (env.player_x, env.player_y) == (0, 0)
    env.player_x, env.player_y = env.width - 1, env.height - 1
    assert env.try_move_player(DOWN) is False
    assert env.try_move_player(RIGHT) is False
    assert (env.player_x, env.player_y) == (env.width - 1, env.height - 1)


# ---------------- tests/test_core_shooting.py


def kat_shoot_flips_tiles_in_line_until_out_of_bounds(make):  # test_core_shooting.py:8
    env = make(5, 1)
    W = env.width
    env.player2.x, env.player2.y = 0, env.height - 1
    env.player_x, env.player_y = W - 3, 0
    for x in range(W):
        env._set_tile(x, 0, BLACK)
    env.step(SHOOT(RIGHT))
    for _ in range(3):
        env.update_bullets()
    assert env._get_tile(W - 2, 0) != BLACK
    assert env._get_tile(W - 1, 0) != BLACK
    for x in range(W - 2):
        assert env._get_tile(x, 0) == BLACK
    assert len(env.bullets) == 0


def kat_bullet_removed_when_out_of_bounds(make):  # test_core_shooting.py:46
    env = make(5, 5)
    W = env.width
    env.player_x, env.player_y = W - 2, 2
    env.spawn_bullet(RIGHT)
    b = env.get_bullets()
    assert len(b) == 1 and b[0].x == W - 2
    env.update_bullets()
    b = env.get_bullets()
    assert len(b) == 1 and b[0].x == W - 1
    env.update_bullets()
    assert len(env.get_bullets()) == 0


def kat_multiple_bullets_update_independently(make):  # test_core_shooting.py:72
    env = make(10, 10)
    env.player2.x, env.player2.y = 0, env.height - 1
    env.player_x, env.player_y = 5, 5
    env.spawn_bullet(LEFT)
    env.spawn_bullet(RIGHT)
    assert len(env.get_bullets()) == 2
    env._set_tile(4, 5, BLACK)
    env._set_tile(6, 5, BLACK)
    env.step(NONE)
    after = env.get_bullets()
    assert len(after) == 2
    lb = next(b for b in after if b.dir == LEFT)
    rb = next(b for b in after if b.dir == RIGHT)
    assert (lb.x, lb.y) == (4, 5)
    assert (rb.x, rb.y) == (6, 5)
    assert env._get_tile(4, 5) == WHITE
    assert env._get_tile(6, 5) == WHITE


def kat_step_shoot_spawns_bullet_and_updates_grid(make):  # test_core_shooting.py:127
    env = make(10, 10)
    env.player2.x, env.player2.y = 0, env.height - 1
    env.player_x, env.player_y = 5, 5
    n0 = len(env.get_bullets())
    env._set_tile(6, 5, BLACK)
    env.step(SHOOT(RIGHT))
    after = env.get_bullets()
    assert len(after) == n0 + 1
    assert env._get_tile(6, 5) == WHITE
    assert (after[0].x, after[0].y, after[0].dir) == (6, 5, RIGHT)


def kat_bullet_flips_tile_at_new_position_not_old(make):  # test_core_shooting.py:163
    env = make(10, 10)
    env.player2.x, env.player2.y = 0, env.height - 1
    env.player_x, env.player_y = 5, 5
    env._set_tile(5, 5, BLACK)
    env._set_tile(6, 5, BLACK)
    env.step(SHOOT(RIGHT))
    assert env._get_tile(5, 5) == BLACK
    assert env._get_tile(6, 5) == WHITE


# ---------------- verify_env_logic.py


def kat_verify_coordinates(make):  # verify_env_logic.py:5-39
    env = make(10, 10)
    env.player1.x, env.player1.y = 5, 5
    env.player2.x, env.player2.y = 5, 2
    obs, extra = env.observation(P1)
    assert obs.shape == (12, env.height, env.width)
    assert obs[2, 5, 5] == 1.0
    assert obs[3, 2, 5] == 1.0
    assert obs[2].sum() == 1.0 and obs[3].sum() == 1.0
    assert (obs[0] + obs[1] == 1.0).all()
    assert list(extra) == [1.0, 1.0, 1.0, 1.0]


def kat_verify_actions(make):  # verify_env_logic.py:41-71
    env = make(10, 10)
    env.player1.x, env.player1.y = 5, 5
    env.player2.alive = False
    env.step_players(5, NONE)  # action id 5 = SHOOT UP
    b = env.get_bullets()
    assert len(b) == 1
    assert (b[0].x, b[0].y, b[0].dir) == (5, 4, UP)


# ---------------- SURVEY.md section 7 "hard part 1": list order is observable (core.py:453,473)


def kat_first_bullet_in_list_order_survives_a_same_owner_merge(make):
    env = make(10, 10)
    env.player1.x, env.player1.y = 0, env.height - 1
    env.player2.x, env.player2.y = 1, env.height - 1
    env.bullets = [Bullet(3, 4, RIGHT, P1), Bullet(4, 3, DOWN, P1)]
    env.update_bullets()
    assert env.bullets == [Bullet(4, 4, RIGHT, P1)]
    env.bullets = [Bullet(4, 3, DOWN, P1), Bullet(3, 4, RIGHT, P1)]
    env.update_bullets()
    assert env.bullets == [Bullet(4, 4, DOWN, P1)]


def kat_head_on_adjacent_bullets_swap_without_cancelling(make):  # SURVEY.md S6 [probed]
    env = make(10, 10)
    env.player1.x, env.player1.y = 0, env.height - 1
    env.player2.x, env.player2.y = 1, env.height - 1
    env.bullets = [Bullet(3, 4, RIGHT, P1), Bullet(4, 4, LEFT, P2)]
    env.update_bullets()
    assert env.bullets == [Bullet(4, 4, RIGHT, P1), Bullet(3, 4, LEFT, P2)]


def kat_mutual_adjacent_shots_kill_both(make):  # SURVEY.md S6 [probed]: tie
    env = make(10, 10)
    env.player1.x, env.player1.y = 4, 4
    env.player2.x, env.player2.y = 5, 4
    env.player1.ammo = env.player2.ammo = MAX_AMMO
    env.step_players(SHOOT(RIGHT), SHOOT(LEFT))
    assert not env.player1.alive and not env.player2.alive
    assert env.is_round_over() and env.get_winner() is None


ALL_KATS = sorted(k for k in globals() if k.startswith("kat_"))
