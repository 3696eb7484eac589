"""CPU checks of the scripted player as a handle-free producer of action ids (inv_scripted_actions)
and of what is built on it: the device function compiled for the host through the test harness
against the C oracle (seat 1 is the reference's dummy, seat 0 the same rule with the players'
roles exchanged), the same under AddressSanitizer / UBSan, the no-device failure of the entry
point, the static opponent assignment of mixed-opponent training, and the argument checks of
`--opponent_mix`, `--pool_size` and `--seats`."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from backends import HostKernelBackend

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HK = os.path.join(ROOT, "tests", "host_kernel")
SEED = 0x1234_5678_9ABC_DEF0
BASE = 4000
M32 = 0xFFFFFFFF


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def scripted_lib(tmp_path_factory):
    """tests/host_kernel/scripted_harness.cpp (harness.cpp + hk_scripted_actions), built for the host."""
    so = str(tmp_path_factory.mktemp("scripted") / "libscripted_harness.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                           "-I", HK, "-o", so, os.path.join(HK, "scripted_harness.cpp")])
    return C.CDLL(so)


def _hk_scripted(lib, b: HostKernelBackend, seat, difficulty):
    out = np.zeros(b.n, np.int8)
    assert lib.hk_scripted_actions(_p(b.planes), C.c_int64(b.n), seat, difficulty, C.c_uint64(b.seed),
                                       C.c_uint32(b.base), _p(out)) == 0
    return out


def _hk_debug_dummy(b: HostKernelBackend, difficulty):
    from inversus_b200 import _capi
    planes = b.planes.copy()
    res = np.zeros(b.n, np.uint8)
    status = np.zeros(1, np.uint32)
    b.lib().hk_debug(_p(planes), C.c_int64(b.n), _capi.PHASE_DUMMY_POLICY, 0, 0, 0, difficulty, C.c_uint64(b.seed),
                     C.c_uint32(b.base), _p(res), _p(status))
    return res.astype(np.int8)


def _states():
    """Pre-step states of random selfplay rollouts (auto-reset), plus copies with a dead P1 / P2."""
    rng = np.random.default_rng(7)
    sc = dict(n=384, mode="selfplay", difficulty="hard", max_steps=60, seed=SEED)
    b = HostKernelBackend(sc, env_id_base=BASE)
    b.reset(None)
    snaps = []
    for t in range(90):
        if t % 6 == 5:
            snaps.append(b.export_state())
        b.step(rng.integers(0, 13, b.n), rng.integers(0, 13, b.n), None, True)
    st = np.concatenate(snaps)
    dead = st[:64].copy()
    dead["p1"][:32, 4] = 0
    dead["p2"][32:, 4] = 0
    return np.concatenate([st, dead])


@pytest.fixture(scope="module")
def states():
    return _states()


def _backend_for(st):
    b = HostKernelBackend(dict(n=len(st), mode="selfplay", difficulty="hard", max_steps=60, seed=SEED),
                          env_id_base=BASE)
    b.import_state(st)
    return b


def _oracle_env(orc, row, gid, difficulty, swap, table=None, seed=SEED):
    e = orc.Env()
    orc.lib().orc_init(C.byref(e), 15, 10, 0, difficulty, 60, seed, gid)
    orc.import_state([e], row)
    e.n_bullets = 0  # the scripted rule never reads a bullet
    if swap:  # P1 <-> P2 and WHITE <-> BLACK: P1's rule is then the reference's P2 rule
        for k in range(150):
            e.grid[k] = 1 - e.grid[k]
        p0 = tuple(getattr(e.p[0], f) for f in ("x", "y", "ammo", "reload", "alive"))
        p1 = tuple(getattr(e.p[1], f) for f in ("x", "y", "ammo", "reload", "alive"))
        for f, v in zip(("x", "y", "ammo", "reload", "alive"), p1):
            setattr(e.p[0], f, v)
        for f, v in zip(("x", "y", "ammo", "reload", "alive"), p0):
            setattr(e.p[1], f, v)
    if table is not None:
        e.table = table.ctypes.data_as(C.POINTER(C.c_uint32))
    return e


def _seat0_draws(orc, gid, episode, step, seed=SEED):
    """The seat-0 counter's first 16 draws: (gid, episode, 0x80000000 | step_count, k/4)."""
    key = (seed & M32, seed >> 32)
    return np.array([v for q in range(4) for v in orc.philox4x32_10((gid, episode, 0x80000000 | step, q), key)],
                    np.uint32)


@pytest.mark.parametrize("difficulty", [0, 1])
def test_seat1_is_the_dummy_of_the_oracle_and_of_the_step(scripted_lib, states, difficulty):
    from oracle import oracle as orc
    b = _backend_for(states)
    got = _hk_scripted(scripted_lib, b, 1, difficulty)
    assert np.array_equal(got, _hk_debug_dummy(b, difficulty))
    want = np.array([orc.lib().orc_dummy_policy(C.byref(_oracle_env(orc, states[i:i + 1], BASE + i, difficulty, False)))
                     for i in range(len(states))], np.int8)
    assert np.array_equal(got, want)
    if difficulty:  # moves and shots are exercised (the easy dummy moves on 0.1 % of its calls)
        assert len(set(got.tolist())) >= 7


@pytest.mark.parametrize("difficulty", [0, 1])
def test_seat0_is_the_dummy_rule_on_the_swapped_board_with_its_own_counter(scripted_lib, states, difficulty):
    from oracle import oracle as orc
    b = _backend_for(states)
    got = _hk_scripted(scripted_lib, b, 0, difficulty)
    want = []
    for i, s in enumerate(states):
        table = _seat0_draws(orc, BASE + i, int(s["episode"]), int(s["step_count"]))
        e = _oracle_env(orc, states[i:i + 1], BASE + i, difficulty, True, table)
        want.append(orc.lib().orc_dummy_policy(C.byref(e)))
    assert np.array_equal(got, np.array(want, np.int8))
    assert np.all(got[states["p1"][:, 4] == 0] == 0)
    if difficulty:  # the shots go at P2
        assert np.any((got >= 5) & (got <= 8))


def test_scripted_actions_under_address_and_ub_sanitizers(tmp_path):
    driver = tmp_path / "driver.cpp"
    driver.write_text(r'''
#include "scripted_harness.cpp"
#include <cstdio>
#include <vector>
int main()
{
    const int64_t n = 301;
    uint64_t rng = 88172645463325252ull;
    auto next = [&]() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return (uint32_t)(rng >> 11); };
    std::vector<uint32_t> planes((size_t)n * 20, 0u);
    std::vector<inv_env_state> states(n);
    for (auto &e : states) e.episode = 0xFFFFFFFFu;
    hk_import_state(planes.data(), n, 0, n, states.data());
    std::vector<float> rew(n);
    std::vector<uint8_t> done(n), info(n), dbg(n);
    std::vector<int32_t> steps(n);
    std::vector<double> ret(n);
    std::vector<int8_t> a1(n), a2(n), s0(n), s1(n);
    uint32_t status = 0;
    hk_reset(planes.data(), n, nullptr, 0, 11, 0xFFFFFF00u, nullptr, nullptr, nullptr, nullptr, nullptr, &status);
    for (int t = 0; t < 300; ++t) {
        const int diff = t & 1;
        hk_scripted_actions(planes.data(), n, 0, diff, 11, 0xFFFFFF00u, s0.data());
        hk_scripted_actions(planes.data(), n, 1, diff, 11, 0xFFFFFF00u, s1.data());
        std::vector<uint32_t> copy = planes;
        hk_debug(copy.data(), n, INV_PHASE_DUMMY_POLICY, 0, 0, 0, diff, 11, 0xFFFFFF00u, dbg.data(), &status);
        for (int64_t i = 0; i < n; ++i) {
            if (s0[i] < 0 || s0[i] > 12 || s1[i] != (int8_t)dbg[i]) { std::printf("bad action at %d/%ld\n", t, (long)i); return 1; }
            a1[i] = (next() & 3) ? s0[i] : (int8_t)(next() % 13);
            a2[i] = (next() & 3) ? s1[i] : (int8_t)(next() % 13);
        }
        hk_step(planes.data(), n, a1.data(), a2.data(), nullptr, 1, diff, 45, 1, 11, 0xFFFFFF00u, nullptr, nullptr,
                nullptr, nullptr, rew.data(), done.data(), info.data(), steps.data(), ret.data(), &status);
    }
    if (status != 0) { std::printf("unexpected status %u\n", status); return 1; }
    std::printf("scripted sanitizer run ok\n");
    return 0;
}
''')
    exe = str(tmp_path / "scripted_san")
    cmd = ["g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-Wno-unknown-pragmas", "-fsanitize=address,undefined",
           "-fno-sanitize-recover=all", "-I", HK, "-o", exe, str(driver)]
    b = subprocess.run(cmd, capture_output=True, text=True)
    if b.returncode != 0 and ("asan" in b.stderr.lower() or "sanitize" in b.stderr.lower()):
        pytest.skip("sanitizer runtime not available: " + b.stderr[-200:])
    assert b.returncode == 0, b.stderr[-2000:]
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0, r.stdout[-1000:] + r.stderr[-3000:]
    assert "scripted sanitizer run ok" in r.stdout


@pytest.mark.parametrize("count", [4, 0])
def test_no_device_error_names_the_entry_point(count):
    from inversus_b200 import _capi
    lib = _capi.load()
    if lib.inv_device_count() > 0:
        pytest.skip("a GPU is present")
    handle = C.c_void_p()
    assert lib.inv_create(C.byref(_capi.Config(n_envs=0)), C.byref(handle)) == _capi.ERR_INVALID_ARG
    assert _capi.last_error().startswith("inv_create:")
    fake = 1 << 20  # never dereferenced: the device check comes first
    rc = lib.inv_scripted_actions(fake, 4, count, 0, 1, 1, 1, fake, None)
    msg = _capi.last_error()
    assert rc == _capi.ERR_NO_DEVICE and msg.startswith("inv_scripted_actions:") and "no CPU fallback" in msg, msg


# ------------------------------------------------------------------------------- opponent_ranges
def _slot_of_every_id(ranges, n):
    out = [None] * n
    for name, lo, hi in ranges:
        for g in range(lo, hi):
            assert out[g] is None, g
            out[g] = name
    assert None not in out
    return out


@pytest.mark.parametrize("n,mix,pool,sizes", [
    (10, "hard=0.25,latest=0.25,pool=0.5", 4, {"hard": 3, "latest": 2, "pool[0]": 2, "pool[1]": 1, "pool[2]": 1,
                                               "pool[3]": 1}),
    (7, "easy=1,hard=1,latest=1", 4, {"easy": 3, "hard": 2, "latest": 2}),
    (100, "pool=3,hard=1", 3, {"hard": 25, "pool[0]": 25, "pool[1]": 25, "pool[2]": 25}),
    (11, "latest=0.5,hard=0.3,easy=0.2", 1, {"easy": 2, "hard": 3, "latest": 6}),  # 2.2, 3.3, 5.5: the .5 wins
    (5, {"hard": 1}, 4, {"hard": 5}),
])
def test_opponent_ranges_follow_the_largest_remainder_rule_in_slot_order(n, mix, pool, sizes):
    from inversus_b200.sharding import opponent_ranges
    r = opponent_ranges(n, mix, pool)
    assert [name for name, _, _ in r] == list(sizes)
    assert {name: hi - lo for name, lo, hi in r} == sizes
    assert r[0][1] == 0 and r[-1][2] == n and all(r[k][2] == r[k + 1][1] for k in range(len(r) - 1))
    _slot_of_every_id(r, n)


@pytest.mark.parametrize("n", [1000, 4097, 65536 + 13])
def test_opponent_map_does_not_depend_on_the_gpu_count(n):
    """What each rank plays (its shard intersected with the global ranges) reassembles the same
    id -> opponent map for every world size."""
    from inversus_b200.sharding import opponent_ranges, shard_range
    r = opponent_ranges(n, "easy=0.1,hard=0.2,latest=0.3,pool=0.4", 4)
    want = _slot_of_every_id(r, n)
    for world in range(1, 9):
        got = [None] * n
        for rank in range(world):
            first, count = shard_range(n, rank, world)
            for name, lo, hi in r:
                for g in range(max(lo, first), min(hi, first + count)):
                    assert got[g] is None
                    got[g] = name
        assert got == want, world


@pytest.mark.parametrize("n,mix,pool,msg", [
    (3, "hard=0.9,latest=0.1", 4, "slot 'latest' gets 0"),
    (6, "hard=0.5,pool=0.5", 4, "fewer than pool_size"),
    (8, "medium=1", 4, "unknown slot"),
    (8, "hard=1,hard=2", 4, "twice"),
    (8, "hard=-1,latest=2", 4, "negative"),
    (8, "hard=x", 4, "not a number"),
    (8, "hard=0", 4, "sum to more than 0"),
    (8, "hard=1", 0, "pool_size must be at least 1"),
])
def test_opponent_ranges_reject_bad_mixes(n, mix, pool, msg):
    from inversus_b200.sharding import opponent_ranges
    with pytest.raises(ValueError, match=msg):
        opponent_ranges(n, mix, pool)


# ------------------------------------------------------------------------------- argument errors
def _run(module, *args):
    return subprocess.run([sys.executable, "-m", module, *args], cwd=ROOT, capture_output=True, text=True, timeout=300)


@pytest.mark.parametrize("args,message", [
    (["--mode", "vs_dummy", "--opponent_mix", "hard=1"], "only valid with mode='selfplay'"),
    (["--mode", "selfplay", "--opponent_mix", "hard=1,bogus=1"], "unknown slot"),
    (["--mode", "selfplay", "--num_envs", "4", "--opponent_mix", "pool=1", "--pool_size", "8"], "fewer than pool_size"),
    (["--mode", "selfplay", "--opponent_mix", "hard=1", "--pool_size", "0"], "pool_size must be at least 1"),
    (["--mode", "selfplay", "--pool_size", "2"], "--pool_size is only valid with --opponent_mix"),
    (["--mode", "selfplay", "--opponent_mix", "hard=1", "--precision", "fp32"], "packed-encoder"),
])
def test_training_cli_rejects_bad_opponent_mix(args, message):
    r = _run("inversus_b200.training", *args)
    assert r.returncode == 2 and message in r.stderr, r.stderr
    assert "Traceback" not in r.stderr


def test_train_rejects_bad_opponent_mix_before_touching_a_device():
    from inversus_b200.training import train
    with pytest.raises(ValueError, match="selfplay"):
        train("vs_dummy", 8, 8, opponent_mix="hard=1")
    with pytest.raises(ValueError, match="pool_size"):
        train("selfplay", 8, 8, pool_size=2)


@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory):
    import torch
    from inversus_b200 import InversusCNNPolicy
    torch.manual_seed(0)
    path = tmp_path_factory.mktemp("ckpt") / "policy.pt"
    torch.save(InversusCNNPolicy().state_dict(), path)
    return str(path)


@pytest.mark.parametrize("args,message", [
    (["--opponent", "hard", "--seats", "p2"], "invalid choice"),
    (["--opponent", "hard", "--seats", "both", "--num_envs", "1"], "seats='both' needs at least 2 envs"),
])
def test_evaluate_cli_rejects_bad_seats(checkpoint, args, message):
    r = _run("inversus_b200.evaluate", "--model", checkpoint, *args)
    assert r.returncode == 2 and message in r.stderr, r.stderr
    assert "Traceback" not in r.stderr


def test_evaluate_rejects_bad_seats_before_touching_a_device():
    from inversus_b200.evaluate import evaluate
    f = lambda ps: None  # noqa: E731
    with pytest.raises(ValueError, match="seats must be one of"):
        evaluate(f, "hard", 4, 1, seed=0, seats="p2")
    with pytest.raises(ValueError, match="needs at least 2 envs"):
        evaluate(f, "hard", 1, 1, seed=0, seats="both")
