"""inv_scripted_actions on the GPU, and the mixed-opponent trainer and two-seat evaluator built on it.

Seat 1 is the simulator's own dummy: a selfplay handle fed its ids must reproduce a dummy-mode
handle bit for bit. Seat 0 must equal the C oracle's dummy on the player-swapped, colour-inverted
state with the seat-0 counter's draws injected."""
import csv
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _sim(n, mode, difficulty="hard", max_steps=60, seed=11, env_id_base=0):
    from inversus_b200 import BatchedInversus
    sim = BatchedInversus(n, mode, difficulty, max_steps, seed=seed, device=0, obs_dtype="none", auto_reset=True,
                          env_id_base=env_id_base)
    sim.reset()
    return sim


def _outputs(sim):
    return [sim.packed_state, sim.reward, sim.done, sim.info, sim.episode_steps, sim.episode_return, sim.extra]


# ------------------------------------------------------------------------------------------ seat 1
@pytest.mark.parametrize("difficulty", ["easy", "hard"])
@pytest.mark.parametrize("n,seed,base", [(1, 3, 0), (131, 4, 17), (4096, 5, 1000),
                                         (257, 0xFEDC_BA98_7654_3210, 0xFFFFFFFF - 257)])
def test_seat1_ids_make_a_selfplay_handle_reproduce_the_dummy_mode(n, seed, base, difficulty):
    from inversus_b200.evaluate import scripted_actions
    from inversus_b200.fused_ops import PackedStates
    dummy = _sim(n, "dummy", difficulty, seed=seed, env_id_base=base)
    sp = _sim(n, "selfplay", difficulty, seed=seed, env_id_base=base)
    g = torch.Generator(device="cuda").manual_seed(n)
    a1 = torch.randint(0, 13, (600, n), device="cuda", generator=g).to(torch.int8)
    a2 = torch.empty(n, dtype=torch.int8, device="cuda")
    view = PackedStates(sp.packed_state, 1)
    dones = 0
    for t in range(600):
        scripted_actions(view, seat=1, difficulty=difficulty, seed=seed, gid_base=base, out=a2)
        dummy.step(a1[t])
        sp.step(a1[t], a2)
        for x, y in zip(_outputs(dummy), _outputs(sp)):
            assert torch.equal(x, y), t
        dones += int(dummy.done.sum())
    assert dones > 0 and dummy.poll_status() == 0 and sp.poll_status() == 0
    dummy.close()
    sp.close()


# ------------------------------------------------------------------------------------------ seat 0
@pytest.mark.parametrize("difficulty", [0, 1])
def test_seat0_equals_the_oracle_on_gpu_states(difficulty):
    from oracle import oracle as orc
    from test_scripted_host import _oracle_env, _seat0_draws
    from inversus_b200.evaluate import scripted_actions
    from inversus_b200.fused_ops import PackedStates
    n, seed, base = 512, 0x0123_4567_89AB_CDEF, 77
    sim = _sim(n, "selfplay", seed=seed, env_id_base=base)
    rs = np.random.RandomState(difficulty)
    checked = 0
    for t in range(40):
        if t % 8 == 7:
            got = scripted_actions(PackedStates(sim.packed_state, 0), seat=0, difficulty=difficulty, seed=seed,
                                   gid_base=base).cpu().numpy()
            st = sim.export_state()
            want = [orc.lib().orc_dummy_policy(C.byref(_oracle_env(
                orc, st[i:i + 1], base + i, difficulty, True,
                _seat0_draws(orc, base + i, int(st["episode"][i]), int(st["step_count"][i]), seed), seed)))
                for i in range(n)]
            assert np.array_equal(got, np.array(want, np.int8)), t
            checked += 1
        sim.step(torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda(),
                 torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda())
    assert checked == 5
    sim.close()


@pytest.mark.parametrize("seat", [0, 1])
def test_chunks_with_matching_gid_base_equal_one_call(seat):
    from inversus_b200.evaluate import scripted_actions
    from inversus_b200.fused_ops import PackedStates
    n, base, seed = 70001, 12345, 99
    sim = _sim(n, "selfplay", seed=seed, env_id_base=base)
    rs = np.random.RandomState(3)
    for _ in range(5):
        sim.step(torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda(),
                 torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda())
    view = PackedStates(sim.packed_state, seat)
    whole = scripted_actions(view, seat=seat, difficulty="hard", seed=seed, gid_base=base)
    parts = torch.empty_like(whole)
    for lo, hi in ((0, 1), (1, 4096), (4096, 65539), (65539, n)):
        scripted_actions(view.chunk(lo, hi), seat=seat, difficulty="hard", seed=seed, gid_base=base + lo,
                         out=parts[lo:hi])
    assert torch.equal(whole, parts)
    assert len(set(whole.tolist())) >= 7
    sim.close()


def test_invalid_arguments_name_the_entry_point():
    from inversus_b200 import _capi
    lib = _capi.load()
    sim = _sim(8, "selfplay")
    out = torch.empty(8, dtype=torch.int8, device="cuda")
    p, o = sim.packed_state.data_ptr(), out.data_ptr()
    good = dict(packed=p, stride=8, count=8, gid_base=0, seed=1, seat=1, difficulty=1, out=o)
    bad = [dict(count=-1), dict(packed=None), dict(out=None), dict(stride=7), dict(seat=2), dict(seat=-1),
           dict(difficulty=2), dict(gid_base=-1), dict(gid_base=(1 << 32) - 7)]
    for change in bad:
        a = {**good, **change}
        handle = C.c_void_p()
        assert lib.inv_create(C.byref(_capi.Config(n_envs=0)), C.byref(handle)) == _capi.ERR_INVALID_ARG
        rc = lib.inv_scripted_actions(a["packed"], a["stride"], a["count"], a["gid_base"], a["seed"], a["seat"],
                                      a["difficulty"], a["out"], None)
        msg = _capi.last_error()
        assert rc == _capi.ERR_INVALID_ARG and msg.startswith("inv_scripted_actions:"), (change, rc, msg)
    a = {**good, "gid_base": (1 << 32) - 8}  # the last valid base
    assert lib.inv_scripted_actions(a["packed"], a["stride"], a["count"], a["gid_base"], a["seed"], a["seat"],
                                    a["difficulty"], a["out"], None) == _capi.OK
    assert lib.inv_scripted_actions(p, 8, 0, 0, 1, 0, 0, o, None) == _capi.OK
    torch.cuda.synchronize()
    sim.close()


# ------------------------------------------------------------------------------------------ trainer
KEYS = ("episodes", "win_rate", "avg_reward", "avg_ep_len")


@pytest.mark.parametrize("cuda_graph", [False, True])
def test_scripted_mix_trains_exactly_like_vs_dummy(tmp_path, cuda_graph):
    from inversus_b200.training import train
    kw = dict(num_envs=64, total_steps=64 * 128, rollout_steps=128, seed=5, max_episode_steps=60, save=False,
              quiet=True, cuda_graph=cuda_graph)
    mix = train("selfplay", log_dir=str(tmp_path / "mix"), opponent_mix="hard=1", **kw)
    ref = train("vs_dummy", log_dir=str(tmp_path / "ref"), opponent_difficulty="hard", **kw)
    assert mix["episodes"] > 0
    assert [mix[k] for k in KEYS] == [ref[k] for k in KEYS]
    assert mix["per_opponent"]["hard"]["episodes"] == mix["episodes"]
    assert mix["per_opponent"]["hard"]["wins"] == round(ref["last_window"]["wins"])


def test_four_slot_mix_logs_every_episode_once_per_window(tmp_path):
    from inversus_b200.training import train
    n = 256
    out = train("selfplay", n, n * 128 * 3, str(tmp_path), rollout_steps=128, seed=9, max_episode_steps=60,
                save=False, quiet=True, cuda_graph=True, opponent_mix="easy=0.25,hard=0.25,latest=0.25,pool=0.25",
                pool_size=2)
    assert out["cuda_graph"]
    assert [name for name, _, _ in out["opponent_ranges"]] == ["easy", "hard", "latest", "pool[0]", "pool[1]"]
    with open(tmp_path / "training_log.csv") as f:
        train_rows = list(csv.DictReader(f))
    with open(tmp_path / "opponent_log.csv") as f:
        opp_rows = list(csv.DictReader(f))
    assert len(train_rows) == 3
    prev = 0
    for row in train_rows:
        window = [r for r in opp_rows if r["step"] == row["step"]]
        assert {r["opponent"] for r in window} == {"easy", "hard", "latest", "pool[0]", "pool[1]"}
        assert sum(int(r["episodes"]) for r in window) == int(row["episode"]) - prev
        for r in window:
            assert int(r["wins"]) + int(r["losses"]) + int(r["draws"]) == int(r["episodes"])
        prev = int(row["episode"])
    assert sum(v["episodes"] for v in out["per_opponent"].values()) == out["episodes"]


# ------------------------------------------------------------------------------------------ evaluator
def _hand_loop_both_seats(pol, opp, N, K, max_steps, seed):
    """scripted_actions + select_actions + step + the numpy tally, seats split at ceil(N / 2)."""
    from test_cuda_evaluate import _NumpyTally
    from inversus_b200.evaluate import scripted_actions, select_actions
    from inversus_b200.fused_ops import PackedStates
    sim = _sim(N, "selfplay", "easy", max_steps, seed)
    split = -(-N // 2)
    ref = _NumpyTally(N, K)
    for _ in range(K * max_steps + 1):
        v1, v2 = PackedStates(sim.packed_state, 0), PackedStates(sim.packed_state, 1)
        a1 = torch.cat([select_actions(pol(v1)[:split].contiguous(), v1.chunk(0, split), seed=seed, seat=0),
                        scripted_actions(v1.chunk(split, N), seat=0, difficulty=opp, seed=seed, gid_base=split)])
        a2 = torch.cat([scripted_actions(v2.chunk(0, split), seat=1, difficulty=opp, seed=seed),
                        select_actions(pol(v2)[split:].contiguous(), v2.chunk(split, N), seed=seed, seat=1,
                                       gid_base=split)])
        sim.step(a1, a2)
        if ref.add(sim) == 0:
            break
    assert sim.poll_status() == 0
    sim.close()
    c = ref.counts
    seat1 = [int(x) for x in c[:, :split].sum(1)]
    l, w, d, s = c[:, split:].sum(1)
    return seat1, [int(w), int(l), int(d), int(s)], ref.ret[:split].sum()


@pytest.mark.parametrize("cuda_graph", [False, True])
def test_both_seats_against_the_dummy_equal_a_hand_written_loop(cuda_graph):
    from test_cuda_evaluate import Scripted
    from inversus_b200.evaluate import evaluate, play_shard
    N, K, T, seed = 1537, 2, 120, 8
    pol = Scripted(1)
    res = evaluate(pol, "hard", N, K, seed=seed, max_episode_steps=T, cuda_graph=cuda_graph, act_chunk=1000,
                   seats="both")
    seat1, seat2, rsum = _hand_loop_both_seats(pol, "hard", N, K, T, seed)
    split = -(-N // 2)
    for name, want in (("p1", seat1), ("p2", seat2)):
        got = res["per_seat"][name]
        assert [got["wins"], got["losses"], got["draws"]] == want[:3], (name, got, want)
        assert got["mean_episode_length"] == want[3] / got["episodes"]
    assert res["per_seat"]["p1"]["episodes"] == split * K and res["per_seat"]["p2"]["episodes"] == (N - split) * K
    assert res["mean_return"] == pytest.approx(rsum / (split * K), rel=1e-12)
    # the P1 row is what a seats="p1" run over the same ids reports
    p1 = play_shard(pol, "hard", N, K, 0, split, seed=seed, max_episode_steps=T, cuda_graph=cuda_graph)
    assert p1["seats"][0].tolist() == seat1 and int(p1["seats"][1].abs().sum()) == 0


def test_cli_plays_both_seats_from_a_checkpoint(tmp_path):
    from inversus_b200 import InversusCNNPolicy
    torch.manual_seed(0)
    model = tmp_path / "policy.pt"
    torch.save(InversusCNNPolicy().state_dict(), model)
    r = subprocess.run([sys.executable, "-m", "inversus_b200.evaluate", "--model", str(model), "--opponent", "hard",
                        "--num_envs", "4096", "--episodes_per_env", "2", "--seats", "both", "--seed", "7"],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 1
    res = json.loads(lines[0])
    assert res["per_seat"]["p1"]["episodes"] == res["per_seat"]["p2"]["episodes"] == 4096
    assert res["episodes"] == 8192 and res["mean_return"] is not None and res["args"]["seats"] == "both"
