"""The evaluator on the GPU: inv_select_actions against torch.argmax and a Python restatement of its
counter-based sampling, inv_episode_tally against a numpy tally, evaluate() against a hand-written
loop, its invariance to chunking / sharding, and the command line."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = 0xFFFFFFFF


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _sim(n, mode="dummy", difficulty="hard", max_steps=500, seed=11, env_id_base=0):
    from inversus_b200 import BatchedInversus
    sim = BatchedInversus(n, mode, difficulty, max_steps, seed=seed, device=0, obs_dtype="none", auto_reset=True,
                          env_id_base=env_id_base)
    sim.reset()
    return sim


def _advance(sim, steps, seed=0):
    """Random actions for a few steps so that the envs' (episode, step_count) words differ."""
    rs = np.random.RandomState(seed)
    for _ in range(steps):
        a = torch.from_numpy(rs.randint(0, 13, sim.num_envs).astype(np.int8)).cuda()
        a2 = torch.from_numpy(rs.randint(0, 13, sim.num_envs).astype(np.int8)).cuda() if sim.opponent_type == "selfplay" else None
        sim.step(a, a2)
    assert sim.poll_status() == 0


# ------------------------------------------------------------------------------------------ selection
@pytest.mark.parametrize("n", [1, 131, 65539])
def test_greedy_is_torch_argmax(n):
    from inversus_b200.evaluate import select_actions
    from inversus_b200.fused_ops import PackedStates
    sim = _sim(n)
    ps = PackedStates(sim.packed_state, 0)
    g = torch.Generator(device="cuda").manual_seed(n)
    for logits in (torch.randn(n, 13, device="cuda", generator=g) * 4,
                   torch.randint(-2, 3, (n, 13), device="cuda", generator=g).float()):  # many ties
        a = select_actions(logits, ps, seed=5, greedy=True)
        assert a.dtype == torch.int8 and torch.equal(a.long(), logits.argmax(1))
    sim.close()


@pytest.mark.parametrize("greedy", [True, False])
def test_non_finite_rows_give_an_invalid_action(greedy):
    from inversus_b200.constants import STATUS_INVALID_ACTION
    from inversus_b200.evaluate import select_actions
    from inversus_b200.fused_ops import PackedStates
    n = 131
    sim = _sim(n)
    logits = torch.randn(n, 13, device="cuda")
    logits[3, 5] = float("nan")
    logits[7, 12] = float("inf")
    logits[9] = float("-inf")
    logits[11, :12] = float("-inf")  # one finite logit left: a valid row
    a = select_actions(logits, PackedStates(sim.packed_state, 0), seed=5, greedy=greedy).cpu()
    bad = {3, 7, 9}
    assert all(int(a[i]) == -1 for i in bad) and int(a[11]) == 12
    assert all(0 <= int(a[i]) <= 12 for i in range(n) if i not in bad)
    assert sim.poll_status() == 0
    sim.step(a.cuda())
    assert sim.poll_status() & STATUS_INVALID_ACTION
    sim.close()


def _philox_r0(gid, episode, step, seat, seed):
    from ref_harness import philox4x32_10
    return philox4x32_10((gid & M32, episode & M32, step & M32, 0x80000000 | seat), (seed & M32, seed >> 32))[0]


def _sample_reference(logits, st, gid_base, seed, seat):
    """Section 1 of the evaluator design restated: fp32 inverse CDF of one Philox draw per row.
    Returns (ids, clear) where `clear` marks rows whose u*S is not within 1e-5*S of a boundary."""
    l = logits.astype(np.float64)
    e = np.exp(l - l.max(1, keepdims=True))
    S = e.sum(1)
    cum = np.cumsum(e, 1)
    r = np.array([_philox_r0(gid_base + i, int(st["episode"][i]), int(st["step_count"][i]), seat, seed)
                  for i in range(len(l))], np.uint32)
    t = r.astype(np.float32).astype(np.float64) * 2.0 ** -32 * S
    below = t[:, None] < cum
    ids = np.where(below.any(1), below.argmax(1), 12 - np.argmax((e > 0)[:, ::-1], 1))
    clear = np.abs(t[:, None] - cum).min(1) > 1e-5 * S
    return ids, clear


@pytest.mark.parametrize("seat", [0, 1])
def test_sampling_matches_the_python_restatement(seat):
    from inversus_b200.evaluate import select_actions
    from inversus_b200.fused_ops import PackedStates
    n, seed, base = 65539, 0x123456789AB, 1000
    sim = _sim(n, "selfplay", seed=seed, env_id_base=base)
    _advance(sim, 23)
    st = sim.export_state()
    assert len(np.unique(st["step_count"])) > 5 and st["episode"].max() > 0
    g = torch.Generator(device="cuda").manual_seed(seat)
    logits = torch.randn(n, 13, device="cuda", generator=g) * 2
    logits[::7, 4] = float("-inf")  # impossible actions
    a = select_actions(logits, PackedStates(sim.packed_state, seat), seed=seed, seat=seat, greedy=False,
                       gid_base=base).cpu().numpy()
    want, clear = _sample_reference(logits.cpu().numpy(), st, base, seed, seat)
    assert clear.mean() >= 0.999, clear.mean()
    assert np.array_equal(a[clear], want[clear])
    assert not (a[::7] == 4).any()
    sim.close()


def test_sampling_follows_the_softmax():
    from scipy.stats import chisquare
    from inversus_b200.evaluate import select_actions
    from inversus_b200.fused_ops import PackedStates
    n = 1 << 20
    sim = _sim(n, seed=3)
    row = torch.tensor([0.0, 1.0, -1.0, 2.0, 0.5, -0.5, 0.0, 1.5, -2.0, 0.25, 0.75, -1.5, 1.0], device="cuda")
    logits = row.expand(n, 13).contiguous()
    a = select_actions(logits, PackedStates(sim.packed_state, 0), seed=3, greedy=False)
    counts = torch.bincount(a.long(), minlength=13).cpu().numpy()
    p = torch.softmax(row.double(), 0).cpu().numpy()
    assert chisquare(counts, p * n).pvalue > 1e-3
    sim.close()


def test_seats_draw_differently_and_chunks_equal_the_whole():
    from inversus_b200.evaluate import select_actions
    from inversus_b200.fused_ops import PackedStates
    n, seed, base = 10007, 99, 77
    sim = _sim(n, "selfplay", seed=seed, env_id_base=base)
    _advance(sim, 9)
    ps = PackedStates(sim.packed_state, 0)
    logits = torch.zeros(n, 13, device="cuda")
    s0 = select_actions(logits, ps, seed=seed, seat=0, greedy=False, gid_base=base)
    s1 = select_actions(logits, ps, seed=seed, seat=1, greedy=False, gid_base=base)
    assert (s0 == s1).float().mean().item() < 0.15  # independent uniform draws agree 1 time in 13
    logits = torch.randn(n, 13, device="cuda")
    whole = select_actions(logits, ps, seed=seed, seat=1, greedy=False, gid_base=base)
    h = 4099
    lo = select_actions(logits[:h], ps.chunk(0, h), seed=seed, seat=1, greedy=False, gid_base=base)
    hi = select_actions(logits[h:], ps.chunk(h, n), seed=seed, seat=1, greedy=False, gid_base=base + h)
    assert torch.equal(whole, torch.cat([lo, hi]))
    sim.close()


# ------------------------------------------------------------------------------------------ tally
class _NumpyTally:
    def __init__(self, n, quota):
        self.quota = quota
        self.counts = np.zeros((4, n), np.int64)
        self.ret = np.zeros(n, np.float64)

    def add(self, sim):
        done = sim.done.cpu().numpy().astype(bool)
        info = sim.info.cpu().numpy()
        steps = sim.episode_steps.cpu().numpy()
        ret = sim.episode_return.cpu().numpy()
        ep = sim.export_state()["episode"].astype(np.uint32)
        m = done & ((ep - np.uint32(1)) < self.quota)
        win, lose = (info & 4) != 0, (info & 8) != 0
        self.counts[0] += m & win
        self.counts[1] += m & lose
        self.counts[2] += m & ~win & ~lose
        self.counts[3] += np.where(m, steps, 0)
        self.ret[m] += ret[m]
        return int((ep < self.quota).sum())


def test_tally_equals_a_numpy_tally():
    from inversus_b200.evaluate import episode_tally
    n, K, T = 4096, 2, 60
    sim = _sim(n, max_steps=T, seed=21)
    counts = torch.zeros((4, n), dtype=torch.int32, device="cuda")
    ret = torch.zeros(n, dtype=torch.float64, device="cuda")
    remaining = torch.zeros(1, dtype=torch.int32, device="cuda")
    ref = _NumpyTally(n, K)
    rs = np.random.RandomState(4)
    for _ in range(K * T + 1):
        sim.step(torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda())
        episode_tally(sim, K, counts, ret, remaining)
        left = ref.add(sim)
        assert int(remaining.item()) == left
    assert left == 0
    assert np.array_equal(counts.cpu().numpy(), ref.counts)
    assert np.array_equal(ret.cpu().numpy().view(np.uint64), ref.ret.view(np.uint64))
    c = ref.counts
    assert (c[:3].sum(0) == K).all() and c[1].sum() > 0 and c[2].sum() > 0
    with pytest.raises(ValueError):
        episode_tally(sim, (1 << 31) // T + 1, counts, ret, remaining)
    sim.close()


# ------------------------------------------------------------------------------------------ evaluate
class Scripted:
    """A batch-invariant stand-in for a network: logits = integer weights . observation (0/1 planes
    rebuilt from the packed state), so every product and sum is exact in any order or batch split."""

    def __init__(self, seed):
        from inversus_b200 import BatchedInversus
        g = torch.Generator(device="cuda").manual_seed(seed)
        self.w = torch.randint(-2, 3, (13, 1800), device="cuda", generator=g).float()
        self.helper = BatchedInversus(1, device=0, obs_dtype="f32")  # a handle for inv_obs_from_packed
        self.__name__ = f"scripted{seed}"

    def __call__(self, ps):
        from inversus_b200 import _capi
        from inversus_b200.fused_ops import _packed_args
        ptr, stride, count = _packed_args(ps)
        obs = torch.empty((count, 1800), device="cuda")
        extra = torch.empty((count, 4), device="cuda")
        _capi.check(self.helper._lib.inv_obs_from_packed(self.helper._h.ptr, ptr, stride, count, ps.view, 0,
                                                         obs.data_ptr(), extra.data_ptr(),
                                                         torch.cuda.current_stream().cuda_stream))
        return (obs @ self.w.T) * 0.5  # integers below 2^24: exact whatever the summation order


def _hand_loop(pol, opp, N, K, max_steps, seed):
    """BatchedInversus.step + the callables + torch.argmax + the numpy tally."""
    from inversus_b200.fused_ops import PackedStates
    h2h = not isinstance(opp, str)
    sim = _sim(N, "selfplay" if h2h else "dummy", "easy" if h2h else opp, max_steps, seed)
    split = -(-N // 2) if h2h else N
    p1_is_pol = (torch.arange(N, device="cuda") < split)[:, None]
    ref = _NumpyTally(N, K)
    for _ in range(K * max_steps + 1):
        v1, v2 = PackedStates(sim.packed_state, 0), PackedStates(sim.packed_state, 1)
        if h2h:
            a1 = torch.where(p1_is_pol, pol(v1), opp(v1)).argmax(1)
            a2 = torch.where(p1_is_pol, opp(v2), pol(v2)).argmax(1)
            sim.step(a1.to(torch.int8), a2.to(torch.int8))
        else:
            sim.step(pol(v1).argmax(1).to(torch.int8))
        if ref.add(sim) == 0:
            break
    assert sim.poll_status() == 0
    sim.close()
    c = ref.counts
    seat1 = [int(x) for x in c[:, :split].sum(1)]
    l, w, d, s = c[:, split:].sum(1)
    return seat1, [int(w), int(l), int(d), int(s)], ref.ret.sum()


def _strip(res):
    return {k: v for k, v in res.items() if k not in ("wall_s", "env_steps_per_s", "episodes_per_s")}


@pytest.mark.parametrize("cuda_graph", [False, True])
@pytest.mark.parametrize("opponent", ["hard", "policy"])
def test_evaluate_equals_a_hand_written_loop(opponent, cuda_graph):
    from inversus_b200.evaluate import evaluate
    N, K, T, seed = 1536, 2, 120, 8
    pol = Scripted(1)
    opp = Scripted(2) if opponent == "policy" else opponent
    res = evaluate(pol, opp, N, K, seed=seed, max_episode_steps=T, cuda_graph=cuda_graph, act_chunk=1000)
    seat1, seat2, rsum = _hand_loop(pol, opp, N, K, T, seed)
    for name, want in (("p1", seat1), ("p2", seat2)):
        got = res["per_seat"][name]
        assert [got["wins"], got["losses"], got["draws"]] == want[:3], (name, got, want)
        if got["episodes"]:
            assert got["mean_episode_length"] == want[3] / got["episodes"]
    assert res["episodes"] == N * K == res["wins"] + res["losses"] + res["draws"]
    assert res["wins"] == seat1[0] + seat2[0] and res["draws"] == seat1[2] + seat2[2]
    if opponent == "hard":
        assert res["per_seat"]["p2"]["episodes"] == 0 and res["mean_return"] == pytest.approx(rsum / (N * K), rel=1e-12)
    else:
        assert res["per_seat"]["p1"]["episodes"] == res["per_seat"]["p2"]["episodes"] == N * K // 2
        assert res["mean_return"] is None
    assert res["args"]["cuda_graph"] is cuda_graph and res["env_steps"] % N == 0


@pytest.mark.parametrize("actions", ["greedy", "sample"])
def test_evaluate_is_invariant_to_chunking_and_sharding(actions):
    from inversus_b200.evaluate import evaluate, play_shard
    N, K, T, seed = 4097, 2, 100, 5
    pol, opp = Scripted(3), Scripted(4)
    kw = dict(actions=actions, seed=seed, max_episode_steps=T)
    a = evaluate(pol, opp, N, K, act_chunk=65536, **kw)
    b = evaluate(pol, opp, N, K, act_chunk=65536, **kw)
    assert _strip(a) == _strip(b)
    c = evaluate(pol, opp, N, K, act_chunk=1024, **kw)
    for key in ("wins", "losses", "draws", "per_seat", "mean_episode_length"):
        assert a[key] == c[key], key
    whole = play_shard(pol, opp, N, K, 0, N, **kw)["seats"]
    h = 2048  # the seat boundary, ceil(N / 2) = 2049, lies inside the second shard
    halves = play_shard(pol, opp, N, K, 0, h, **kw)["seats"] + play_shard(pol, opp, N, K, h, N - h, **kw)["seats"]
    assert torch.equal(whole, halves)
    assert int(whole[:, :3].sum()) == N * K
    d = evaluate(pol, "easy", N, K, **kw)
    assert d["episodes"] == N * K == d["wins"] + d["losses"] + d["draws"]


# ------------------------------------------------------------------------------------------ CLI
FIELDS = {"episodes", "wins", "losses", "draws", "win_rate", "win_rate_ci95", "score", "score_ci95", "elo", "elo_ci95",
          "mean_episode_length", "mean_return", "per_seat", "env_steps", "wall_s", "env_steps_per_s", "episodes_per_s",
          "args"}


def test_cli_with_a_checkpoint(tmp_path):
    from inversus_b200 import InversusCNNPolicy
    torch.manual_seed(0)
    model = tmp_path / "policy.pt"
    torch.save(InversusCNNPolicy().state_dict(), model)

    def run(opponent, actions, tag):
        out = tmp_path / f"{tag}.json"
        r = subprocess.run([sys.executable, "-m", "inversus_b200.evaluate", "--model", str(model), "--opponent", opponent,
                            "--num_envs", "4096", "--episodes_per_env", "2", "--actions", actions, "--seed", "7",
                            "--json", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        res = json.loads(out.read_text())
        assert res == line and FIELDS <= set(res) and set(res["per_seat"]) == {"p1", "p2"}
        assert res["episodes"] == 4096 * 2 == res["wins"] + res["losses"] + res["draws"]
        return res

    g1 = run("hard", "greedy", "g1")
    assert g1["mean_return"] is not None and g1["per_seat"]["p2"]["episodes"] == 0
    g2 = run("hard", "greedy", "g2")
    assert [g1[k] for k in ("wins", "losses", "draws", "mean_episode_length")] == \
           [g2[k] for k in ("wins", "losses", "draws", "mean_episode_length")]
    run("hard", "sample", "s1")
    for actions in ("greedy", "sample"):
        self_play = run(str(model), actions, "self_" + actions)
        assert self_play["mean_return"] is None
        assert self_play["per_seat"]["p1"]["episodes"] == self_play["per_seat"]["p2"]["episodes"] == 4096
