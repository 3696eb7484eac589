"""GPU parity tests proper: the CUDA product, called through the C ABI, against
  (a) the committed golden fixtures = outputs of the live Python reference, and
  (b) the CPU oracle on fresh seeded inputs at sizes the oracle finishes in seconds.
Bar (BASELINE.json north_star): bit-exact integer state, bullets (ordered), done, info flags and
observations; float rewards within 1e-6 relative -- in fact asserted bit-exact in float32, and the
running fp64 episode return bit-exact too.
"""
import os

import numpy as np
import pytest

from golden.scenarios import SCENARIOS, compare, run_scenario

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_cuda_reproduces_reference_fixture(name):
    from backends import CudaBackend
    sc = SCENARIOS[name]
    gold = dict(np.load(os.path.join(GOLD, f"{name}.npz")))
    rec = run_scenario(CudaBackend(sc), sc)
    compare(rec, gold, float_rtol=1e-6, what=name)
    assert np.array_equal(rec["reward_f32"], gold["reward_f32"])
    assert np.array_equal(rec["reward"], gold["reward"])  # the binary64 reward of the reference, bit for bit
    assert np.array_equal(rec["episode_return"], gold["episode_return"])


FRESH = {
    "gpu_hard": dict(mode="dummy", difficulty="hard", max_steps=500, n=4096, T=600, seed=201, actions="uniform", draws="philox", resets="auto"),
    "gpu_easy": dict(mode="dummy", difficulty="easy", max_steps=120, n=2048, T=300, seed=202, actions="shooty", draws="philox", resets="auto"),
    "gpu_selfplay": dict(mode="selfplay", difficulty="hard", max_steps=200, n=2048, T=300, seed=203, actions="shooty", draws="philox", resets="auto"),
    "gpu_charge": dict(mode="dummy", difficulty="hard", max_steps=500, n=3000, T=250, seed=204, actions="charge", draws="philox", resets="auto"),
    "gpu_table": dict(mode="dummy", difficulty="hard", max_steps=90, n=1000, T=200, seed=205, actions="passive", draws="table", resets="manual"),
    "gpu_ragged": dict(mode="selfplay", difficulty="hard", max_steps=50, n=131, T=120, seed=206, actions="uniform", draws="philox", resets="manual"),
    "gpu_one": dict(mode="dummy", difficulty="hard", max_steps=30, n=1, T=100, seed=207, actions="uniform", draws="philox", resets="auto"),
    # 64-bit seed (both Philox key words in use) and a large env_id_base (see the test body)
    "gpu_bigseed": dict(mode="dummy", difficulty="hard", max_steps=45, n=700, T=150, seed=0xDEADBEEFCAFEF00D, actions="uniform", draws="philox", resets="auto"),
}


@pytest.mark.parametrize("name", sorted(FRESH))
def test_cuda_matches_oracle_on_fresh_seeds(name):
    """Differential test vs the oracle, every step, every env, every observable (incl. all 1800
    observation elements of both views). Sizes include ragged tiles (131, 3000, 1) and > 1 tile."""
    from backends import CudaBackend, OracleBackend
    sc = FRESH[name]
    base = 4_000_000_000 if name == "gpu_bigseed" else 0  # global env ids near the top of the u32 range
    want = run_scenario(OracleBackend(sc, nthreads=8, env_id_base=base), sc)
    got = run_scenario(CudaBackend(sc, env_id_base=base), sc)
    compare(got, want, float_rtol=1e-6, what=name)
    assert np.array_equal(got["reward_f32"], want["reward_f32"])
    assert np.array_equal(got["episode_return"], want["episode_return"])


def test_results_do_not_depend_on_the_shard_count():
    """Envs [0,N) on one handle == two handles owning [0,N/2) and [N/2,N) (env_id_base): the
    multi-GPU layout of DESIGN.md with no collective in the step path."""
    import torch
    from inversus_b200 import BatchedInversus
    from inversus_b200.sharding import shard_range
    n, T = 1000, 80
    rs = np.random.RandomState(5)
    acts = rs.randint(0, 13, size=(T, n)).astype(np.int8)
    whole = BatchedInversus(n, "dummy", "hard", 60, seed=9)
    parts = []
    for r in range(3):
        first, count = shard_range(n, r, 3)
        parts.append((first, count, BatchedInversus(count, "dummy", "hard", 60, seed=9, env_id_base=first)))
    whole.reset()
    for _, _, p in parts:
        p.reset()
    for t in range(T):
        whole.step(torch.from_numpy(acts[t]).cuda())
        for first, count, p in parts:
            p.step(torch.from_numpy(acts[t, first:first + count]).cuda())
    ws = whole.export_state()
    for first, count, p in parts:
        ps = p.export_state()
        for f in ws.dtype.names:
            assert np.array_equal(ws[f][first:first + count], ps[f]), f
        assert torch.equal(whole.obs[first:first + count], p.obs)
        assert torch.equal(whole.reward[first:first + count], p.reward)


@pytest.mark.parametrize("dtype", ["bf16", "u8"])
def test_narrow_observation_dtypes_are_lossless(dtype):
    """bf16 / u8 observation planes carry exactly the f32 values (all are 0 or 1)."""
    import torch
    from inversus_b200 import BatchedInversus
    n, T = 777, 40
    rs = np.random.RandomState(3)
    a = BatchedInversus(n, "selfplay", "hard", 30, seed=4, obs_dtype="f32")
    b = BatchedInversus(n, "selfplay", "hard", 30, seed=4, obs_dtype=dtype)
    a.reset(), b.reset()
    assert torch.equal(a.obs, b.obs.float())
    for _ in range(T):
        a1 = torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda()
        a2 = torch.from_numpy(rs.randint(5, 13, n).astype(np.int8)).cuda()
        a.step(a1, a2), b.step(a1, a2)
        assert torch.equal(a.obs, b.obs.float())
        assert torch.equal(a.obs_p2, b.obs_p2.float())
        assert torch.equal(a.extra, b.extra) and torch.equal(a.reward, b.reward)


def test_obs_from_packed_snapshots_matches_live_observations():
    """K3: observations rebuilt from 80-byte packed-state snapshots == the observations the step
    kernel wrote, for both views and all three dtypes."""
    import torch
    from inversus_b200 import BatchedInversus
    n = 1500
    rs = np.random.RandomState(8)
    s = BatchedInversus(n, "selfplay", "hard", 40, seed=6)
    s.reset()
    for _ in range(25):
        s.step(torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda(),
               torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda())
    snap = s.snapshot()
    for view, (g, e) in enumerate(((s.obs, s.extra), (s.obs_p2, s.extra_p2))):
        for dt in ("f32", "bf16", "u8"):
            og, oe = s.obs_from_packed(snap, view=view, obs_dtype=dt)
            assert torch.equal(og.float(), g) and torch.equal(oe, e)
    # a sub-range of a larger snapshot buffer (count < stride)
    og, oe = s.obs_from_packed(snap, view=0, count=100)
    assert torch.equal(og, s.obs[:100]) and torch.equal(oe, s.extra[:100])


def test_invalid_action_ids_are_rejected_not_ignored():
    import torch
    from inversus_b200 import BatchedInversus, MultiEnvRunner
    from inversus_b200.constants import STATUS_INVALID_ACTION
    r = MultiEnvRunner(4, "dummy", "hard", 500, seed=0)
    r.reset()
    before = r.sim.export_state()
    with pytest.raises(ValueError, match="Invalid action_id"):  # env_wrappers.py:66
        r.step(np.array([0, 13, 1, 2]))
    with pytest.raises(ValueError, match="Invalid action_id"):
        r.step(np.array([0, -1, 1, 2]))
    after = r.sim.export_state()
    assert all(np.array_equal(before[f], after[f]) for f in before.dtype.names)  # nothing was stepped
    s = BatchedInversus(64, "dummy", "hard", 500, seed=0)
    s.reset()
    bad = torch.zeros(64, dtype=torch.int8, device="cuda")
    bad[5] = 13
    s.step(bad)
    assert s.poll_status() & STATUS_INVALID_ACTION
    assert s.poll_status() == 0  # sticky bit is cleared by the poll
    with pytest.raises(ValueError):
        BatchedInversus(4, "nonsense")  # env_wrappers.py:316
    sp = BatchedInversus(4, "selfplay", seed=0)
    sp.reset()
    with pytest.raises(ValueError, match="opponent_policy required"):  # env_wrappers.py:309
        sp.step(torch.zeros(4, dtype=torch.int8, device="cuda"))


def test_step_before_reset_fails_loudly():
    import torch
    from inversus_b200 import BatchedInversus, InversusError
    s = BatchedInversus(8, seed=0)
    with pytest.raises(InversusError):
        s.step(torch.zeros(8, dtype=torch.int8, device="cuda"))


@pytest.mark.parametrize("mode", ["dummy", "selfplay"])
def test_host_buffer_paths_deliver_identical_observations(mode):
    """inv_step_host: plain PCIe copy vs packed-rows + host expansion (any DMA share) must hand
    the caller bit-identical float32 observations and outputs; checked against the device views."""
    import torch
    from inversus_b200 import BatchedInversus
    n, T = 6000, 12
    rs = np.random.RandomState(21)
    sims = {}
    for name, (nt, frac) in {"plain": (0, 0.0), "expand_all": (4, 0.0), "hybrid": (3, 0.5), "auto": (None, -1.0)}.items():
        s = BatchedInversus(n, mode, "hard", 30, seed=17, auto_reset=True)
        s.set_host_path(nt, frac)
        s.reset()
        sims[name] = (s, s.host_buffers(pinned=(name != "expand_all")))
    for _ in range(T):
        a1 = rs.randint(0, 13, n).astype(np.int8)
        a2 = rs.randint(0, 13, n).astype(np.int8) if mode == "selfplay" else None
        for name, (s, out) in sims.items():
            s.step_host(a1, a2, out)
        ref_s, ref = sims["plain"]
        assert np.array_equal(ref["obs"], ref_s.obs.cpu().numpy())
        for name, (s, out) in sims.items():
            for k in ("obs", "extra", "reward", "done", "info", "episode_steps", "episode_return") + (
                    ("obs_p2", "extra_p2") if mode == "selfplay" else ()):
                assert np.array_equal(out[k], ref[k]), (name, k)
    assert sims["hybrid"][0].host_path()["dma_fraction"] == 0.5
    assert 0.0 <= sims["auto"][0].host_path()["dma_fraction"] <= 0.9


@pytest.mark.parametrize("n,chunks", [(37, 1), (4096 * 3 + 5, 1), (70001, 4), (70001, 3)])
def test_host_step_with_episode_events_matches_the_dense_outputs(n, chunks, monkeypatch):
    """inv_step_host_events (the trainer's view, training.py:140-151): reward / done / info dense and
    the finished episodes as a compact list. The list must be exactly the dense episode_steps /
    episode_return / info of the envs whose done flag is set, in env order; the device state and the
    observations left on the device must equal the dense call's. Short episodes (max 12 steps) make
    the list outgrow the prefix that travels with the count (second-copy path) from step 12 on."""
    import torch
    from inversus_b200 import BatchedInversus, _capi
    monkeypatch.setenv("INV_HOST_STAGED_MAX", "0")
    rs = np.random.RandomState(11)
    for mode in ("dummy", "selfplay"):
        monkeypatch.delenv("INV_HOST_CHUNKS", raising=False)
        ref = BatchedInversus(n, mode, "hard", 12, seed=9, auto_reset=True)
        got = BatchedInversus(n, mode, "hard", 12, seed=9, auto_reset=True)
        ref.reset()
        got.reset()
        ro = ref.host_buffers(pinned=False)
        eo = got.host_event_buffers(pinned=(mode == "dummy"))
        seen = 0
        for t in range(30):
            a1 = rs.randint(0, 13, n).astype(np.int8)
            a2 = rs.randint(0, 13, n).astype(np.int8) if mode == "selfplay" else None
            monkeypatch.delenv("INV_HOST_CHUNKS", raising=False)
            ref.step_host(a1, a2, ro)
            if chunks > 1:
                monkeypatch.setenv("INV_HOST_CHUNKS", str(chunks))
            eo["events"][:] = np.zeros(1, _capi.EVENT_DTYPE)[0]
            if t % 2:       # ids in page-locked memory go to the device from where they are
                pa = torch.empty(n, dtype=torch.int8, pin_memory=True)
                pa.numpy()[:] = a1
                ev = got.step_host_events(pa.numpy(), a2, eo)
            else:
                ev = got.step_host_events(a1, a2, eo)
            for k in ("reward", "done", "info"):
                assert np.array_equal(eo[k], ro[k]), (mode, t, k)
            idx = np.flatnonzero(ro["done"])
            assert ev.shape[0] == idx.size, (mode, t)
            assert np.array_equal(ev["env"], idx)
            assert np.array_equal(ev["episode_steps"], ro["episode_steps"][idx])
            assert np.array_equal(ev["episode_return"], ro["episode_return"][idx])   # binary64, bit for bit
            assert np.array_equal(ev["info"], ro["info"][idx].astype(np.uint32))
            seen += idx.size
            assert torch.equal(got.packed_state, ref.packed_state)
            assert torch.equal(got.obs, ref.obs) and torch.equal(got.extra, ref.extra)
        assert seen > n                     # every env finished at least twice on average
        assert got.poll_status() == 0
        # a list that does not fit: the true count comes back with the error
        small = dict(eo)
        small["events"] = np.zeros(1, _capi.EVENT_DTYPE)
        for _ in range(12):
            a1 = np.zeros(n, np.int8)
            try:
                got.step_host_events(a1, a1 if mode == "selfplay" else None, small)
            except ValueError as e:
                assert "events buffer" in str(e)
                break
        else:
            raise AssertionError("no overflow reported within one episode length")
        before = got.packed_state.clone()
        for pos, val in ((n - 1, 13), (5, -1), (n // 2, 127)):   # vector body and scalar tail of the id check
            with pytest.raises(ValueError):
                keep = torch.zeros(n, dtype=torch.int8, pin_memory=(pos == 5))  # both the staged and the direct path
                bad = keep.numpy()
                bad[pos] = val
                got.step_host_events(np.zeros(n, np.int8) if mode == "selfplay" else bad,
                                     bad if mode == "selfplay" else None, eo)
        assert torch.equal(got.packed_state, before)             # nothing was stepped
        ref.close()
        got.close()


@pytest.mark.parametrize("chunks", [2, 3, 4, 8])
def test_chunked_host_pipeline_delivers_the_same_bytes(chunks, monkeypatch):
    """inv_step_host cuts large batches into env chunks (kernel c+1 overlaps the copies of chunk c,
    direct copies into the caller's arrays, tapered chunks when no observation is requested). Forced
    here at a small batch: every output must equal the single-chunk call and the device views."""
    import torch
    from inversus_b200 import BatchedInversus
    n, T = 7000, 10
    monkeypatch.setenv("INV_HOST_STAGED_MAX", "0")        # small outputs go straight to the caller's arrays
    rs = np.random.RandomState(5)
    for mode in ("dummy", "selfplay"):
        monkeypatch.delenv("INV_HOST_CHUNKS", raising=False)
        ref = BatchedInversus(n, mode, "hard", 25, seed=3, auto_reset=True)
        got = BatchedInversus(n, mode, "hard", 25, seed=3, auto_reset=True)
        ref.reset()
        got.reset()
        ro, go = ref.host_buffers(pinned=True), got.host_buffers(pinned=False)
        small = {k: v for k, v in go.items() if not k.startswith("obs")}
        for t in range(T):
            a1 = rs.randint(0, 13, n).astype(np.int8)
            a2 = rs.randint(0, 13, n).astype(np.int8) if mode == "selfplay" else None
            monkeypatch.delenv("INV_HOST_CHUNKS", raising=False)
            ref.set_host_path(0, 0.0)
            ref.step_host(a1, a2, ro)
            monkeypatch.setenv("INV_HOST_CHUNKS", str(chunks))
            got.set_host_path(3 if t % 2 else 0, 0.4)      # plain copies and packed rows + host expansion
            if t % 3 == 2:
                for v in small.values():
                    if isinstance(v, np.ndarray):
                        v[...] = 0
                got.step_host(a1, a2, small)                # no observation requested: tapered chunks
                keys = [k for k in small if k != "_pins"]
            else:
                got.step_host(a1, a2, go)
                keys = [k for k in go if k != "_pins"]
            for k in keys:
                assert np.array_equal(go[k], ro[k]), (mode, chunks, t, k)
            assert torch.equal(got.packed_state, ref.packed_state)
        assert got.poll_status() == 0
        with pytest.raises(ValueError):
            bad = np.zeros(n, np.int8)
            bad[n - 1] = 13
            got.step_host(bad, bad if mode == "selfplay" else None, go)
        ref.close()
        got.close()


@pytest.mark.parametrize("dtype", ["f32", "bf16", "u8"])
def test_indexed_reset_for_every_observation_dtype(dtype):
    """MultiEnvRunner.envs[i].reset() path (inv_reset_envs) for all obs dtypes and both views:
    only the listed envs change, and what they become equals a handle that reset them all."""
    import torch
    from inversus_b200 import BatchedInversus
    n = 500
    a = BatchedInversus(n, "selfplay", "hard", 50, seed=12, obs_dtype=dtype, auto_reset=False)
    a.reset()
    rs = np.random.RandomState(0)
    for _ in range(10):
        a.step(torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda(),
               torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda())
    before = a.export_state()
    obs_before, obs2_before = a.obs.clone(), a.obs_p2.clone()
    idx = np.array(sorted(rs.choice(n, 77, replace=False)))
    a.reset_envs(idx)
    after = a.export_state()
    keep = np.setdiff1d(np.arange(n), idx)
    for f in before.dtype.names:
        assert np.array_equal(before[f][keep], after[f][keep]), f
    assert torch.equal(a.obs[keep], obs_before[keep]) and torch.equal(a.obs_p2[keep], obs2_before[keep])
    assert (after["episode"][idx] == 1).all() and (after["step_count"][idx] == 0).all()
    assert (after["n_bullets"][idx] == 0).all() and (after["episode_return"][idx] == 0).all()
    # the reset envs' observations equal a rebuild from their new state, in this dtype, for both views
    snap = a.snapshot()
    for view, got in ((0, a.obs), (1, a.obs_p2)):
        want, _ = a.obs_from_packed(snap, view=view, obs_dtype=dtype)
        assert torch.equal(got[idx].float(), want[idx].float())


def test_state_import_export_roundtrip_and_validation():
    from backends import check_state_import_export
    from inversus_b200 import BatchedInversus
    s = BatchedInversus(64, "dummy", "hard", 500, seed=1)
    s.reset()
    check_state_import_export(s.export_state, s.import_state)


def test_two_devices_in_one_process():
    """Handles on different GPUs of one process (function attributes and SM counts are per device)."""
    import torch
    from inversus_b200 import BatchedInversus
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sims = [BatchedInversus(5000, "selfplay", "hard", 50, seed=1, device=d, obs_dtype="u8") for d in (0, 1)]
    rs = np.random.RandomState(0)
    for s in sims:
        s.reset()
    for _ in range(5):
        a1, a2 = rs.randint(0, 13, 5000).astype(np.int8), rs.randint(0, 13, 5000).astype(np.int8)
        for d, s in enumerate(sims):
            s.step(torch.from_numpy(a1).cuda(d), torch.from_numpy(a2).cuda(d))
    assert torch.equal(sims[0].obs.cpu(), sims[1].obs.cpu()) and torch.equal(sims[0].reward.cpu(), sims[1].reward.cpu())


@pytest.mark.parametrize("mode", ["dummy", "selfplay"])
def test_snapshot_restore_resumes_bit_identically(mode):
    """Checkpoint/resume of the simulation: a snapshot of the packed state restored into a fresh
    handle (same seed) continues exactly like the original, observations included."""
    import torch
    from inversus_b200 import BatchedInversus
    n = 3000
    rs = np.random.RandomState(4)
    acts = [torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda() for _ in range(40)]
    a = BatchedInversus(n, mode, "hard", 25, seed=77, env_id_base=123)
    a.reset()
    for t in range(20):
        a.step(acts[t], acts[39 - t] if mode == "selfplay" else None)
    snap = a.snapshot()
    obs0 = a.obs.clone()
    b = BatchedInversus(n, mode, "hard", 25, seed=77, env_id_base=123)
    obs, extra = b.restore(snap)
    assert torch.equal(obs, obs0) and torch.equal(extra, a.extra)
    if mode == "selfplay":
        assert torch.equal(b.obs_p2, a.obs_p2)
    for t in range(20, 40):
        a.step(acts[t], acts[39 - t] if mode == "selfplay" else None)
        b.step(acts[t], acts[39 - t] if mode == "selfplay" else None)
        assert torch.equal(a.obs, b.obs) and torch.equal(a.reward, b.reward) and torch.equal(a.done, b.done)
    assert torch.equal(a.packed_state, b.packed_state)
    c = BatchedInversus(n, mode, "hard", 25, seed=78, env_id_base=123)  # a different seed diverges
    c.restore(snap)
    c.step(acts[20], acts[19] if mode == "selfplay" else None)
    if mode == "dummy":
        a2 = BatchedInversus(n, mode, "hard", 25, seed=77, env_id_base=123)
        a2.restore(snap)
        a2.step(acts[20])
        assert not torch.equal(c.packed_state, a2.packed_state)


def test_out_of_range_reset_indices_are_rejected_not_written():
    import torch
    from inversus_b200 import BatchedInversus
    from inversus_b200.constants import STATUS_BAD_INDEX
    s = BatchedInversus(100, "dummy", "hard", 50, seed=1, auto_reset=False)
    s.reset()
    before, obs_before = s.packed_state.clone(), s.obs.clone()
    s.reset_envs(torch.tensor([3, 100, -1, 10 ** 12, 7], dtype=torch.int64))
    assert s.poll_status() & STATUS_BAD_INDEX
    changed = (s.packed_state != before).any(dim=(0, 2)).nonzero().flatten().tolist()
    assert changed == [3, 7]
    keep = [i for i in range(100) if i not in (3, 7)]
    assert torch.equal(s.obs[keep], obs_before[keep])
