"""GPU checks of the PPO rows: the GAE kernel against the reference's golden vectors and the numpy
restatement (bit-exact float32), the bf16 policy path within its stated tolerance, the packed
rollout store, and short end-to-end training runs on the device-resident loop."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_gae_kernel_matches_reference_golden_and_numpy():
    import torch
    from inversus_b200.ppo_agent import compute_gae, gae_numpy
    g = np.load(os.path.join(GOLD, "gae_reference.npz"))
    for case in "abc":  # the reference's flat-list GAE = N 1
        r, v, d = (torch.from_numpy(g[f"{case}_{k}"]).cuda().view(-1, 1) for k in ("reward", "value", "done"))
        adv, ret = compute_gae(r, v, d, None, 0.99, 0.95)
        assert np.array_equal(adv.view(-1).cpu().numpy(), g[f"{case}_adv"])
        assert np.array_equal(ret.view(-1).cpu().numpy(), g[f"{case}_ret"])
    rs = np.random.RandomState(0)
    for T, N in ((128, 1000), (1, 5), (37, 4097)):
        r, v = rs.randn(T, N).astype(np.float32), rs.randn(T, N).astype(np.float32)
        d = (rs.rand(T, N) < 0.07).astype(np.uint8)
        lv = rs.randn(N).astype(np.float32)
        want = gae_numpy(r, v, d, lv, 0.99, 0.95)
        got = compute_gae(torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(d).cuda(),
                          torch.from_numpy(lv).cuda(), 0.99, 0.95)
        assert np.array_equal(got[0].cpu().numpy(), want[0]) and np.array_equal(got[1].cpu().numpy(), want[1])


def test_bf16_policy_path_tracks_fp32():
    import torch
    from inversus_b200.policies import InversusCNNPolicy
    torch.manual_seed(0)
    m = InversusCNNPolicy().cuda()
    g = (torch.rand(512, 12, 10, 15, device="cuda") > 0.7)
    e = torch.rand(512, 4, device="cuda")
    with torch.no_grad():
        a = m(g.float(), e)
        for obs in (g.float(), g.to(torch.bfloat16), g.to(torch.uint8)):
            b = m.infer(obs, e)
            # tolerance: 3e-2 absolute on fp32 logits/value (bf16 has 8 mantissa bits; |logit| ~ 0.1-1)
            assert (a[0] - b[0]).abs().max() < 3e-2 and (a[1] - b[1]).abs().max() < 3e-2
            assert (a[0].argmax(-1) == b[0].argmax(-1)).float().mean() > 0.9


def test_packed_rollout_decodes_to_the_observations_the_policy_saw():
    import torch
    from inversus_b200 import BatchedInversus, DeviceRollout
    n, T = 300, 12
    sim = BatchedInversus(n, "dummy", "hard", 20, seed=1)
    packed = DeviceRollout(T, n, "cuda", store="packed")
    full = DeviceRollout(T, n, "cuda", store="obs")
    obs, extra = sim.reset()
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    for _ in range(T):
        a = torch.randint(0, 13, (n,), device="cuda", generator=g)
        z = torch.zeros(n, device="cuda")
        packed.store_pre(sim, a, z, z)
        full.store_pre((obs, extra), a, z, z)
        (obs, extra), r, d, _ = sim.step(a.to(torch.int8))
        packed.store_post(r, d)
        full.store_post(r, d)
    idx = torch.randperm(T * n, device="cuda", generator=g)[:1000]
    og, oe = packed.minibatch_obs(idx, sim)
    fg, fe = full.minibatch_obs(idx, sim)
    assert torch.equal(og, fg) and torch.equal(oe, fe)
    assert torch.equal(packed.rewards, full.rewards) and torch.equal(packed.dones, full.dones)


def test_vs_dummy_training_runs_on_the_device_resident_loop(tmp_path):
    """BASELINE.json configs[0] shape (vs_dummy PPO, num_envs=4) for a few updates + a wider run."""
    import torch
    from inversus_b200 import train_vs_dummy
    torch.manual_seed(0)
    out = train_vs_dummy(num_envs=4, total_steps=2048, log_dir=str(tmp_path / "a"), opponent_difficulty="hard",
                         precision="fp32", reference_gae=True, seed=1, quiet=True)
    assert out["steps"] == 2048 and out["steps_per_env"] == 512 and out["batch_size"] == 512
    assert out["episodes"] > 0 and np.isfinite(out["policy_loss"]) and np.isfinite(out["value_loss"])
    assert 0.0 < out["entropy"] <= np.log(13) + 1e-3
    rows = open(os.path.join(str(tmp_path / "a"), "training_log.csv")).read().splitlines()
    assert rows[0].startswith("step,episode,avg_reward,win_rate") and len(rows) >= 2
    sd = torch.load(os.path.join(str(tmp_path / "a"), "policy_final.pt"), map_location="cpu")
    from inversus_b200.policies import REFERENCE_STATE_DICT_SHAPES
    assert {k: tuple(v.shape) for k, v in sd.items()} == REFERENCE_STATE_DICT_SHAPES  # loads into the reference
    out = train_vs_dummy(num_envs=2048, total_steps=2048 * 16 * 2, log_dir=str(tmp_path / "b"),
                         opponent_difficulty="hard", precision="bf16", rollout_steps=16, batch_size=4096, seed=2,
                         quiet=True, save=False)
    assert out["steps"] == 2048 * 32 and out["episodes"] > 100 and np.isfinite(out["policy_loss"])


def test_selfplay_training_runs(tmp_path):
    import torch
    from inversus_b200 import train_selfplay
    torch.manual_seed(0)
    out = train_selfplay(num_envs=512, total_steps=512 * 16 * 3, log_dir=str(tmp_path), precision="bf16",
                         rollout_steps=16, batch_size=2048, seed=3, quiet=True, save=False)
    assert out["steps"] == 512 * 48 and np.isfinite(out["policy_loss"]) and np.isfinite(out["entropy"])


def test_ppo_learns_to_beat_the_easy_dummy(tmp_path):
    """Learning-quality smoke: against the easy (sitting-duck) dummy a short run must raise the
    kill frequency (wins per 1000 env-steps in the last logging window) clearly above what the
    same untrained policy achieves (lr = 0 control, same seed)."""
    import torch
    from inversus_b200 import train_vs_dummy
    kw = dict(num_envs=4096, log_dir=str(tmp_path), opponent_difficulty="easy", precision="bf16",
              rollout_steps=64, batch_size=8192, seed=5, quiet=True, save=False)
    torch.manual_seed(0)
    base = train_vs_dummy(total_steps=4096 * 64 * 2, lr=0.0, **kw)
    torch.manual_seed(0)
    out = train_vs_dummy(total_steps=4096 * 64 * 10, lr=3e-4, **kw)
    print("control:", base["wins_per_kstep"], base["last_window"], "trained:", out["wins_per_kstep"], out["last_window"],
          {k: out[k] for k in ("samples_per_s", "rollout_s", "update_s", "rollout_env_steps_per_s")})
    assert out["wins_per_kstep"] > 1.5 * base["wins_per_kstep"], (base, out)


def test_fused_layernorm_relu_kernels_match_torch():
    """csrc/policy_kernels.cu vs the plain PyTorch fp32 reference of the same op, for the three
    layer widths of the policy (D = 4800, 9600, 19200), with and without the residual input.
    Tolerances: forward 2e-2 relative to the output range (bf16 output, 8-bit mantissa); dx cosine
    > 0.999 and max error < 2 % of its max magnitude; dgamma/dbeta (fp32 accumulation, compared
    after their bf16 rounding) within 2 % of max."""
    import torch
    import torch.nn.functional as F
    from inversus_b200.fused_ops import layer_norm_relu
    torch.manual_seed(0)
    for D in (4800, 9600, 19200):
        for with_res in (False, True):
            for B in (3, 700):
                x = torch.randn(B, D, device="cuda").to(torch.bfloat16).requires_grad_()
                r = torch.randn(B, D, device="cuda").to(torch.bfloat16).requires_grad_() if with_res else None
                g = (torch.rand(D, device="cuda") + 0.5).to(torch.bfloat16).requires_grad_()
                b = (torch.rand(D, device="cuda") - 0.5).to(torch.bfloat16).requires_grad_()
                dy = torch.randn(B, D, device="cuda").to(torch.bfloat16)
                C_ = {4800: 32, 9600: 64, 19200: 128}[D]
                cb = torch.randn(C_, device="cuda").to(torch.bfloat16).requires_grad_()  # folded conv bias
                y = layer_norm_relu(x, g, b, 1e-5, residual=r, channel_bias=cb, channels=C_)
                y.backward(dy)
                xf = x.detach().float().requires_grad_()
                rf = r.detach().float().requires_grad_() if with_res else None
                gf, bf_ = g.detach().float().requires_grad_(), b.detach().float().requires_grad_()
                cbf = cb.detach().float().requires_grad_()
                z = xf + cbf.repeat(D // C_)  # HWC rows: channel = index % C
                z = z + rf if with_res else z
                yr = F.relu(F.layer_norm(z, (D,), gf, bf_, 1e-5))
                yr.backward(dy.float())
                assert (y.float() - yr).abs().max() < 2e-2 * max(1.0, yr.abs().max().item())
                pairs = [(x.grad, xf.grad), (g.grad, gf.grad), (b.grad, bf_.grad), (cb.grad, cbf.grad)]
                if with_res:
                    pairs.append((r.grad, rf.grad))
                for got, want in pairs:
                    got = got.float()
                    assert F.cosine_similarity(got.flatten(), want.flatten(), dim=0) > 0.999
                    assert (got - want).abs().max() <= 0.02 * want.abs().max() + 1e-3, (D, with_res, B)


def test_fused_policy_path_matches_unfused():
    import torch
    from inversus_b200.policies import InversusCNNPolicy
    torch.manual_seed(0)
    m = InversusCNNPolicy().cuda()
    for i in (1, 2, 3, 4):
        n = getattr(m, f"norm{i}")
        n.weight.data.uniform_(0.5, 1.5)
        n.bias.data.uniform_(-0.5, 0.5)
    g = (torch.rand(256, 12, 10, 15, device="cuda") > 0.7)
    e = torch.rand(256, 4, device="cuda")
    outs, grads = [], []
    for fused in (True, False):
        m.use_fused_kernels = fused
        m.zero_grad()
        lo, va = m.forward_bf16(g, e)
        (lo.sum() + va.sum()).backward()
        outs.append((lo.detach(), va.detach()))
        grads.append([p.grad.clone() for p in m.parameters()])
    assert (outs[0][0] - outs[1][0]).abs().max() < 3e-2 and (outs[0][1] - outs[1][1]).abs().max() < 3e-2
    for (name, _), a, b in zip(m.named_parameters(), *grads):
        cs = torch.nn.functional.cosine_similarity(a.flatten(), b.flatten(), dim=0)
        assert cs > 0.99, (name, cs.item())


def test_cuda_graph_rollout_fills_the_same_rollout_as_the_eager_loop(tmp_path):
    """The graph-captured step (policy inference + sampling + fused env step + rollout stores, time
    index on the device) must leave a complete, self-consistent rollout: with lr = 0 and fp32 the
    stored values/log-probs must equal a fresh forward of the stored observations."""
    import torch
    from inversus_b200 import BatchedInversus, DeviceRollout, InversusCNNPolicy, PPOAgent
    torch.manual_seed(0)
    torch.backends.cudnn.allow_tf32 = False  # true fp32 convolutions, so batch size does not change results
    n, T = 64, 24
    sim = BatchedInversus(n, "dummy", "hard", 30, seed=3, auto_reset=True)
    agent = PPOAgent(InversusCNNPolicy(), device="cuda", precision="fp32")
    ro = DeviceRollout(T, n, "cuda", store="packed")
    obs, extra = sim.reset()
    t_dev = torch.zeros(1, dtype=torch.int64, device="cuda")

    def step():
        a, lp, v = agent.act(obs, extra)
        ro.store_pre_at(t_dev, sim, a, lp, v)
        sim.step(a.to(torch.int8))
        ro.store_post_at(t_dev, sim.reward, sim.done)
        t_dev.add_(1)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            t_dev.zero_()
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    t_dev.zero_()
    with torch.cuda.graph(graph):
        step()
    sim.reset()
    t_dev.zero_()
    for _ in range(T):
        graph.replay()
    torch.cuda.synchronize()
    assert int(t_dev.item()) == T
    ro.t = T
    idx = torch.arange(T * n, device="cuda")
    g, e = ro.minibatch_obs(idx, sim)
    with torch.no_grad():
        logits, values = agent.policy(g, e)
    lp = torch.log_softmax(logits, -1).gather(1, ro.actions.reshape(-1, 1)).squeeze(1)
    assert torch.allclose(values.squeeze(-1), ro.values.reshape(-1), atol=1e-4)
    assert torch.allclose(lp, ro.log_probs.reshape(-1), atol=1e-4)
    assert int(ro.dones.sum()) > 0 and bool(torch.isfinite(ro.rewards).all())
    assert sim.poll_status() == 0


def test_head_weight_transpose_cast_kernel():
    import torch
    from inversus_b200.fused_ops import head_weight_to_hwc
    torch.manual_seed(0)
    for R, C_, P_, extra in ((512, 128, 150, 4), (3, 5, 7, 0), (40, 33, 65, 9)):
        w = torch.randn(R, C_ * P_ + extra, device="cuda", requires_grad=True)
        out = head_weight_to_hwc(w, C_, P_)
        want = w[:, : C_ * P_].detach().to(torch.bfloat16).reshape(R, C_, P_).permute(0, 2, 1).reshape(R, -1)
        assert torch.equal(out, want)
        g = torch.randn_like(out)
        out.backward(g)
        gw = torch.zeros_like(w)
        gw[:, : C_ * P_] = g.float().reshape(R, P_, C_).permute(0, 2, 1).reshape(R, -1)
        assert torch.equal(w.grad, gw)
