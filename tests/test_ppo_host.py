"""CPU checks of the PPO rows (SURVEY.md section 8f): checkpoint compatibility of the policy, GAE
against the reference's golden vectors, and -- when the live reference is present -- bit-exact
agreement of a whole PPO update with inversus_rl.ppo_agent.PPOAgent."""
import os

import numpy as np
import pytest
import torch

from ref_harness import SKIP_REASON, reference_available

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_policy_has_the_reference_checkpoint_layout():
    from inversus_b200.policies import REFERENCE_STATE_DICT_SHAPES, InversusCNNPolicy
    m = InversusCNNPolicy()
    sd = m.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == REFERENCE_STATE_DICT_SHAPES
    assert sum(p.numel() for p in m.parameters()) == 10_249_582  # SURVEY.md section 2 #7
    logits, value = m(torch.zeros(1, 12, 10, 15), torch.zeros(1, 4))  # tests/test_rl_env_wrapper.py:132
    assert logits.shape == (1, 13) and value.shape == (1, 1)


def test_gae_matches_reference_golden_vectors():
    from inversus_b200.ppo_agent import gae_numpy
    g = np.load(os.path.join(GOLD, "gae_reference.npz"))
    for case in "abc":
        r, v, d = g[f"{case}_reward"], g[f"{case}_value"], g[f"{case}_done"]
        adv, ret = gae_numpy(r[:, None], v[:, None], d[:, None], None, 0.99, 0.95)  # flat list = N 1
        assert np.array_equal(adv[:, 0], g[f"{case}_adv"]) and np.array_equal(ret[:, 0], g[f"{case}_ret"])


def test_per_env_gae_is_the_flat_gae_of_each_column():
    from inversus_b200.ppo_agent import gae_numpy
    rs = np.random.RandomState(0)
    T, N = 50, 7
    r, v = rs.randn(T, N).astype(np.float32), rs.randn(T, N).astype(np.float32)
    d = (rs.rand(T, N) < 0.1)
    lv = rs.randn(N).astype(np.float32)
    adv, ret = gae_numpy(r, v, d, lv, 0.99, 0.95)
    for n in range(N):
        a1, r1 = gae_numpy(r[:, n:n + 1], v[:, n:n + 1], d[:, n:n + 1], lv[n:n + 1], 0.99, 0.95)
        assert np.array_equal(adv[:, n], a1[:, 0]) and np.array_equal(ret[:, n], r1[:, 0])


@pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
def test_policy_forward_is_bit_identical_to_the_live_reference():
    from ref_harness import import_reference
    import_reference()
    from inversus_rl.policies import InversusCNNPolicy as Ref
    from inversus_b200.policies import InversusCNNPolicy
    torch.manual_seed(0)
    ref, mine = Ref(12, 10, 15, 4), InversusCNNPolicy()
    mine.load_state_dict(ref.state_dict())
    g = (torch.rand(6, 12, 10, 15) > 0.7).float()
    e = torch.rand(6, 4)
    with torch.no_grad():
        a, b, c = ref(g, e), mine(g, e), mine.infer(g, e)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # bf16 autocast path: tolerance 2e-2 absolute on logits/value of a random-init net (|logit| ~ 0.1)
    assert (a[0] - c[0]).abs().max() < 2e-2 and (a[1] - c[1]).abs().max() < 2e-2


@pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
def test_ppo_update_is_bit_identical_to_the_live_reference():
    """Same buffers, same numpy shuffle seed -> identical GAE, losses (1e-6) and parameters (exact)."""
    from ref_harness import import_reference
    import_reference()
    from inversus_rl.policies import InversusCNNPolicy as RefPol
    from inversus_rl.ppo_agent import PPOAgent as RefAgent
    from inversus_b200.policies import InversusCNNPolicy
    from inversus_b200.ppo_agent import PPOAgent
    torch.manual_seed(0)
    rp, mp = RefPol(12, 10, 15, 4), InversusCNNPolicy()
    mp.load_state_dict(rp.state_dict())
    ra = RefAgent(rp, batch_size=48, epochs=2)
    ma = PPOAgent(mp, batch_size=48, epochs=2, gae_mode="reference", shuffle="numpy")
    rs = np.random.RandomState(1)
    for _ in range(150):
        g = (rs.rand(12, 10, 15) > 0.8).astype(np.float32)
        e = rs.rand(4).astype(np.float32)
        args = (g, e, int(rs.randint(13)), float(-rs.rand() * 3), float(rs.randn()), float(rs.randn() * 0.1),
                bool(rs.rand() < 0.05))
        ra.store_step(*args)
        ma.store_step(*args)
    a1, r1 = ra.compute_advantages()
    a2, r2 = ma.compute_advantages()
    assert np.array_equal(a1, a2) and np.array_equal(r1, r2)
    np.random.seed(5)
    s1 = ra.update()
    np.random.seed(5)
    s2 = ma.update()
    for k in s1:
        assert abs(s1[k] - s2[k]) <= 1e-6 * max(1.0, abs(s1[k])), k
    for p, q in zip(rp.parameters(), mp.parameters()):
        assert torch.equal(p, q)
    # act(): numpy in -> numpy out with the reference's shapes and dtypes (ppo_agent.py:68-106)
    torch.manual_seed(3)
    x = ra.act(np.zeros((4, 12, 10, 15), np.float32), np.zeros((4, 4), np.float32))
    torch.manual_seed(3)
    y = ma.act(np.zeros((4, 12, 10, 15), np.float32), np.zeros((4, 4), np.float32))
    for u, w in zip(x, y):
        assert isinstance(w, np.ndarray) and u.shape == w.shape and np.array_equal(u, w)


def test_training_logger_writes_the_reference_columns(tmp_path):
    from inversus_b200.training import TrainingLogger
    lg = TrainingLogger(str(tmp_path))
    lg.log(2048, 3, 1.5, 0.33, 20.0, 0.1, 0.2, 2.5)
    rows = open(os.path.join(str(tmp_path), "training_log.csv")).read().splitlines()
    assert rows[0] == "step,episode,avg_reward,win_rate,avg_ep_len,policy_loss,value_loss,entropy"  # training.py:28-31
    assert rows[1].startswith("2048,3,1.5,0.33,20.0,")


def test_bf16_path_matches_fp32_forward_and_gradients():
    """forward_bf16 restructures the network (channels-last, HWC-permuted LayerNorm parameters and
    head-weight columns, fused + K-split head GEMM). Against the plain fp32 forward with
    randomised LayerNorm affines: outputs within 2e-2 absolute, every parameter gradient with
    cosine similarity > 0.99 (bf16 has an 8-bit mantissa)."""
    import torch.nn.functional as F
    from inversus_b200.policies import InversusCNNPolicy
    torch.manual_seed(0)
    m = InversusCNNPolicy()
    for i in (1, 2, 3, 4):
        n = getattr(m, f"norm{i}")
        n.weight.data.uniform_(0.5, 1.5)
        n.bias.data.uniform_(-0.5, 0.5)
    g = (torch.rand(5, 12, 10, 15) > 0.7).float()
    e = torch.rand(5, 4)
    a, b = m(g, e), m.forward_bf16(g, e)
    assert (a[0] - b[0]).abs().max() < 2e-2 and (a[1] - b[1]).abs().max() < 2e-2
    ga = torch.autograd.grad(a[0].sum() + a[1].sum(), list(m.parameters()))
    gb = torch.autograd.grad(b[0].sum() + b[1].sum(), list(m.parameters()))
    for (name, _), x, y in zip(m.named_parameters(), ga, gb):
        assert F.cosine_similarity(x.flatten(), y.flatten(), dim=0) > 0.99, name
    for obs in (g.to(torch.uint8), g.to(torch.bfloat16)):
        c = m.infer(obs, e)
        assert torch.equal(c[0], b[0].detach()) and torch.equal(c[1], b[1].detach())


def test_inference_cache_follows_optimizer_steps():
    from inversus_b200.policies import InversusCNNPolicy
    torch.manual_seed(1)
    m = InversusCNNPolicy()
    g, e = (torch.rand(3, 12, 10, 15) > 0.6).float(), torch.rand(3, 4)
    a = m.infer(g, e)
    assert torch.equal(m.infer(g, e)[0], a[0])          # served from the cache
    opt = torch.optim.SGD(m.parameters(), lr=0.5)
    loss = m(g, e)[0].sum()
    loss.backward()
    opt.step()                                            # in-place update bumps tensor versions
    b = m.infer(g, e)
    assert not torch.equal(a[0], b[0])
    assert torch.equal(b[0], m.forward_bf16(g, e)[0].detach())
    # fused optimizers do not bump tensor versions: the agent marks the policy updated itself, and the
    # cached tensors are refreshed IN PLACE (a captured CUDA graph keeps reading the same addresses)
    from inversus_b200.ppo_agent import PPOAgent
    agent = PPOAgent(m, lr=0.05, epochs=1, batch_size=3)
    agent.optimizer = torch.optim.Adam(m.parameters(), lr=0.05, fused=True)
    cached = m.inference_weights()
    ptrs = {k: v.data_ptr() for k, v in cached.items()}
    for i in range(3):
        agent.store_step(g[i].numpy(), e[i].numpy(), 1, -2.0, 0.0, 1.0, False)
    agent.update()
    c = m.infer(g, e)
    assert not torch.equal(b[0], c[0])
    assert torch.equal(c[0], m.forward_bf16(g, e)[0].detach())
    assert {k: v.data_ptr() for k, v in m.inference_weights().items()} == ptrs
