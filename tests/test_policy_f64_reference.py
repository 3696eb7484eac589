"""The float64 references and error bounds of tests/policy_f64.py checked on the CPU: the references
against float64 autograd and F.conv2d at small shapes, and the bounds against fp32 emulations of
what the kernels compute (same operations and roundings, summed in torch's own order -- hence the
depth of the whole sum), so a bound that is too tight for a correct kernel fails here first."""
import pytest
import torch
import torch.nn.functional as F

import policy_f64 as P


def _ln_case(B=7, D=96, C=8, res=True, cb=True, seed=0):
    gen = torch.Generator().manual_seed(seed)
    x, r, c, g, b = P.ln_inputs(B, D, C, res, cb, gen, "cpu")
    dy = P.integer_dy((B, D), gen, "cpu")
    return x, r, c, g, b, dy


@pytest.mark.parametrize("res,cb", [(False, False), (True, True), (False, True)])
def test_layernorm_reference_matches_autograd(res, cb):
    D, C = 96, 8
    x, r, c, g, b, dy = _ln_case(res=res, cb=cb)
    z, ez = P.ln_input(x, r, c, C)
    f = P.ln_forward(z, ez, g, b, 1e-5, depth=D)
    eps = float(torch.tensor(1e-5, dtype=torch.float32))
    zz = z.clone().requires_grad_()
    gg, bb = g.double().requires_grad_(), b.double().requires_grad_()
    o = F.layer_norm(zz, (D,), gg, bb, eps)
    assert torch.allclose(f["o"], o, rtol=1e-12, atol=1e-12)
    torch.relu(o).backward(dy.double())
    t = P.ln_backward(z, ez, dy, g, b, f["mean"], f["rstd"], D)  # at the exact statistics, like autograd
    assert torch.allclose(t["dx"], zz.grad, rtol=1e-9, atol=1e-9)
    cols = P.ColumnSums(D, "cpu")
    cols.add(t)
    assert torch.allclose(cols.dg, gg.grad, rtol=1e-9, atol=1e-9)
    assert torch.equal(cols.db, bb.grad)  # integer dy: exact on both sides
    if cb:  # d(channel bias) = sum over positions and samples of dz
        assert torch.allclose(t["dx"].view(x.shape[0], -1, C).sum((0, 1)), zz.grad.view(x.shape[0], -1, C).sum((0, 1)),
                              rtol=1e-9, atol=1e-9)


def _bf(t):
    return t.to(torch.bfloat16).float()


def _kernel_like_ln(x, r, c, g, b, C, pack):
    """fp32 restatement of ln_relu_fwd / the clustered backward (one-pass variance, rsqrt, folded
    affine, bf16 h / w between the passes with pack)."""
    D = x.shape[1]
    z = x.float() + (c.float().repeat(D // C) if c is not None else 0.0)
    if r is not None:
        z = z + r.float()
    inv_d = torch.tensor(1.0 / D, dtype=torch.float32)
    mean = z.sum(1, keepdim=True) * inv_d
    var = ((z * z).sum(1, keepdim=True) * inv_d - mean * mean).clamp_min(0)
    rstd = torch.rsqrt(var + torch.tensor(1e-5, dtype=torch.float32))
    sg = g.float() * rstd
    y = _bf(torch.relu(z * sg + (b.float() - mean * sg)))
    return z, mean.squeeze(1), rstd.squeeze(1), y


@pytest.mark.parametrize("pack", [False, True])
@pytest.mark.parametrize("res,cb", [(False, False), (True, True), (False, True)])
def test_layernorm_bounds_hold_for_an_fp32_restatement(res, cb, pack):
    B, D, C = 60, 1200, 8
    x, r, c, g, b, dy = _ln_case(B, D, C, res, cb, seed=3)
    zf, mean, rstd, y = _kernel_like_ln(x, r, c, g, b, C, pack)
    z, ez = P.ln_input(x, r, c, C)
    f = P.ln_forward(z, ez, g, b, 1e-5, depth=D)
    chk = P.Checker()
    chk("mean", mean, f["mean"], f["e_mean"])
    chk("rstd", rstd, f["rstd"], f["e_rstd"])
    yr, ey = P.relu_bf16_bound(f["o"], f["e_o"])
    chk("y", y, yr, ey)
    # backward in fp32 from the restated statistics
    m, rs = mean.unsqueeze(1), rstd.unsqueeze(1)
    h = zf * rs - m * rs
    gy = torch.where(h * g.float() + b.float() > 0, dy.float(), torch.zeros(()))
    w = gy * g.float()
    t1, t2 = w.sum(1, keepdim=True), (w * h).sum(1, keepdim=True)
    hp, wp = (_bf(h), _bf(w)) if pack else (h, w)
    inv_d = torch.tensor(1.0 / D, dtype=torch.float32)
    dx32 = hp * (-(t2 * inv_d * rs)) + (wp * rs - t1 * inv_d * rs)
    t = P.ln_backward(z, ez, dy, g, b, mean, rstd, D, pack)
    assert int(t["amb"].sum()) <= P.AMBIGUOUS_MAX * B * D + 1
    chk("dx", _bf(dx32), t["dx"], t["e_dx"], mask=~t["amb"])
    cols = P.ColumnSums(D, "cpu")
    cols.add(t)
    bg, bb = cols.bounds(B)
    chk("dgamma", (gy * h).sum(0), cols.dg, bg)
    chk("dbeta", gy.sum(0), cols.db, bb)
    chk.exact("dbeta exact", gy.sum(0), cols.db, mask=cols.namb == 0)


def test_checker_rejects_nan_and_out_of_bound_elements_and_keeps_the_worst_ratio():
    chk = P.Checker()
    ref = torch.zeros(4, dtype=torch.float64)
    bound = torch.ones(4, dtype=torch.float64)
    assert chk("a", torch.tensor([0.5, 0.0, 0.0, -0.25]), ref, bound) == 0.5
    with pytest.raises(AssertionError, match="NaN"):
        chk("a", torch.tensor([0.0, float("nan"), 0.0, 0.0]), ref, bound)
    with pytest.raises(AssertionError, match="outside"):
        chk("a", torch.tensor([0.0, 1.5, 0.0, 0.0]), ref, bound)
    chk("a", torch.tensor([0.0, 9.0, 0.0, 0.0]), ref, bound, mask=torch.tensor([True, False, True, True]))
    assert chk.worst["a"] == 1.5
    with pytest.raises(AssertionError, match="differ"):
        chk.exact("b", torch.tensor([1.0]), torch.tensor([1.0 + 2 ** -30], dtype=torch.float64))


def _obs(n, gen, p=0.2):
    """0/1 observation planes: exactly one of the two tile planes set, sparse object planes."""
    white = (torch.rand(n, 1, 10, 15, generator=gen) < 0.5).float()
    sparse = (torch.rand(n, 10, 10, 15, generator=gen) < p * 0.1).float()
    return torch.cat([1 - white, white, sparse], 1)


def test_encoder_reference_matches_autograd_of_conv_layernorm_relu():
    gen = torch.Generator().manual_seed(1)
    n = 5
    obs = _obs(n, gen)
    w1 = 0.2 * torch.randn(32, 12, 3, 3, generator=gen)
    b1 = 0.1 * torch.randn(32, generator=gen)
    g = 1 + 0.3 * torch.randn(4800, generator=gen)
    b = 0.2 * torch.randn(4800, generator=gen)
    dy = P.integer_dy((n, 4800), gen, "cpu")
    z, ez = P.encoder_conv(obs, w1, b1)
    w, bias = w1.double().requires_grad_(), b1.double().requires_grad_()
    zz = F.conv2d(obs.double(), w, bias, padding=1)
    assert torch.allclose(z, zz.permute(0, 2, 3, 1).reshape(n, -1), rtol=0, atol=1e-12)
    gg = g.double().view(10, 15, 32).permute(2, 0, 1).requires_grad_()
    bb = b.double().view(10, 15, 32).permute(2, 0, 1).requires_grad_()
    f = P.ln_forward(z, ez, g, b, 1e-5, depth=4800)
    eps = float(torch.tensor(1e-5, dtype=torch.float32))
    o = F.layer_norm(zz, (32, 10, 15), gg, bb, eps)
    assert torch.allclose(f["o"], o.permute(0, 2, 3, 1).reshape(n, -1), atol=1e-12)
    torch.relu(o).backward(dy.double().view(n, 10, 15, 32).permute(0, 3, 1, 2))
    t = P.ln_backward(z, ez, dy, g, b, f["mean"], f["rstd"], 4800)
    wg = P.EncoderWeightGrad("cpu")
    wg.add(obs, t["dx"], t["e_dx32"])
    assert torch.allclose(wg.dw, w.grad, rtol=1e-9, atol=1e-9)
    assert torch.allclose(wg.db, bias.grad, rtol=1e-9, atol=1e-9)
    cols = P.ColumnSums(4800, "cpu")
    cols.add(t)
    assert torch.allclose(cols.dg, gg.grad.permute(1, 2, 0).reshape(-1), rtol=1e-9, atol=1e-9)
    assert torch.equal(cols.db, bb.grad.permute(1, 2, 0).reshape(-1))
    # the black-tap bound covers every in-board tap: at least the white-tap bound of the same entry
    bw, _ = wg.bounds(10)
    assert bool((bw[:, 0] >= bw[:, 1]).all())


def test_encoder_bound_holds_for_a_bf16_restatement_of_the_feature_map():
    """The kernel's map: fp32 dense part rounded to bf16, then one bf16 rounding per sparse object."""
    gen = torch.Generator().manual_seed(2)
    n = 6
    obs = _obs(n, gen, p=1.0)
    w1 = 0.2 * torch.randn(32, 12, 3, 3, generator=gen)
    b1 = 0.1 * torch.randn(32, generator=gen)
    zt = _bf(F.conv2d(obs[:, :2], w1[:, :2], b1, padding=1))
    for s in range(n):
        for c, y0, x0 in torch.nonzero(obs[s, 2:]).tolist():
            for ky in range(3):
                for kx in range(3):
                    py, px = y0 - (ky - 1), x0 - (kx - 1)
                    if 0 <= py < 10 and 0 <= px < 15:
                        zt[s, :, py, px] = _bf(zt[s, :, py, px] + w1[:, c + 2, ky, kx])
    z, ez = P.encoder_conv(obs, w1, b1)
    P.Checker()("z", zt.permute(0, 2, 3, 1).reshape(n, -1), z, ez)


def test_exact_encoder_weights_give_an_exact_bf16_map_and_mean():
    gen = torch.Generator().manual_seed(3)
    obs = _obs(16, gen, p=3.0)
    w1, b1 = P.exact_encoder_weights(gen, "cpu")
    z, ez = P.encoder_conv(obs, w1, b1)
    assert not bool(ez.any())  # no rounding anywhere: the bound is exactly 0
    assert torch.equal(z.to(torch.bfloat16).double(), z) and bool((z.abs() < 16).all())
    assert torch.equal((z * 16).round(), z * 16)
    zf = z.float()
    s = torch.zeros(16, dtype=torch.float32)
    for j in range(4800):  # any fp32 summation order of the row is exact
        s = s + zf[:, j]
    assert torch.equal(P.exact_mean(z), (s * torch.tensor(1 / 4800, dtype=torch.float32)).double())


@pytest.mark.parametrize("cin,cout", [(32, 64), (64, 128)])
def test_wgrad_reference_matches_autograd_and_integer_operands_are_exact(cin, cout):
    gen = torch.Generator().manual_seed(cin)
    B = 3
    x = torch.randint(-1, 2, (B, 10, 15, cin), generator=gen).to(torch.bfloat16)
    dy = torch.randint(-1, 2, (B, 10, 15, cout), generator=gen).to(torch.bfloat16)
    ref, absum = P.wgrad_ref(dy, x)
    w = torch.zeros(cout, cin, 3, 3, dtype=torch.float64, requires_grad=True)
    F.conv2d(x.double().permute(0, 3, 1, 2), w, padding=1).backward(dy.double().permute(0, 3, 1, 2))
    assert torch.equal(ref, w.grad.permute(0, 2, 3, 1))
    assert torch.equal(ref.float().double(), ref) and bool((ref.abs() <= absum).all())
    # tap (ky, kx) pairs dy at (y, x) with x at (y + ky - 1, x + kx - 1)
    assert float(ref[0, 0, 0, 0]) == float((dy[:, 1:, 1:, 0].double() * x[:, :-1, :-1, 0].double()).sum())
    n, parts = P.wgrad_depth(32771, 128, 148)
    assert parts == 49 and n == 10 * 669
    assert P.wgrad_depth(5, 64, 148) == (10, 5)
