"""The policy kernels on the PPO update path -- inv_ln_relu_fwd / _bwd, inv_encode_fwd / _bwd and
inv_conv3x3_wgrad -- against float64 references, element by element, at the trainer's batch sizes.
Every element has its own bound from a rounding model of the kernel (tests/policy_f64.py); the
bounds are checked to be able to fail. The C entry points are called directly on NaN-filled output
and scratch buffers, so the fp32 outputs are seen before any bf16 rounding and an element a kernel
does not write (or a stale partial it reads) shows up. Exact checks need no tolerance at all:
integer operands make the weight gradient and dbeta exact, and exact encoder weights make the
encoder's pre-LayerNorm map, and so its row mean, exact."""
import os
import subprocess
import sys

import pytest

import policy_f64 as P

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 1 << 22  # elements per float64 reference chunk (tens of temporaries: well under 2 GB)
EPS = 1e-5
CHECK = P.Checker()


def _variant():
    """Which LayerNorm backward the library runs in this process (it reads the variables once)."""
    if os.environ.get("INV_LN_BWD", "").startswith("pe"):
        return "percta"
    return "S2" if os.environ.get("INV_LN_BWD_S", "").startswith("2") else "cluster"


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    peak = _torch().cuda.max_memory_reserved() / 2 ** 30
    print(f"\nlargest error / bound per check ({_variant()} LayerNorm backward; peak device memory {peak:.2f} GiB):")
    for k, v in sorted(CHECK.worst.items()):
        print(f"  {k:28s} {v:.3g}")


def _torch():
    import torch
    return torch


def _lib():
    from inversus_b200 import _capi
    return _capi.load(), _capi.check


def _stream():
    return _torch().cuda.current_stream().cuda_stream


def _nan(*shape, dtype=None):
    torch = _torch()
    return torch.full(shape, float("nan"), dtype=dtype or torch.float32, device="cuda")


def _ptr(t):
    return None if t is None else t.data_ptr()


def _sms():
    return _torch().cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------
# LayerNorm + ReLU
def _ln_run(B, D, with_res, with_cb, dy_kind, beta_neg=False):
    torch = _torch()
    C = D // 150
    gen = torch.Generator(device="cuda")
    gen.manual_seed(B * 7919 + D + 2 * with_res + with_cb + 5 * beta_neg + (dy_kind == "int"))
    x, res, cb, g, b = P.ln_inputs(B, D, C, with_res, with_cb, gen, "cuda", beta_neg)
    if dy_kind == "int":
        dy = P.integer_dy((B, D), gen, "cuda")
    else:
        dy = torch.randn(B, D, generator=gen, device="cuda").to(torch.bfloat16)
    lib, chk = _lib()
    bf = torch.bfloat16
    o = dict(y=_nan(B, D, dtype=bf), mean=_nan(B), rstd=_nan(B), dx=_nan(B, D, dtype=bf), dgamma=_nan(D),
             dbeta=_nan(D), dcbias=_nan(C), partials=_nan(lib.inv_ln_relu_partials(D), 2 * D + C))
    chk(lib.inv_ln_relu_fwd(x.data_ptr(), _ptr(res), _ptr(cb), g.data_ptr(), b.data_ptr(), B, D, C, EPS,
                            o["y"].data_ptr(), o["mean"].data_ptr(), o["rstd"].data_ptr(), _stream()))
    chk(lib.inv_ln_relu_bwd(dy.data_ptr(), x.data_ptr(), _ptr(res), _ptr(cb), g.data_ptr(), b.data_ptr(),
                            o["mean"].data_ptr(), o["rstd"].data_ptr(), B, D, C, o["dx"].data_ptr(),
                            o["dgamma"].data_ptr(), o["dbeta"].data_ptr(), o["dcbias"].data_ptr(),
                            o["partials"].data_ptr(), _stream()))
    torch.cuda.synchronize()
    inp = dict(B=B, D=D, C=C, x=x, res=res, cb=cb, g=g, b=b, dy=dy, int_dy=dy_kind == "int")
    return inp, o


def _ln_geometry(inp, partials):
    """Chain lengths of the backward's column sums, from the parts it wrote into the NaN-filled
    partials: percta, one row of 2D + C per CTA; clustered, 2D per cluster plus C per CTA."""
    B, D, C = inp["B"], inp["D"], inp["C"]
    written = int(_torch().isfinite(partials).sum())
    v = _variant()
    if v == "percta":
        parts = written // (2 * D + C)
        assert parts * (2 * D + C) == written and 1 <= parts <= B
        chain, nctas, fold, pack = -(-B // parts), parts, 512 // (C // 8), False
    else:
        cs = -(-(D // 8) // 320)
        S = 2 if (inp["res"] is not None or v == "S2") else 4
        groups = -(-B // S)
        parts = written // (2 * D + cs * C)
        assert parts * (2 * D + cs * C) == written and 1 <= parts <= groups
        chain, nctas, fold, pack = S * -(-groups // parts), parts * cs, 320 // (C // 8), S == 4
    # dgamma / dbeta: one accumulator per column over `chain` samples, then the parts
    # d conv bias: the same chain, a fold over the threads of a channel group, then the CTAs
    return dict(d_col=chain + parts + 2, d_cb=chain + fold + nctas + 2, pack=pack)


def _ln_check(inp, o, chk):
    torch = _torch()
    B, D, C = inp["B"], inp["D"], inp["C"]
    geo = _ln_geometry(inp, o["partials"])
    v = _variant()
    cols = P.ColumnSums(D, "cuda")
    dcb = torch.zeros(3, C, dtype=torch.float64, device="cuda")  # reference, sum(|dx| + e), sum(e)
    namb = nrest = 0
    rows = max(1, CHUNK // D)
    for a in range(0, B, rows):
        sl = slice(a, min(B, a + rows))
        n = sl.stop - a
        z, ez = P.ln_input(inp["x"][sl], None if inp["res"] is None else inp["res"][sl], inp["cb"], C)
        # forward: per thread <= 5 vectors x 4 pairs in a chain, + pair, 5 warp, 4 block levels <= 32
        f = P.ln_forward(z, ez, inp["g"], inp["b"], EPS, depth=32)
        chk("ln_fwd.mean", o["mean"][sl], f["mean"], f["e_mean"])
        chk("ln_fwd.rstd", o["rstd"][sl], f["rstd"], f["e_rstd"])
        yr, ey = P.relu_bf16_bound(f["o"], f["e_o"])
        chk("ln_fwd.y", o["y"][sl], yr, ey)
        # row sums: clustered 4 + 1 + 5 + 10 warps + 8 ranks; percta 40 + 5 + 4: both <= 64
        t = P.ln_backward(z, ez, inp["dy"][sl], inp["g"], inp["b"], o["mean"][sl], o["rstd"][sl], 64, geo["pack"])
        # In a (nearly) constant row, h is rstd (up to eps^-1/2 = 316) times the rounding noise of
        # the mean, so every column whose |beta| lies inside that noise is ambiguous by construction.
        # The rarity check covers the other rows (var >= 1e-2, i.e. rstd < 10; the typical and
        # offset rows have var >= 1, the nearly constant ones var <~ 1e-4).
        live = (f["rstd"] < 10).unsqueeze(1)
        namb += int((t["amb"] & live).sum())
        nrest += int(live.sum()) * D
        chk(f"ln_bwd[{v}].dx", o["dx"][sl], t["dx"], t["e_dx"], mask=~t["amb"])
        cols.add(t)
        dcb[0] += t["dx"].view(n, -1, C).sum((0, 1))
        dcb[1] += (t["dx"].abs() + t["e_dx32"]).view(n, -1, C).sum((0, 1))
        dcb[2] += t["e_dx32"].view(n, -1, C).sum((0, 1))
    assert namb <= P.AMBIGUOUS_MAX * nrest, (namb, nrest)
    bg, bb = cols.bounds(geo["d_col"])
    chk(f"ln_bwd[{v}].dgamma", o["dgamma"], cols.dg, bg)
    chk(f"ln_bwd[{v}].dbeta", o["dbeta"], cols.db, bb)
    if inp["int_dy"]:
        chk.exact(f"ln_bwd[{v}].dbeta(int dy)", o["dbeta"], cols.db, mask=cols.namb == 0)
    chk(f"ln_bwd[{v}].dcbias", o["dcbias"], dcb[0], dcb[2] + P.gam(geo["d_cb"]) * dcb[1])
    return cols


LN_B = (1, 2, 3, 5, 37, 149, 4097, 16384, 32771)
LN_CASES = [(D, res, cb, B, "int") for D in (4800, 9600, 19200) for res in (False, True) for cb in (False, True)
            for B in LN_B]
LN_CASES += [(D, res, True, B, "real") for D in (4800, 9600, 19200) for res in (False, True) for B in (37, 4097, 32771)]


def _ln_id(c):
    D, res, cb, B, dy = c
    return f"D{D}-{'res' if res else 'nores'}-{'cb' if cb else 'nocb'}-B{B}-{dy}"


@pytest.mark.parametrize("case", LN_CASES, ids=_ln_id)
def test_ln_relu_matches_float64(case):
    D, res, cb, B, dy = case
    inp, o = _ln_run(B, D, res, cb, dy)
    _ln_check(inp, o, CHECK)


@pytest.mark.parametrize("D", [4800, 9600, 19200])
@pytest.mark.parametrize("res", [False, True], ids=["nores", "res"])
def test_ln_relu_matches_float64_with_most_units_off(D, res):
    inp, o = _ln_run(4097, D, res, True, "int", beta_neg=True)
    _ln_check(inp, o, CHECK)


@pytest.mark.parametrize("env", [{"INV_LN_BWD": "percta"}, {"INV_LN_BWD_S": "2"}], ids=["percta", "S2"])
def test_ln_relu_alternative_backward_kernels(env):
    """INV_LN_BWD=percta and INV_LN_BWD_S=2 select two more backward kernels; the library reads each
    variable once per process, so the same cases run in a child interpreter (S = 2 only differs
    from the default without the residual input)."""
    if os.environ.get("POLICY_F64_CHILD"):
        pytest.skip("runs in the parent interpreter only")
    sel = "test_ln_relu_matches" + (" and nores" if "INV_LN_BWD_S" in env else "")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", os.path.abspath(__file__), "-q", "-s", "-m", "gpu", "-k", sel, "-p", "no:cacheprovider"]
    r = subprocess.run(cmd, env=dict(os.environ, POLICY_F64_CHILD="1", **env), cwd=ROOT, capture_output=True,
                       text=True)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-3000:]


def test_ln_relu_checks_reject_small_defects():
    """Each injected defect in real kernel outputs must be rejected by the same checks."""
    torch = _torch()
    inp, o = _ln_run(4097, 19200, False, True, "int")
    _ln_check(inp, o, P.Checker())
    bad = dict(o, dx=o["dx"].clone())
    bad["dx"][[0, 1]] = o["dx"][[1, 0]]  # two samples of one group swapped
    with pytest.raises(AssertionError, match="dx"):
        _ln_check(inp, bad, P.Checker())
    k = 2049  # one sample's contribution to dgamma and dbeta dropped
    z, ez = P.ln_input(inp["x"][k:k + 1], None, inp["cb"], inp["C"])
    t = P.ln_backward(z, ez, inp["dy"][k:k + 1], inp["g"], inp["b"], o["mean"][k:k + 1], o["rstd"][k:k + 1], 64)
    for name, drop in (("dgamma", (t["gy"] * t["h"])[0]), ("dbeta", t["gy"][0])):
        bad = dict(o, **{name: (o[name].double() - drop).float()})
        assert not torch.equal(bad[name], o[name])
        with pytest.raises(AssertionError, match=name):
            _ln_check(inp, bad, P.Checker())


# ------------------------------------------------------------------------------------------------
# conv3x3 weight gradient
def _wgrad_run(dy, x):
    torch = _torch()
    lib, chk = _lib()
    B, cout, cin = dy.shape[0], dy.shape[3], x.shape[3]
    dw = _nan(cout, 3, 3, cin)
    scratch = _nan(lib.inv_conv3x3_wgrad_scratch_floats(cin, cout))
    chk(lib.inv_conv3x3_wgrad(dy.data_ptr(), x.data_ptr(), B, cin, cout, dw.data_ptr(), scratch.data_ptr(), _stream()))
    torch.cuda.synchronize()
    return dw


def _wgrad_ref(dy, x):
    torch = _torch()
    ref = absum = 0
    rows = max(1, CHUNK // (150 * max(dy.shape[3], x.shape[3])))
    for a in range(0, dy.shape[0], rows):
        r, s = P.wgrad_ref(dy[a:a + rows], x[a:a + rows])
        ref, absum = ref + r, absum + s
    return ref, absum


def _wgrad_operands(B, cin, cout, integer, seed):
    torch = _torch()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    if integer:  # {-1, 0, 1}: every partial sum is an integer below B * 150 <= 4.9 M < 2^24
        mk = lambda c: torch.randint(-1, 2, (B, 10, 15, c), generator=gen, device="cuda").to(torch.bfloat16)  # noqa: E731
    else:
        mk = lambda c: torch.randn(B, 10, 15, c, generator=gen, device="cuda").to(torch.bfloat16)  # noqa: E731
    return mk(cout), mk(cin)


@pytest.mark.parametrize("cin,cout", [(128, 128), (64, 128), (32, 64)])
@pytest.mark.parametrize("B", [1, 2, 48, 49, 50, 147, 148, 149, 16384, 32771])
def test_conv3x3_wgrad_matches_float64(cin, cout, B):
    dy, x = _wgrad_operands(B, cin, cout, True, B * 131 + cin)
    ref, _ = _wgrad_ref(dy, x)
    CHECK.exact("wgrad.int (bit-exact)", _wgrad_run(dy, x), ref)
    dy, x = _wgrad_operands(B, cin, cout, False, B * 137 + cin)
    ref, absum = _wgrad_ref(dy, x)
    CHECK(f"wgrad.real {cout}x{cin}", _wgrad_run(dy, x), ref, P.wgrad_bound(absum, B, cin, _sms()))


@pytest.mark.parametrize("cin,cout", [(128, 128), (64, 128), (32, 64)])
def test_conv3x3_wgrad_checks_reject_small_defects(cin, cout):
    torch = _torch()
    B = 149
    dy, x = _wgrad_operands(B, cin, cout, True, 11)
    dw = _wgrad_run(dy, x)
    ref, _ = _wgrad_ref(dy, x)
    P.Checker().exact("wgrad", dw, ref)
    one, _ = P.wgrad_ref(dy[77:78], x[77:78])  # one sample's contribution dropped
    with pytest.raises(AssertionError):
        P.Checker().exact("wgrad", (dw.double() - one).float(), ref)
    # tap (1, 1) reading its operand one position further along the row-major board
    xs = torch.zeros_like(x).view(B, 150, cin)
    xs[:, :-1] = x.view(B, 150, cin)[:, 1:]
    shifted, _ = _wgrad_ref(dy, xs.view_as(x))
    bad = dw.clone()
    bad[:, 1, 1] = shifted[:, 1, 1].float()
    with pytest.raises(AssertionError):
        P.Checker().exact("wgrad", bad, ref)


# ------------------------------------------------------------------------------------------------
# encoder
_POOL = {}


def _crafted_states(n=64):
    """States no rollout reaches on purpose: 16 bullets, coinciding bullets, dead players, players and
    bullets on all four edges and corners; env 0 is an all-white board with one black tile."""
    import numpy as np
    from inversus_b200 import BatchedInversus
    sim = BatchedInversus(n, "selfplay", "hard", 30, seed=4, obs_dtype="f32", auto_reset=False, p2_view=True)
    sim.reset()
    st = sim.export_state()
    rs = np.random.RandomState(8)
    edge = [(0, 0), (14, 0), (0, 9), (14, 9), (7, 0), (0, 5), (14, 4), (6, 9)]
    for i in range(n):
        st["tiles"][i] = rs.randint(0, 2 ** 32, 5, dtype=np.uint64).astype(np.uint32)
        st["tiles"][i, 4] &= (1 << 22) - 1  # 150 tile bits
        for p, k in (("p1", i), ("p2", i + 3)):
            st[p][i, :2] = edge[k % 8]
            st[p][i, 2] = rs.randint(0, 7)
            st[p][i, 4] = int(rs.rand() > 0.25)
        nb = 16 if i % 2 == 0 else rs.randint(0, 16)
        st["n_bullets"][i] = nb
        for j in range(nb):
            ex, ey = edge[rs.randint(0, 8)] if rs.rand() < 0.5 else (rs.randint(0, 15), rs.randint(0, 10))
            st["bullets"][i, j] = [ex, ey, rs.randint(0, 4), rs.randint(0, 2)]
        if nb >= 4:
            st["bullets"][i, 1] = st["bullets"][i, 0]  # same tile, direction and owner
            st["bullets"][i, 3] = st["bullets"][i, 2]
            st["bullets"][i, 3, 3] ^= 1  # same tile and direction, other owner
    st["tiles"][0] = [0xFFFFFFFF] * 4 + [(1 << 22) - 1]
    st["tiles"][0, 2] &= ~np.uint32(1 << 9)  # one black tile at bit 73: (x, y) = (13, 4)
    sim.import_state(st)
    return sim


def _pool():
    """[crafted 64 | dummy rollout | selfplay rollout] packed states, and a sim to decode them."""
    if not _POOL:
        torch = _torch()
        from inversus_b200 import BatchedInversus
        parts = [_crafted_states().snapshot()]
        for mode, seed in (("dummy", 5), ("selfplay", 6)):
            n = 33000
            sim = BatchedInversus(n, mode, "hard", 30, seed=seed, obs_dtype="none", auto_reset=True, p2_view=True)
            sim.reset()
            g = torch.Generator(device="cuda")
            g.manual_seed(seed)
            for _ in range(41):
                a = torch.randint(0, 13, (n,), device="cuda", generator=g).to(torch.int8)
                sim.step(a, torch.randint(0, 13, (n,), device="cuda", generator=g).to(torch.int8) if mode == "selfplay" else None)
            parts.append(sim.snapshot())
            del sim
        _POOL["planes"] = torch.cat(parts, 1).contiguous()
        _POOL["sim"] = BatchedInversus(4, "selfplay", "hard", 30, seed=1, obs_dtype="f32", auto_reset=False, p2_view=True)
    return _POOL["planes"], _POOL["sim"]


def _enc_params(exact, seed):
    torch = _torch()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    if exact:
        w1, b1 = P.exact_encoder_weights(gen, "cuda")
    else:
        w1 = 0.2 * torch.randn(32, 12, 3, 3, generator=gen, device="cuda")
        b1 = 0.1 * torch.randn(32, generator=gen, device="cuda")
    g = 1.0 + 0.3 * torch.randn(4800, generator=gen, device="cuda")
    b = 0.2 * torch.randn(4800, generator=gen, device="cuda")
    return w1, b1, g, b, gen


def _enc_run(lo, count, view, exact, seed=0):
    """Both encoder kernels on entries [lo, lo + count) of the pool, a view with stride > count at
    a non-zero offset, exactly as PackedStates.chunk passes it."""
    torch = _torch()
    planes, sim = _pool()
    w1, b1, g, b, gen = _enc_params(exact, seed + count + 17 * view)
    dy = P.integer_dy((count, 4800), gen, "cuda")
    lib, chk = _lib()
    ptr, stride = planes.data_ptr() + lo * 16, planes.shape[1]
    o = dict(y=_nan(count, 4800, dtype=torch.bfloat16), extra=_nan(count, 4), mean=_nan(count), rstd=_nan(count),
             dw1=_nan(32, 12, 3, 3), db1=_nan(32), dgamma=_nan(4800), dbeta=_nan(4800),
             partials=_nan(lib.inv_encode_partials_floats()))
    chk(lib.inv_encode_fwd(ptr, stride, count, view, w1.data_ptr(), b1.data_ptr(), g.data_ptr(), b.data_ptr(), EPS,
                           o["y"].data_ptr(), o["extra"].data_ptr(), o["mean"].data_ptr(), o["rstd"].data_ptr(),
                           _stream()))
    chk(lib.inv_encode_bwd(ptr, stride, count, view, w1.data_ptr(), b1.data_ptr(), g.data_ptr(), b.data_ptr(),
                           o["mean"].data_ptr(), o["rstd"].data_ptr(), dy.data_ptr(), o["dw1"].data_ptr(),
                           o["db1"].data_ptr(), o["dgamma"].data_ptr(), o["dbeta"].data_ptr(), o["partials"].data_ptr(),
                           _stream()))
    torch.cuda.synchronize()
    window = planes[:, lo:lo + count].contiguous()
    obs, extra = sim.obs_from_packed(window, view=view, obs_dtype="f32")
    inp = dict(count=count, view=view, exact=exact, w1=w1, b1=b1, g=g, b=b, dy=dy, obs=obs, extra=extra, window=window)
    return inp, o


def _enc_check(inp, o, chk, fwd_only=False):
    torch = _torch()
    count = inp["count"]
    chk.exact("enc_fwd.extra", o["extra"], inp["extra"].double())
    cols = P.ColumnSums(4800, "cuda")
    wg = P.EncoderWeightGrad("cuda")
    namb = 0
    rows = max(1, CHUNK // 4800 // 4)
    for a in range(0, count, rows):
        sl = slice(a, min(count, a + rows))
        z, ez = P.encoder_conv(inp["obs"][sl], inp["w1"], inp["b1"])
        if inp["exact"]:
            chk.exact("enc_fwd.mean (exact weights)", o["mean"][sl], P.exact_mean(z))
        # per lane 75 steps of two terms + 5 shuffle levels: chains <= 155 for both sums
        f = P.ln_forward(z, ez, inp["g"], inp["b"], EPS, depth=160)
        chk("enc_fwd.mean", o["mean"][sl], f["mean"], f["e_mean"])
        chk("enc_fwd.rstd", o["rstd"][sl], f["rstd"], f["e_rstd"])
        yr, ey = P.relu_bf16_bound(f["o"], f["e_o"])
        chk("enc_fwd.y", o["y"][sl], yr, ey)
        if fwd_only:
            continue
        t = P.ln_backward(z, ez, inp["dy"][sl], inp["g"], inp["b"], o["mean"][sl], o["rstd"][sl], 160)
        namb += int(t["amb"].sum())
        cols.add(t)
        e_dz = t["e_dx32"] + P.UB * (t["dx"].abs() + t["e_dx32"])  # dz is stored as bf16 before the tap sums
        wg.add(inp["obs"][sl], t["dx"], e_dz)
    if fwd_only:
        return None
    # With real weights the bf16 feature map moves a pre-activation by up to 2^-8 Zabs (1 + k) rstd |g|,
    # which leaves about 1 % of the ReLU decisions undetermined by the kernel's own arithmetic. No
    # element check excludes them here (y needs no exclusion, dz is not an output); they only widen
    # the column-sum bounds below by their largest contribution. With exact weights the map is
    # exact, and there they must be rare.
    if inp["exact"]:
        assert namb <= P.AMBIGUOUS_MAX * count * 4800, namb
    # partial sums: `rounds` samples per warp, 8 warps per CTA, CTAs summed in 8 strided chains + 8
    grid = min(-(-count // 8), _sms())
    rounds = -(-count // (8 * grid))
    tail = -(-grid // 8) + 8 + 2
    bg, bb = cols.bounds(8 * rounds + tail)
    chk("enc_bwd.dgamma", o["dgamma"], cols.dg, bg)
    chk("enc_bwd.dbeta", o["dbeta"], cols.db, bb)
    chk.exact("enc_bwd.dbeta (int dy)", o["dbeta"], cols.db, mask=cols.namb == 0)
    # dw1: 150 positions per sample into one lane's accumulator, 8 warps, the CTAs, 9 border corrections
    bw, bb1 = wg.bounds(150 * rounds + 8 + tail + 9)
    chk("enc_bwd.dw1 (white, sparse)", o["dw1"][:, 1:], wg.dw[:, 1:], bw[:, 1:])
    chk("enc_bwd.dw1 (black)", o["dw1"][:, :1], wg.dw[:, :1], bw[:, :1])
    chk("enc_bwd.db1", o["db1"], wg.db, bb1)
    return wg


NPOOL = 64 + 2 * 33000
ENC_CASES = [(5, 1), (3, 7), (64 + 33000 - 600, 8 * 148 + 1), (64 + 33000 + 7, 16384), (11, 32771)]


@pytest.mark.parametrize("lo,count", ENC_CASES, ids=[f"count{c}" for _, c in ENC_CASES])
@pytest.mark.parametrize("view", [0, 1])
@pytest.mark.parametrize("exact", [True, False], ids=["exact_w", "real_w"])
def test_encoder_matches_float64(lo, count, view, exact):
    inp, o = _enc_run(lo, count, view, exact)
    _enc_check(inp, o, CHECK)


def test_encoder_checks_reject_small_defects():
    torch = _torch()
    # a tile bit flipped in the reference state: the forward check must see it
    inp, o = _enc_run(3, 7, 0, False)
    _enc_check(inp, o, P.Checker())
    planes, sim = _pool()
    flipped = inp["window"].clone()
    flipped[0, 0, 0] ^= 1  # tile (0, 0) of entry 0
    obs, _ = sim.obs_from_packed(flipped, view=0, obs_dtype="f32")
    with pytest.raises(AssertionError, match="enc_fwd.y"):
        _enc_check(dict(inp, obs=obs), o, P.Checker(), fwd_only=True)
    # one black tap's dw1 changed by its smallest term: entry 0 of the pool has a single black tile,
    # so each black tap has at most one term. Exact weights: with real ones ~1 % of the ReLU decisions
    # are ambiguous, and their largest contributions over all in-board taps exceed one term.
    inp, o = _enc_run(0, 1, 0, True)
    wg = _enc_check(inp, o, P.Checker())
    z, ez = P.encoder_conv(inp["obs"], inp["w1"], inp["b1"])
    t = P.ln_backward(z, ez, inp["dy"], inp["g"], inp["b"], o["mean"], o["rstd"], 160)
    dz = P.from_hwc(t["dx"])
    term = torch.nn.grad.conv2d_weight(inp["obs"].double()[:, :1], (32, 1, 3, 3), dz, padding=1)[:, 0]
    bound = wg.bounds(150 + 8 + 1 + 8 + 2 + 9)[0][:, 0]
    co, tap = divmod(int((term.abs() / bound).flatten().argmax()), 9)
    bad = o["dw1"].clone()
    bad[co, 0, tap // 3, tap % 3] -= float(term[co, tap // 3, tap % 3])
    with pytest.raises(AssertionError, match="black"):
        _enc_check(inp, dict(o, dw1=bad), P.Checker())
