"""float64 references of the policy kernels (csrc/policy_kernels.cu, encoder_kernels.cu,
wgrad_kernels.cu) with an error bound for every element, derived from a rounding model of what
each kernel does. No GPU needed: every function takes torch tensors on any device.

Notation: U = 2^-24 is the unit roundoff of fp32 (24 significant bits, round to nearest) and
UB = 2^-8 that of bf16: it keeps 8 significant bits, so a rounded value is within half a step of
2^-7 relative, i.e. 2^-8 |value| (2^-9 would be the bound for 9 bits).
A sum of n terms evaluated in fp32 in any order whose longest chain of additions has `depth`
additions is off by at most gam(depth) * sum|terms| (Higham, Accuracy and Stability, eq. 4.4);
every "depth" below is counted from the kernel's loop structure where it is used.

An element whose float64 pre-activation |h*gamma + beta| lies inside its own rounding bound may take
either ReLU branch in the kernel ("ambiguous"): it is left out of the element checks of y and dx, and
its largest possible contribution is added to the bounds of every sum it enters.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

U = 2.0 ** -24
UB = 2.0 ** -8
AMBIGUOUS_MAX = 1e-4  # at most this fraction of the elements may be ambiguous
BOARD_H, BOARD_W = 10, 15


def gam(n):
    """gamma_n = n U / (1 - n U): bound of n successive fp32 roundings."""
    return n * U / (1.0 - n * U)


class Checker:
    """Element checks |got - ref| <= bound; keeps the largest error/bound ratio of every named check."""

    def __init__(self):
        self.worst = {}

    def __call__(self, name, got, ref, bound, mask=None):
        got = got.double()
        if mask is not None:
            got, ref, bound = got[mask], ref[mask], bound[mask]
        assert not torch.isnan(got).any(), f"{name}: NaN (an element the kernel did not write)"
        err = (got - ref).abs()
        bad = err > bound
        ratio = float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0
        self.worst[name] = max(self.worst.get(name, 0.0), ratio)
        if bool(bad.any()):
            i = int(torch.nonzero(bad.flatten())[0])
            raise AssertionError(f"{name}: {int(bad.sum())} of {err.numel()} elements outside their bound; first at "
                                 f"flat index {i}: got {float(got.flatten()[i])!r}, ref {float(ref.flatten()[i])!r}, "
                                 f"bound {float(bound.flatten()[i])!r}")
        return ratio

    def exact(self, name, got, ref, mask=None):
        """Bit-exact: the reference is an fp32-representable value and the kernel must return it."""
        if mask is not None:
            got, ref = got[mask], ref[mask]
        assert torch.equal(got.double(), ref), f"{name}: {int((got.double() != ref).sum())} elements differ"
        self.worst.setdefault(name, 0.0)


# ------------------------------------------------------------------------------------------------
# LayerNorm + ReLU
def ln_input(x, res, cb, C):
    """z = x + channel bias (+ residual) in float64, and ez, the bound of the kernel's fp32 z: at most
    two fp32 additions, each rounded, so |z' - z| <= 2 U (|x| + |cb| + |res|)."""
    D = x.shape[1]
    z = x.double()
    Z = z.abs()
    if cb is not None:
        c = cb.double().repeat(D // C)
        z = z + c
        Z = Z + c.abs()
    if res is not None:
        r = res.double()
        z = z + r
        Z = Z + r.abs()
    return z, 2 * U * Z


def ln_forward(z, ez, g, b, eps, depth, ops=3):
    """Row statistics and pre-ReLU output o = (z - mean) rstd g + b, with bounds, for rows of z.

    The kernel forms mean = fl(sum z' * fl(1/D)) and var = fl(sum z'^2 * fl(1/D)) - mean^2 (one pass),
    each sum a chain of `depth` fp32 additions, then rstd = rsqrtf(var + eps):
      e_mean = mean(ez) + gam(depth + 4) mean(|z| + ez)                      (terms, chain, 1/D, product)
      e_E    = mean(ez (2|z| + ez)) + gam(depth + 4) mean((|z| + ez)^2)
      e_var  = e_E + (2|mean| + e_mean) e_mean + 2 U (E + mean^2)            (mean^2, subtraction)
    The last term is where the condition factor (mean^2 + var) / var enters: the one-pass variance is
    only as good as e_var / var. rstd is bounded without linearising, which covers var ~ 0:
      rstd in [ (var + e_var + eps)^-1/2 (1 - 5U), (max(var - e_var, 0) + eps)^-1/2 (1 + 5U) ]
    (rsqrtf is within 2 ulp = 4 U; the + eps rounds once more, half of it after the square root).
    The output takes `ops` more roundings (fp32 multiplies / fmas), each at most U times the
    magnitude it rounds. The LayerNorm kernel evaluates z (rstd g) + (b - mean (rstd g)), so that
    magnitude is up to |g| rstd (|z| + |mean|) + |b| + |o|, not |g| rstd |z - mean|:
      e_o = |g| r_hi (ez + e_mean) + |g| |z - mean| e_rstd + ops U (|g| r_hi (|z| + |mean| + ez + e_mean) + |b| + |o|)
    """
    eps = float(torch.tensor(eps, dtype=torch.float32))
    D = z.shape[1]
    mean = z.mean(1, keepdim=True)
    zc = z - mean
    var = (zc * zc).mean(1, keepdim=True)
    Zm = z.abs() + ez
    e_mean = ez.mean(1, keepdim=True) + gam(depth + 4) * Zm.mean(1, keepdim=True)
    E = (z * z).mean(1, keepdim=True)
    e_E = (ez * (2 * z.abs() + ez)).mean(1, keepdim=True) + gam(depth + 4) * (Zm * Zm).mean(1, keepdim=True)
    e_var = e_E + (2 * mean.abs() + e_mean) * e_mean + 2 * U * (E + mean * mean)
    rstd = (var + eps).rsqrt()
    r_hi = ((var - e_var).clamp_min(0) + eps).rsqrt() * (1 + 5 * U)
    r_lo = (var + e_var + eps).rsqrt() * (1 - 5 * U)
    e_rstd = torch.maximum(r_hi - rstd, rstd - r_lo)
    g, b = g.double(), b.double()
    o = zc * rstd * g + b
    ag = g.abs()
    e_o = (ag * r_hi * (ez + e_mean) + ag * zc.abs() * e_rstd
           + ops * U * (ag * r_hi * (z.abs() + mean.abs() + ez + e_mean) + b.abs() + o.abs()))
    assert D == g.numel()
    return dict(mean=mean.squeeze(1), e_mean=e_mean.squeeze(1), rstd=rstd.squeeze(1), e_rstd=e_rstd.squeeze(1),
                o=o, e_o=e_o)


def relu_bf16_bound(o, e_o):
    """y = bf16(relu(o')) with |o' - o| <= e_o: relu is 1-Lipschitz, the bf16 rounding adds UB |y|."""
    y = o.clamp_min(0)
    return y, e_o + UB * (y + e_o)


def ln_backward(z, ez, dy, g, b, mean, rstd, depth_row, pack=False):
    """LayerNorm+ReLU backward of rows of z given the kernel's fp32 mean / rstd inputs (taken as exact):
        h = (z - mean) rstd,  gy = dy [h g + b > 0],  w = gy g,  m1 = mean(w),  m2 = mean(w h),
        dx = rstd (w - m1 - h m2),  dgamma = sum_rows gy h,  dbeta = sum_rows gy.
    Bounds (the kernel's fp32 values are primed):
      e_h   = rstd (ez + U (|z| + |mean|)) + 2 U |h|     fma(z', rstd, -mean rstd) or (z' - mean) rstd
      e_pre = 2 |g| e_h + 2 U |pre|                       the ReLU test; inside it the branch is ambiguous
      e_t1  = (gam(depth_row) + U) sum|w| + sum_amb |dy g|
      e_t2  = gam(depth_row) sum|w h| + sum |w| (e_h + 2 U |h|) + sum_amb |dy g| (|h| + e_h)
    With pack (the S = 4 clustered kernel parks h and w as bf16 between its passes) w and h each take
    one more bf16 rounding before pass 2. dx' = rstd w' - rstd m1' - h' rstd m2' in at most 6 roundings:
      e_dx32 = rstd (e_w + e_t1 / D + |h| e_t2 / D + (|m2| + e_t2 / D) e_hp) + 6 U rstd (|w| + |m1| + |h m2|)
    and the bf16 output adds UB |dx|. An ambiguous element's own dx may differ by rstd |dy g| more."""
    D = z.shape[1]
    dy, g, b = dy.double(), g.double(), b.double()
    mean, rstd = mean.double().unsqueeze(1), rstd.double().unsqueeze(1)
    h = (z - mean) * rstd
    pre = h * g + b
    e_h = rstd * (ez + U * (z.abs() + mean.abs())) + 2 * U * h.abs()
    ag = g.abs()
    e_pre = 2 * ag * e_h + 2 * U * pre.abs()
    amb = (pre.abs() <= e_pre) & (dy != 0)
    gy = torch.where(pre > 0, dy, torch.zeros_like(dy))
    w = gy * g
    m1 = w.mean(1, keepdim=True)
    m2 = (w * h).mean(1, keepdim=True)
    dx = rstd * (w - m1 - h * m2)
    aw, ah = w.abs(), h.abs()
    adg = torch.where(amb, dy.abs() * ag, torch.zeros_like(dy))
    e_t1 = (gam(depth_row) + U) * aw.sum(1, keepdim=True) + adg.sum(1, keepdim=True)
    e_t2 = (gam(depth_row) * (aw * ah).sum(1, keepdim=True) + (aw * (e_h + 2 * U * ah)).sum(1, keepdim=True)
            + (adg * (ah + e_h)).sum(1, keepdim=True))
    e_w = U * aw + (UB * (1 + U) * aw if pack else 0.0)
    e_hp = e_h + (UB * (ah + e_h) if pack else 0.0)
    e_dx32 = (rstd * (e_w + e_t1 / D + ah * e_t2 / D + (m2.abs() + e_t2 / D) * e_hp)
              + 6 * U * rstd * (aw + m1.abs() + ah * m2.abs()))
    e_dx = e_dx32 + UB * (dx.abs() + e_dx32)
    return dict(h=h, e_h=e_h, gy=gy, amb=amb, dx=dx, e_dx32=e_dx32 + rstd * adg, e_dx=e_dx,
                ady=torch.where(amb, dy.abs(), torch.zeros_like(dy)))


class ColumnSums:
    """dgamma / dbeta references and bounds, accumulated in float64 over row chunks.
    Per column: the kernel sums fp32 products gy h' (error |gy| (e_h + U |h|) each) in a chain of at most
    `depth` additions, then ambiguous elements may add or drop |dy| (|h| + e_h) and |dy|:
      bound(dgamma) = (1 + gam(depth)) sum|gy| (e_h + U|h|) + gam(depth) sum|gy h| + sum_amb |dy| (|h| + e_h)
      bound(dbeta)  = gam(depth) sum|gy| + sum_amb |dy|."""

    def __init__(self, D, device):
        z = lambda: torch.zeros(D, dtype=torch.float64, device=device)  # noqa: E731
        self.dg, self.db, self.ag, self.eg, self.mg, self.ab, self.mb = z(), z(), z(), z(), z(), z(), z()
        self.namb = torch.zeros(D, dtype=torch.int64, device=device)

    def add(self, t):
        gy, h, e_h, ady = t["gy"], t["h"], t["e_h"], t["ady"]
        self.dg += (gy * h).sum(0)
        self.db += gy.sum(0)
        self.ag += (gy * h).abs().sum(0)
        self.eg += (gy.abs() * (e_h + U * h.abs())).sum(0)
        self.mg += (ady * (h.abs() + e_h)).sum(0)
        self.ab += gy.abs().sum(0)
        self.mb += ady.sum(0)
        self.namb += t["amb"].sum(0)

    def bounds(self, depth):
        return ((1 + gam(depth)) * self.eg + gam(depth) * self.ag + self.mg, gam(depth) * self.ab + self.mb)


def integer_dy(shape, gen, device, lo=-3, hi=3):
    """dy with small integer values: every partial sum of gy is then an integer below 2^24, so the
    kernel's dbeta is exact in every column without an ambiguous element."""
    return torch.randint(lo, hi + 1, shape, generator=gen, device=device).to(torch.bfloat16)


def ln_inputs(B, D, C, with_res, with_cb, gen, device, beta_neg=False):
    """bf16 inputs of one LayerNorm case. Rows cycle through three families:
    0 typical (x ~ N(0, 1)); 1 a large common offset, |mean| ~ 8 std; 2 constant (no channel bias) or
    nearly constant rows, var <~ eps: x = bf16(c - cbias), residual 0, every other row with a little
    noise. gamma in [0.5, 1.5]; beta in [-0.5, 0.5], or in [-3, -2] with beta_neg (most units off)."""
    bf = torch.bfloat16
    rnd = lambda *s: torch.randn(*s, generator=gen, device=device)  # noqa: E731
    uni = lambda *s: torch.rand(*s, generator=gen, device=device)  # noqa: E731
    fam = torch.arange(B, device=device) % 3
    cb = (0.5 * rnd(C)).to(bf) if with_cb else None
    k = 1.0 + (0.25 if with_cb else 0.0) + (1.0 if with_res else 0.0)
    x = rnd(B, D)
    sign = torch.where(uni(B, 1) < 0.5, -1.0, 1.0)
    x = torch.where((fam == 1).unsqueeze(1), x + 8 * math.sqrt(k) * sign, x)
    c = 4 * uni(B, 1) - 2
    noise = torch.where((torch.arange(B, device=device) % 2 == 1).unsqueeze(1), 2.0 ** -8 * rnd(B, D), torch.zeros(B, D, device=device))
    flat = c + noise - (cb.float().repeat(D // C) if with_cb else 0.0)
    x = torch.where((fam == 2).unsqueeze(1), flat, x).to(bf)
    res = None
    if with_res:
        res = torch.where((fam == 2).unsqueeze(1), torch.zeros(B, D, device=device), rnd(B, D)).to(bf)
    g = (0.5 + uni(D)).to(bf)
    b = ((-2.0 - uni(D)) if beta_neg else (uni(D) - 0.5)).to(bf)
    return x, res, cb, g, b


# ------------------------------------------------------------------------------------------------
# encoder (conv1 + bias + LayerNorm + ReLU from the observation)
def encoder_conv(obs, w1, b1):
    """Pre-LayerNorm map z [n, 4800] in HWC order and its bound. The kernel builds it in fp32 (dense
    part: at most 6 additions of w1 values, gam(8) |.|) and stores it as bf16, then adds every sparse
    object's 9 taps into the bf16 map, one more bf16 rounding per object hitting the position. Every
    intermediate is at most Zabs = conv(obs, |w1|) + |b1| in magnitude (obs is 0/1), so after 1 + k
    roundings: |z' - z| <= ((1 + UB)^(1 + k) - 1 + gam(8)) Zabs, k = sparse bits within the 3x3 window.
    When w1 and b1 are multiples of 2^-4, every partial sum at a position is a multiple of 2^-4 of
    magnitude at most Zabs; where Zabs < 16 that is at most 255 units, 8 significant bits, which bf16
    (and fp32) hold exactly, so there no rounding happens and the bound is 0."""
    o = obs.double()
    w = w1.double()
    z = F.conv2d(o, w, b1.double(), padding=1)
    zabs = F.conv2d(o, w.abs(), b1.double().abs(), padding=1)
    k = F.conv2d(o[:, 2:].sum(1, keepdim=True), torch.ones(1, 1, 3, 3, dtype=torch.float64, device=o.device), padding=1)
    ez = (torch.pow(1 + UB, 1 + k) - 1 + gam(8)) * zabs
    on_grid = lambda t: bool(torch.equal(t * 16, (t * 16).round()))  # noqa: E731
    if on_grid(w) and on_grid(b1.double()):
        ez = torch.where(zabs < 16, torch.zeros_like(ez), ez)
    hwc = lambda t: t.permute(0, 2, 3, 1).reshape(t.shape[0], -1)  # noqa: E731
    return hwc(z), hwc(ez.expand_as(z))


def from_hwc(t):
    return t.reshape(t.shape[0], BOARD_H, BOARD_W, -1).permute(0, 3, 1, 2)


class EncoderWeightGrad:
    """dw1 / db1 references and bounds, accumulated over sample chunks. The kernel sums its bf16 dz'
    (|dz' - dz| <= e_dz) over the taps: white and sparse taps where the observation bit is set, the
    black taps as (sum over all in-board taps) - (white taps) -- so a black tap's error is bounded by the
    sums over ALL in-board taps, not only the black ones:
      bound = sum_taps e_dz + gam(depth) sum_taps (|dz| + e_dz)        (taps: set bits; black: all, twice)"""

    def __init__(self, device):
        self.dw = torch.zeros(32, 12, 3, 3, dtype=torch.float64, device=device)
        self.ew, self.aw = torch.zeros_like(self.dw), torch.zeros_like(self.dw)
        self.db = torch.zeros(32, dtype=torch.float64, device=device)
        self.eb, self.ab = torch.zeros_like(self.db), torch.zeros_like(self.db)

    def add(self, obs, dz, e_dz):
        o = obs.double()
        dz, e_dz = from_hwc(dz), from_hwc(e_dz)
        cw = lambda inp, g: torch.nn.grad.conv2d_weight(inp, (32, inp.shape[1], 3, 3), g, padding=1)  # noqa: E731
        self.dw += cw(o, dz)
        e, a = cw(o, e_dz), cw(o, dz.abs() + e_dz)
        ones = torch.ones_like(o[:, :1])
        e[:, :1] = cw(ones, e_dz)
        a[:, :1] = 2 * cw(ones, dz.abs() + e_dz)
        self.ew += e
        self.aw += a
        self.db += dz.sum((0, 2, 3))
        self.eb += e_dz.sum((0, 2, 3))
        self.ab += (dz.abs() + e_dz).sum((0, 2, 3))

    def bounds(self, depth):
        return self.ew + gam(depth) * self.aw, self.eb + gam(depth) * self.ab


def exact_encoder_weights(gen, device):
    """w1 in {-1, 0, 1} 2^-4 and b1 multiples of 2^-4 with |b1| <= 1: every conv value and every partial
    sum of the sparse additions is a multiple of 2^-4 below 16 (at most 108 taps + 1), which bf16 holds
    exactly, so the kernel's pre-LayerNorm map is exact; its row sum (below 2^24 units of 2^-4) too."""
    w1 = torch.randint(-1, 2, (32, 12, 3, 3), generator=gen, device=device).float() * 2.0 ** -4
    b1 = torch.randint(-16, 17, (32,), generator=gen, device=device).float() * 2.0 ** -4
    return w1, b1


def exact_mean(z):
    """fp32(sum * fp32(1/4800)) of an exactly summed row: what the kernel returns when z is exact."""
    s = z.sum(1).float()  # exact: an integer count of 2^-4 below 2^24
    return (s * torch.tensor(1.0 / z.shape[1], dtype=torch.float32, device=z.device)).double()


# ------------------------------------------------------------------------------------------------
# conv3x3 weight gradient
def wgrad_ref(dy, x):
    """dW [cout, 3, 3, cin] (the kernel's layout) of a 3x3 / padding-1 convolution, from channels-last
    [n, 10, 15, c] operands, in float64, and sum |dy x| over the same terms."""
    d, xx = dy.double().permute(0, 3, 1, 2), x.double().permute(0, 3, 1, 2)
    cw = lambda inp, g: torch.nn.grad.conv2d_weight(inp, (g.shape[1], inp.shape[1], 3, 3), g, padding=1)  # noqa: E731
    return cw(xx, d).permute(0, 2, 3, 1), cw(xx.abs(), d.abs()).permute(0, 2, 3, 1)


def wgrad_depth(B, cin, sms):
    """Chain length of the tcgen05 kernel: a part of ceil(B / parts) samples is 10 MMAs of 16 positions
    per sample into one TMEM accumulator, then the parts are summed in fp32."""
    parts = max(1, min(sms // (3 if cin == 128 else 1), B))
    return 10 * -(-B // parts), parts


def wgrad_bound(absum, B, cin, sms):
    """Tensor-core MMAs add their K = 16 exact bf16 products to the fp32 accumulator with the
    significands aligned to the largest and truncated (Fasi et al., PeerJ CS 2021): at most
    (K + 1) 2^-23 times (|acc| + sum|products|) per MMA. Over n MMAs and `parts` fp32 additions:
      |dW' - dW| <= (n 17 2^-23 + gam(parts + 1)) sum|dy x|"""
    n, parts = wgrad_depth(B, cin, sms)
    return (n * 17 * 2.0 ** -23 + gam(parts + 1)) * absum
