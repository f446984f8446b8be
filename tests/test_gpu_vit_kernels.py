"""Operator tests of the depth-network kernels (csrc/depth_kernels.cu, csrc/zoe_kernels.cu) and of the ViT GEMM shapes.

Each GPU test drives one kernel through its C export and compares it with a float64 evaluation of the same upstream
operation on the exact fp16 / fp32 operands the kernel receives, rounded to fp16 only where the kernel stores fp16.
Outputs are filled with a sentinel before each call and followed by a guard band that must keep it, so a stray write
shows up as a value mismatch.  The CPU tests (no GPU marker) evaluate plausible wrong variants of each operator with
the same references and show that every one lands at least 5x outside the bound its GPU test uses.

Interpolation coordinates follow ATen's align_corners=True rule for fp16 / fp32 tensors: the source coordinate
scale * dst is an fp32 number (upsample_bilinear2d computes it in its fp32 accumulate type), everything after it is
float64 here.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.util import log_metric
from nunif_b200 import _lib
from oracle.zoedepth import relative_position_index

DEV = "cuda:0"
LOG2E = 1.4426950408889634
GUARD = 1 << 16          # guard-band elements after every output
SENT16 = 1234.0          # fp16 sentinel (exact)
SENT32 = -7777.0         # fp32 sentinel


# ------------------------------------------------------------------------------------------ helpers
def ulp16(x):
    """Spacing of fp16 numbers at |x| (subnormal spacing 2^-24 below 2^-14): the power of two of |x| (exponent bits of
    the float64), times 2^-10."""
    bits = x.double().abs().clamp_min(2.0 ** -14).view(torch.int64) & 0x7FF0000000000000
    return bits.view(torch.float64) * 2.0 ** -10


def guarded(n, dtype, fill, device=DEV):
    """A flat buffer of n + GUARD elements filled with `fill`; returns (buffer, first n elements)."""
    buf = torch.full((n + GUARD,), fill, dtype=dtype, device=device)
    return buf, buf[:n]


def assert_guard(buf, n, fill, what):
    tail = buf[n:]
    assert bool((tail == fill).all()), f"{what}: write past the end of the output"


def ac_coords(n_in, n_out):
    """ATen bilinear align_corners=True: (i0, i1, l0, l1) per destination index (fp32 source coordinate)."""
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0)
    src = (np.float32(scale) * np.arange(n_out, dtype=np.float32)).astype(np.float32)
    i0 = np.minimum(np.floor(src).astype(np.int64), n_in - 1)
    i1 = np.minimum(i0 + 1, n_in - 1)
    l1 = src.astype(np.float64) - i0
    return torch.from_numpy(i0), torch.from_numpy(i1), torch.from_numpy(1.0 - l1), torch.from_numpy(l1)


def interp_ac(x, H, W, align_corners=True):
    """float64 bilinear resize of NHWC x [B][h][w][C] to [B][H][W][C]."""
    x = x.double()
    if not align_corners:
        return F.interpolate(x.permute(0, 3, 1, 2), (H, W), mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    dev = x.device
    y0, y1, hy, ly = (t.to(dev) for t in ac_coords(x.shape[1], H))
    x0, x1, hx, lx = (t.to(dev) for t in ac_coords(x.shape[2], W))
    hx, lx = hx.view(1, 1, W, 1), lx.view(1, 1, W, 1)
    top = hx * x[:, y0][:, :, x0] + lx * x[:, y0][:, :, x1]
    bot = hx * x[:, y1][:, :, x0] + lx * x[:, y1][:, :, x1]
    return hy.view(1, H, 1, 1) * top + ly.view(1, H, 1, 1) * bot


def bilinear_bound(x, ref16, H, W):
    """1 fp16 ulp of fp16(ref64), plus 4 * 2^-24 * bilinear(|x|): the fp32 rounding of the three-level lerp.  Without the
    second term outputs where corners of size ~10 cancel to ~0 miss 1 ulp (the subnormal spacing 6e-8) in any fp32
    evaluation; on a B200 the kernel missed it by up to 5 such ulps (3e-7) at (224, 392) -> (392, 686)."""
    return ulp16(ref16) + 4 * 2.0 ** -24 * interp_ac(x.double().abs(), H, W)


def report(name, err, bound, **kv):
    """Log max / mean error and the bound at the worst element; return max(err / bound)."""
    ratio = (err / bound)
    i = int(torch.argmax(ratio.flatten()))
    r = float(ratio.flatten()[i])
    log_metric(name, **kv, err_max=f"{float(err.max()):.3e}", err_mean=f"{float(err.mean()):.3e}",
               bound_at_worst=f"{float(bound.flatten()[i]):.3e}", err_over_bound=f"{r:.4f}")
    return r


def stream():
    return _lib.stream_ptr()


# ------------------------------------------------------------------------------------------ float64 references
def rel_bias_ref(table, ph, pw, cls_swapped=False):
    """MiDaS beit.py relative-position gather, times log2 e in fp32 (what zoe_expand_rel_bias stores): [heads][N][N]."""
    idx = relative_position_index(ph, pw).to(table.device)
    if cls_swapped:   # nrd-2 <-> nrd-3 (class-token row and column entries exchanged)
        nrd = (2 * ph - 1) * (2 * pw - 1) + 3
        a, b = idx == nrd - 2, idx == nrd - 3
        idx = idx.clone()
        idx[a], idx[b] = nrd - 3, nrd - 2
    n = ph * pw + 1
    return (table[idx.view(-1)].view(n, n, -1).permute(2, 0, 1) * torch.tensor(LOG2E, dtype=torch.float32)).contiguous()


def attention_ref(qkv, B, N, heads, bias=None, variant=None):
    """softmax(q k^T / 8 + bias / log2 e) v in float64; qkv fp16 [B*N][3*heads*64] as reshape(B, N, 3, heads, 64);
    bias fp32 [heads][N][>= N] (log2 units).  Returns (out [B*N][heads*64], per-(image, head) max|v| [B][heads])."""
    x = qkv.view(B, N, 3, heads, 64).double()
    q, k, v = (x[:, :, i].transpose(1, 2) for i in range(3))          # [B][heads][N][64]
    scale = (1.0 if variant == "no_scale" else 0.125) * LOG2E
    if variant == "tail_unmasked":   # the padded keys of the last 64-block read as copies of key N-1
        pad = -N % 64
        k = torch.cat([k, k[:, :, -1:].expand(-1, -1, pad, -1)], 2)
        v = torch.cat([v, v[:, :, -1:].expand(-1, -1, pad, -1)], 2)
    out = torch.empty(B, heads, N, 64, dtype=torch.float64, device=qkv.device)
    hc = max(1, min(heads, (1 << 25) // (N * N)))                     # bounded N x N score chunks
    for b in range(B):
        for h0 in range(0, heads, hc):
            h1 = min(heads, h0 + hc)
            s = q[b, h0:h1] @ k[b, h0:h1].transpose(-1, -2) * scale
            if bias is not None:
                bb = bias[h0:h1, :, :N].double()
                if variant == "bias_transposed":
                    bb = bb.transpose(-1, -2)
                s = s + bb
            out[b, h0:h1] = torch.softmax(s * math.log(2.0), -1) @ v[b, h0:h1]
    vmax = x[:, :, 2].abs().amax(dim=(1, 3))                           # [B][heads]
    return out.transpose(1, 2).reshape(B * N, heads * 64), vmax


def attention_bound(ref, vmax, B, N, heads):
    """1 fp16 ulp of |ref| + 2^-10 max|v| of that (image, head): P is rounded to fp16 before PV."""
    vb = vmax.view(B, 1, heads, 1).expand(B, N, heads, 64).reshape(B * N, heads * 64)
    return ulp16(ref) + 2.0 ** -10 * vb


def layernorm_ref(x32, w, b, eps=1e-6):
    x = x32.double()
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w.double() + b.double()


def layernorm_bound(x32, w, ref16, eps=1e-6):
    """1 fp16 ulp of fp16(ref64), plus the fp32 rounding of the row mean carried into every output: the kernel's sum has
    at most 15 rounding levels (dim / 128 float4 per lane, pairwise inside the float4, 5 shuffle levels), so the mean
    is off by <= 16 * 2^-24 * mean|x|, and that error times rstd * |w| lands on each output.  Without this term a row
    with a common offset of 50 cannot meet 1 ulp at its near-zero outputs in any fp32 evaluation (an fp32 emulation
    misses by up to 127 ulp = 1.2e-5 there); it is ~5e-7 on the std-1e-3 rows, where the eps is checked."""
    x = x32.double()
    rstd = 1.0 / torch.sqrt(x.var(-1, unbiased=False, keepdim=True) + eps)
    return ulp16(ref16) + 16 * 2.0 ** -24 * x.abs().mean(-1, keepdim=True) * rstd * w.double().abs()


def inv_attractor(dx):
    return dx / (1.0 + 300.0 * dx * dx)


def attractor_ref(apre, na, prev, H, W, variant=None):
    """AttractorLayerUnnormed: c = bilinear_ac(prev_bin), a = softplus(apre[:, :na]); c + mean_j inv_attractor(a_j - c)."""
    B = prev.shape[0]
    c = interp_ac(prev, H, W).reshape(B * H * W, 64)
    a = F.softplus(apre[:, :na].double())
    delta = inv_attractor(a.unsqueeze(2) - c.unsqueeze(1)).sum(1)
    return c + (delta if variant == "sum" else delta / na)


def attractor_bound(prev):
    return 1e-5 * float(prev.max() - prev.min())


def log_binom(n, k, eps=1e-7):
    n = n + eps
    k = k + eps
    return n * torch.log(n) - k * torch.log(k) - (n - k) * torch.log(n - k + eps)


def clb_ref(g, w2, b2, bins, H, W, variant=None):
    """ConditionalLogBinomial tail on the fp32 conv output (not rounded to fp16) + sum_k prob_k * centre_k.
    Returns depth [P], temperature [P], bound [P]."""
    B = bins.shape[0]
    a = F.softplus(g[:, :80].double() @ w2.double().t() + b2.double()) + 1e-4
    p = a[:, 0] / (a[:, 0] + a[:, 1])
    temp = (50.0 - 0.0212) * (a[:, 2] / (a[:, 2] + a[:, 3])) + 0.0212
    if variant == "no_clamp":
        lp, lq = torch.log(p), torch.log(1 - p)
    else:
        lp, lq = torch.log(p.clamp(1e-4, 1)), torch.log((1 - p).clamp(1e-4, 1))
    k = torch.arange(64, dtype=torch.float64, device=g.device)
    y = (log_binom(torch.tensor(63.0, dtype=torch.float64, device=g.device), k) + k * lp[:, None] + (63 - k) * lq[:, None])
    prob = torch.softmax(y / temp[:, None], -1)
    c = interp_ac(bins, H, W).reshape(B * H * W, 64)
    depth = (prob * c).sum(1)
    # fp32 error analysis of the kernel: the logit numerator is a sum of terms whose magnitudes add up to
    # S = 3 * 63 ln 63 (Stirling log-binomial, cancelling to <= 42) + 63 (|ln p| + |ln(1-p)|) <= ~1370; about eight fp32
    # roundings of size <= 2^-24 S each put its error below 2^-21 S, i.e. 2^-21 S / T on the logits (~0.03 at
    # T = 0.0212, logits up to ~3e4 there).  A logit error d moves sum_k prob_k c_k by at most d * (max - min centre).
    # The fp32 sum of 64 prob * centre products and the division add <= 2^-17 max|centre|.
    S = 3 * 63 * math.log(63) + 63 * (lp.abs() + lq.abs())
    rng = c.max(1).values - c.min(1).values
    bound = 2.0 ** -21 * S / temp * rng + 2.0 ** -17 * c.abs().max(1).values
    return depth, temp, bound


# ------------------------------------------------------------------------------------------ operand generators
def make_qkv(B, N, heads, dist, gen, device):
    """(a) "normal": N(0, 1); (b) "peaked": q x 10, logits span about +-40; (c) "dominant": one key with a logit 40 above
    the rest, key N-1 (the last, partial 64-block) for even rows and key 0 (block 0) for odd rows."""
    x = torch.randn(B, N, 3, heads, 64, generator=gen, device=device)
    if dist == "peaked":
        x[:, :, 0] *= 10
    elif dist == "dominant":
        q, k = x[:, :, 0], x[:, :, 1]
        q[..., :2] = 0
        k[..., :2] = 0
        k[:, N - 1, :, 0] = 8
        k[:, 0, :, 1] = 8
        q[:, 0::2, :, 0] = 40
        q[:, 1::2, :, 1] = 40
    return x.half().reshape(B * N, 3 * heads * 64).contiguous()


def grid_for(N):
    """A (ph, pw) token grid with ph * pw + 1 == N: the real DA / ZoeD grids, else the squarest factorisation."""
    real = {769: (24, 32), 1057: (24, 44), 1370: (37, 37), 1373: (28, 49), 4129: (48, 86)}
    if N in real:
        return real[N]
    P = N - 1
    ph = max(d for d in range(1, int(P ** 0.5) + 1) if P % d == 0)
    return ph, P // ph


def make_bias(N, heads, ldb, gen, device):
    """Relative-position bias [heads][N][ldb] (log2 units) as zoe_expand_rel_bias stores it, padding columns [N, ldb) NaN,
    rows 2 mod 5 pushed down by 1000 on the keys of block 0.  Returns (buffer with guard band, [heads][N][ldb] view)."""
    buf = torch.full((heads * N * ldb + GUARD,), float("nan"), dtype=torch.float32, device=device)
    bias = buf[:heads * N * ldb].view(heads, N, ldb)
    if N == 1:
        bias[:, :, :1] = torch.randn(heads, 1, 1, generator=gen, device=device) * 3
    else:
        ph, pw = grid_for(N)
        table = torch.randn((2 * ph - 1) * (2 * pw - 1) + 3, heads, generator=gen, device=device) * 3
        bias[:, :, :N] = rel_bias_ref(table, ph, pw)
    bias[:, 2::5, :min(N, 64)] -= 1000.0
    return buf, bias


def make_ln_rows(rows, dim, gen, device):
    """Rows of three kinds, cycling: N(0, 1); N(0, 1) + 50; N(0, 1e-3) (where eps = 1e-6 versus 1e-5 matters)."""
    x = torch.randn(rows, dim, generator=gen, device=device)
    scale = torch.tensor([1.0, 1.0, 1e-3], device=device).repeat(rows // 3 + 1)[:rows, None]
    offset = torch.tensor([0.0, 50.0, 0.0], device=device).repeat(rows // 3 + 1)[:rows, None]
    delta = (torch.randn(rows, dim, generator=gen, device=device) * 0.5 * scale).half()
    return (x * scale + offset).float(), delta, scale


def make_attractor_inputs(B, h, w, H, W, na, gen, device):
    """prev_bin log-uniform in [0.1, 10]; apre [P][16] whose softplus lands near a centre (|dx| ~ 0), near 1/sqrt(300) from
    one (the inv_attractor extremum), anywhere in [0.1, 10], or is a pre-activation above the threshold 20; columns
    na..15 hold 1e4 and must be ignored."""
    prev = torch.exp(torch.empty(B, h, w, 64, device=device).uniform_(math.log(0.1), math.log(10.0), generator=gen)).float()
    P = B * H * W
    c = interp_ac(prev, H, W).reshape(P, 64)
    kj = torch.randint(0, 64, (P, 16), generator=gen, device=device)
    cj = torch.gather(c, 1, kj)
    sign = torch.randint(0, 2, (P, 16), generator=gen, device=device).double() * 2 - 1
    kind = (torch.arange(P, device=device)[:, None] + torch.arange(16, device=device)[None]) % 4
    u = torch.rand(P, 16, generator=gen, device=device, dtype=torch.float64)
    target = torch.where(kind == 0, cj + sign * 2e-3 * u,
                         torch.where(kind == 1, cj + sign / math.sqrt(300.0), 0.1 + 9.9 * u)).clamp_min(1e-3)
    pre = torch.log(torch.expm1(target))
    pre = torch.where(kind == 3, 20.5 + 20 * u, pre)
    apre = pre.half()
    apre[:, na:] = 1e4
    return prev, apre.contiguous()


def make_clb_inputs(B, h, w, H, W, gen, device):
    """g [P][96] fp16 (columns 80..95 NaN, never read); channels 0..3 sweep [-12, 12] independently and w2 routes channel o
    to output o, so p reaches both 1e-4 clamps, both p-terms can be near the 1e-4 epsilon, and the temperature sweeps
    [0.0212, 50]; the other 76 channels add small N(0, 1) * 0.02 terms.  Bin centres log-uniform in [0.1, 10]."""
    P = B * H * W
    g = torch.randn(P, 96, generator=gen, device=device)
    g[:, :4] = torch.empty(P, 4, device=device).uniform_(-12, 12, generator=gen)
    g[:, 80:] = float("nan")
    w2 = torch.randn(4, 80, generator=gen, device=device) * 0.02
    w2[:, :4] = torch.eye(4, device=device)
    b2 = torch.randn(4, generator=gen, device=device) * 0.1
    bins = torch.exp(torch.empty(B, h, w, 64, device=device).uniform_(math.log(0.1), math.log(10.0), generator=gen))
    return g.half().contiguous(), w2.contiguous(), b2.contiguous(), bins.float().contiguous()


# ------------------------------------------------------------------------------------------ GPU: attention
ATTN_CASES = ([(N, heads, B) for N in (1, 2, 63, 64, 65, 127, 128, 129) for heads, B in ((4, 1), (6, 3), (12, 1), (16, 3))]
              + [(769, 16, 3), (1057, 16, 1), (1370, 6, 3), (1370, 12, 1), (1373, 6, 1), (1373, 16, 3), (4129, 16, 1)])
DISTS = ("normal", "peaked", "dominant")


def run_attention(qkv, B, N, heads, bias=None, ldb=0):
    buf, out = guarded(B * N * heads * 64, torch.float16, SENT16)
    _lib.check(_lib.lib().nb200_vit_attention_f16(_lib.ptr(qkv), _lib.ptr(out), B, N, heads, _lib.ptr(bias), ldb, stream()))
    torch.cuda.synchronize()
    assert_guard(buf, out.numel(), SENT16, "attention")
    return out.view(B * N, heads * 64)


@pytest.mark.gpu
@pytest.mark.parametrize("N,heads,B", ATTN_CASES)
def test_vit_attention(N, heads, B):
    gen = torch.Generator(device=DEV).manual_seed(N * 131 + heads * 7 + B)
    for dist in DISTS:
        qkv = make_qkv(B, N, heads, dist, gen, DEV)
        got = run_attention(qkv, B, N, heads)
        ref, vmax = attention_ref(qkv, B, N, heads)
        r = report("vit_attention", (got.double() - ref).abs(), attention_bound(ref, vmax, B, N, heads), N=N, heads=heads, B=B,
                   dist=dist)
        assert r <= 1.0, (dist, r)


@pytest.mark.gpu
@pytest.mark.parametrize("N,heads,B", ATTN_CASES)
def test_vit_attention_rel_bias(N, heads, B):
    """BEiT attention: the bias is shared by the B images, its padding columns [N, ldb) are NaN and must be masked."""
    gen = torch.Generator(device=DEV).manual_seed(N * 131 + heads * 7 + B + 1)
    ldb0 = -(-N // 64) * 64
    for dist in DISTS:
        for ldb in (ldb0, ldb0 + 10):
            qkv = make_qkv(B, N, heads, dist, gen, DEV)
            bbuf, bias = make_bias(N, heads, ldb, gen, DEV)
            before = bbuf.clone()
            got = run_attention(qkv, B, N, heads, bias, ldb)
            assert torch.equal(bbuf.isnan(), before.isnan()) and torch.equal(bbuf.nan_to_num(), before.nan_to_num())
            ref, vmax = attention_ref(qkv, B, N, heads, bias)
            r = report("vit_attention_bias", (got.double() - ref).abs(), attention_bound(ref, vmax, B, N, heads), N=N, heads=heads,
                       B=B, dist=dist, ldb=ldb)
            assert r <= 1.0, (dist, ldb, r)


@pytest.mark.gpu
def test_vit_attention_rejects_bad_bias_stride():
    N, heads, B = 65, 4, 1
    gen = torch.Generator(device=DEV).manual_seed(3)
    qkv = make_qkv(B, N, heads, "normal", gen, DEV)
    bias = torch.zeros(heads * N * 130, device=DEV)
    for ldb in (129, 126, 64):        # odd; >= N but not whole 64-key blocks; < N
        buf, out = guarded(B * N * heads * 64, torch.float16, SENT16)
        rc = _lib.lib().nb200_vit_attention_f16(_lib.ptr(qkv), _lib.ptr(out), B, N, heads, _lib.ptr(bias), ldb, stream())
        torch.cuda.synchronize()
        assert rc != 0 and b"stride" in _lib.lib().nb200_last_error(), ldb
        assert bool((buf == SENT16).all()), ldb


# ------------------------------------------------------------------------------------------ GPU: add + LayerNorm
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [256, 384, 768, 1024])
@pytest.mark.parametrize("rows", [1, 7, 8, 9, 2746, 4129])
def test_vit_add_layernorm(dim, rows):
    gen = torch.Generator(device=DEV).manual_seed(rows * 3 + dim)
    x0, delta, _ = make_ln_rows(rows, dim, gen, DEV)
    w = (1 + 0.1 * torch.randn(dim, generator=gen, device=DEV)).float()
    b = (0.1 * torch.randn(dim, generator=gen, device=DEV)).float()
    n = rows * dim
    for use_delta, use_out in ((True, True), (False, True), (True, False)):
        xbuf, x = guarded(n, torch.float32, SENT32)
        x.copy_(x0.flatten())
        obuf, out = guarded(n, torch.float16, SENT16)
        d = delta if use_delta else None
        _lib.check(_lib.lib().nb200_vit_add_layernorm(_lib.ptr(x), _lib.ptr(d), _lib.ptr(w), _lib.ptr(b),
                                                      _lib.ptr(out if use_out else None), rows, dim, stream()))
        torch.cuda.synchronize()
        assert_guard(xbuf, n, SENT32, "residual")
        want_x = x0 + delta.float() if use_delta else x0          # the fp32 residual add, IEEE-rounded like the kernel's
        assert torch.equal(x.view(rows, dim), want_x), "residual not bit-exact"
        if not use_out:
            assert bool((obuf == SENT16).all()), "out written although null"
            continue
        assert_guard(obuf, n, SENT16, "layernorm out")
        ref = layernorm_ref(x.view(rows, dim), w, b).half().double()
        r = report("vit_add_layernorm", (out.view(rows, dim).double() - ref).abs(), layernorm_bound(x.view(rows, dim), w, ref),
                   rows=rows, dim=dim, delta=use_delta)
        assert r <= 1.0, (use_delta, r)


@pytest.mark.gpu
def test_vit_add_layernorm_rejects_dim():
    x = torch.ones(4 * 512, device=DEV)
    w = torch.ones(512, device=DEV)
    out = torch.full((4 * 512,), SENT16, dtype=torch.float16, device=DEV)
    rc = _lib.lib().nb200_vit_add_layernorm(_lib.ptr(x), None, _lib.ptr(w), _lib.ptr(w), _lib.ptr(out), 4, 512, stream())
    torch.cuda.synchronize()
    assert rc != 0 and b"dim" in _lib.lib().nb200_last_error()
    assert bool((x == 1).all()) and bool((out == SENT16).all())


# ------------------------------------------------------------------------------------------ GPU: BEiT bias expansion
@pytest.mark.gpu
@pytest.mark.parametrize("ph,pw", [(24, 44), (44, 24), (24, 32), (6, 6), (1, 5), (5, 1), (1, 1)])
@pytest.mark.parametrize("heads", [4, 16])
def test_zoe_expand_rel_bias(ph, pw, heads):
    gen = torch.Generator(device=DEV).manual_seed(ph * 100 + pw + heads)
    N = ph * pw + 1
    ldb = -(-N // 64) * 64
    table = torch.randn((2 * ph - 1) * (2 * pw - 1) + 3, heads, generator=gen, device=DEV) * 3
    buf, flat = guarded(heads * N * ldb, torch.float32, SENT32)
    _lib.check(_lib.lib().nb200_zoe_expand_rel_bias(_lib.ptr(table), ph, pw, heads, _lib.ptr(flat), ldb, stream()))
    torch.cuda.synchronize()
    assert_guard(buf, flat.numel(), SENT32, "rel bias")
    got = flat.view(heads, N, ldb)
    assert bool((got[:, :, N:] == SENT32).all()), "padding columns written"
    ref = rel_bias_ref(table, ph, pw)
    mism = int((got[:, :, :N] != ref).sum())
    log_metric("zoe_expand_rel_bias", ph=ph, pw=pw, heads=heads, mismatches=mism, bound=0)
    assert mism == 0


# ------------------------------------------------------------------------------------------ GPU: attractor
@pytest.mark.gpu
@pytest.mark.parametrize("B,h,w,H,W", [(2, 12, 16, 24, 32), (1, 24, 44, 24, 44), (1, 5, 7, 10, 14)])
@pytest.mark.parametrize("na", [16, 8, 4, 1])
def test_zoe_attractor(B, h, w, H, W, na):
    gen = torch.Generator(device=DEV).manual_seed(h * w + H + na)
    prev, apre = make_attractor_inputs(B, h, w, H, W, na, gen, DEV)
    n = B * H * W * 64
    buf, out = guarded(n, torch.float32, SENT32)
    _lib.check(_lib.lib().nb200_zoe_attractor(_lib.ptr(apre), 16, na, _lib.ptr(prev), B, h, w, H, W, _lib.ptr(out), stream()))
    torch.cuda.synchronize()
    assert_guard(buf, n, SENT32, "attractor")
    ref = attractor_ref(apre, na, prev, H, W)
    err = (out.view(B * H * W, 64).double() - ref).abs()
    r = report("zoe_attractor", err, torch.full_like(err, attractor_bound(prev)), h=h, w=w, H=H, W=W, na=na)
    assert r <= 1.0, r


# ------------------------------------------------------------------------------------------ GPU: log-binomial head
@pytest.mark.gpu
@pytest.mark.parametrize("B,h,w,H,W", [(2, 24, 32, 48, 64), (1, 24, 44, 48, 88), (1, 7, 9, 14, 18)])
def test_zoe_clb_final(B, h, w, H, W):
    gen = torch.Generator(device=DEV).manual_seed(h * w + H * W)
    g, w2, b2, bins = make_clb_inputs(B, h, w, H, W, gen, DEV)
    P = B * H * W
    buf, out = guarded(P, torch.float32, SENT32)
    _lib.check(_lib.lib().nb200_zoe_clb_final(_lib.ptr(g), 96, _lib.ptr(w2), _lib.ptr(b2), _lib.ptr(bins), B, h, w, H, W,
                                              _lib.ptr(out), stream()))
    torch.cuda.synchronize()
    assert_guard(buf, P, SENT32, "clb_final")
    ref, temp, bound = clb_ref(g, w2, b2, bins, H, W)
    err = (out.double() - ref).abs()
    c = interp_ac(bins, H, W).reshape(P, 64)
    rel = err / (c.max(1).values - c.min(1).values)
    i = int(torch.argmax(rel))
    r = report("zoe_clb_final", err, bound, h=h, w=w, H=H, W=W, temp_min=f"{float(temp.min()):.4f}",
               temp_max=f"{float(temp.max()):.2f}", worst_err_over_range=f"{float(rel[i]):.3e}",
               worst_pixel_temp=f"{float(temp[i]):.4f}")
    assert r <= 1.0, r
    assert float(temp.min()) < 0.022 and float(temp.max()) > 49.0       # the temperature sweep really happened


# ------------------------------------------------------------------------------------------ GPU: DPT bilinear
@pytest.mark.gpu
@pytest.mark.parametrize("B,h,w,C,H,W", [(2, 19, 25, 64, 37, 49), (1, 14, 25, 32, 28, 49), (1, 48, 64, 32, 84, 112),
                                         (1, 224, 392, 32, 392, 686), (2, 1, 3, 8, 2, 1), (1, 3, 1, 16, 1, 2),
                                         (1, 37, 37, 128, 74, 74)])
def test_dpt_upsample_bilinear(B, h, w, C, H, W):
    gen = torch.Generator(device=DEV).manual_seed(h * w + C + H)
    x = (torch.randn(B, h, w, C, generator=gen, device=DEV) * 4).half()
    n = B * H * W * C
    buf, out = guarded(n, torch.float16, SENT16)
    _lib.check(_lib.lib().nb200_dpt_upsample_bilinear_f16(_lib.ptr(x), B, h, w, C, _lib.ptr(out), H, W, stream()))
    torch.cuda.synchronize()
    assert_guard(buf, n, SENT16, "upsample")
    ref = interp_ac(x, H, W).half().double()
    r = report("dpt_upsample_bilinear", (out.view(B, H, W, C).double() - ref).abs(), bilinear_bound(x, ref, H, W), h=h, w=w,
               C=C, H=H, W=W)
    assert r <= 1.0, r


# ------------------------------------------------------------------------------------------ GPU: ViT GEMM shapes
GEMM_KN = [(384, 1152, 0), (384, 1536, 2), (1536, 384, 0), (768, 2304, 0), (3072, 768, 0), (1024, 3072, 0), (1024, 4096, 2),
           (4096, 1024, 0)]


def gemm_case(M, K, N, act, a_stride=False, out_gap=0):
    gen = torch.Generator(device=DEV).manual_seed(M * 7 + K * 3 + N)
    Ci = 2 * K if a_stride else K
    A = torch.full((M, Ci), float("nan"), dtype=torch.float16, device=DEV)
    A[:, :K] = torch.randn(M, K, generator=gen, device=DEV).half()
    Wt = (torch.randn(N, K, generator=gen, device=DEV) / K ** 0.5).half()
    bias = torch.randn(N, generator=gen, device=DEV)
    ldo = N + out_gap
    buf, flat = guarded(M * ldo, torch.float16, SENT16)
    _lib.check(_lib.lib().nb200_conv_gemm_f16(_lib.ptr(A), 1, 1, M, Ci, K, 0, _lib.ptr(Wt), N, _lib.ptr(bias), act,
                                              _lib.ptr(flat), ldo, 0, 0, None, 0, 0, 0, 0, 0, 0, stream()))
    torch.cuda.synchronize()
    assert_guard(buf, flat.numel(), SENT16, "gemm")
    out = flat.view(M, ldo)
    if out_gap:
        assert bool((out[:, N:] == SENT16).all()), "gap columns written"
    a, wt = A[:, :K].double(), Wt.double()
    ref = a @ wt.t() + bias.double()
    if act == 2:
        ref = F.gelu(ref)
    # 1 fp16 ulp of the stored result + the fp32 accumulation bound K 2^-23 sum|a w|
    bound = ulp16(ref) + K * 2.0 ** -23 * (a.abs() @ wt.abs().t())
    return report("vit_gemm", (out[:, :N].double() - ref).abs(), bound, M=M, K=K, N=N, act=act, a_stride=a_stride,
                  out_gap=out_gap)


@pytest.mark.gpu
@pytest.mark.parametrize("K,N,act", GEMM_KN)
@pytest.mark.parametrize("M", [769, 2114, 2746, 5480])
def test_vit_gemm_shapes(M, K, N, act):
    assert gemm_case(M, K, N, act) <= 1.0


@pytest.mark.gpu
def test_vit_gemm_strided_operands():
    assert gemm_case(2746, 1536, 384, 0, a_stride=True) <= 1.0          # A row stride 2 K, the unread half NaN
    assert gemm_case(769, 1024, 3072, 2, out_gap=64) <= 1.0             # ldo = N + 64, the gap keeps its sentinel


# ------------------------------------------------------------------------------------------ CPU: the bounds bite
def worst_ratio(wrong, ref, bound):
    return float(((wrong - ref).abs() / bound).max())


def test_attention_bound_catches_wrong_variants():
    gen = torch.Generator().manual_seed(0)
    B, N, heads = 1, 129, 2
    qkv = make_qkv(B, N, heads, "normal", gen, "cpu")
    ref, vmax = attention_ref(qkv, B, N, heads)
    bound = attention_bound(ref, vmax, B, N, heads)
    for variant in ("tail_unmasked", "no_scale"):
        wrong, _ = attention_ref(qkv, B, N, heads, variant=variant)
        assert worst_ratio(wrong, ref, bound) >= 5, variant
    ph, pw = grid_for(N)
    table = torch.randn((2 * ph - 1) * (2 * pw - 1) + 3, heads, generator=gen) * 3
    bias = rel_bias_ref(table, ph, pw)
    ref, vmax = attention_ref(qkv, B, N, heads, bias)
    bound = attention_bound(ref, vmax, B, N, heads)
    wrong, _ = attention_ref(qkv, B, N, heads, bias, variant="bias_transposed")
    assert worst_ratio(wrong, ref, bound) >= 5, "bias_transposed"
    wrong, _ = attention_ref(qkv, B, N, heads, rel_bias_ref(table, ph, pw, cls_swapped=True))
    assert worst_ratio(wrong, ref, bound) >= 5, "cls_swapped"


def test_layernorm_bound_catches_eps():
    gen = torch.Generator().manual_seed(1)
    x, _, _ = make_ln_rows(9, 384, gen, "cpu")
    w, b = torch.ones(384), torch.zeros(384)
    ref = layernorm_ref(x, w, b).half().double()
    wrong = layernorm_ref(x, w, b, eps=1e-5).half().double()
    assert worst_ratio(wrong, ref, layernorm_bound(x, w, ref)) >= 5


def test_bilinear_bound_catches_align_corners_false():
    gen = torch.Generator().manual_seed(2)
    x = (torch.randn(1, 19, 25, 8, generator=gen) * 4).half()
    ref = interp_ac(x, 37, 49).half().double()
    wrong = interp_ac(x, 37, 49, align_corners=False).half().double()
    assert worst_ratio(wrong, ref, bilinear_bound(x, ref, 37, 49)) >= 5
    assert torch.allclose(interp_ac(x, 37, 49), F.interpolate(x.double().permute(0, 3, 1, 2), (37, 49), mode="bilinear",
                                                              align_corners=True).permute(0, 2, 3, 1), atol=1e-5)


def test_log_binomial_bound_catches_missing_clamps():
    gen = torch.Generator().manual_seed(3)
    g, w2, b2, bins = make_clb_inputs(1, 8, 8, 16, 16, gen, "cpu")
    ref, temp, bound = clb_ref(g, w2, b2, bins, 16, 16)
    wrong, _, _ = clb_ref(g, w2, b2, bins, 16, 16, variant="no_clamp")
    assert worst_ratio(wrong, ref, bound) >= 5
    assert float(temp.min()) < 0.022 and float(temp.max()) > 49.0


def test_attractor_bound_catches_sum_instead_of_mean():
    gen = torch.Generator().manual_seed(4)
    for na in (16, 8, 4):
        prev, apre = make_attractor_inputs(1, 4, 5, 8, 10, na, gen, "cpu")
        ref = attractor_ref(apre, na, prev, 8, 10)
        wrong = attractor_ref(apre, na, prev, 8, 10, variant="sum")
        assert worst_ratio(wrong, ref, torch.full_like(ref, attractor_bound(prev))) >= 5, na
