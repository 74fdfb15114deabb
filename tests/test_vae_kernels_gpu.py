"""SD-VAE kernels (csrc/vae.cu, the nine `mdt_vae_*` entry points), the tcgen05 GEMM at the VAE's shapes, and the
building blocks of `vae._VaeBase`, each against a plain float64 reference of the same operation.

An end-to-end rel-L2 bound over ~30 convolutions cannot see an error that stays in one place (a wrong border row of
an im2col window, one GroupNorm group with wrong statistics, an unwritten pad column, image b reading image b+1), so
every kernel here is checked element by element:
  * every output buffer is prefilled with NaN, so an element the kernel should write but does not fails the test;
  * max-abs error is taken relative to the output scale (max |reference|), rel-L2 only in addition;
  * each bound is derived in the test's docstring from the arithmetic the kernel does, and the measured error is
    printed (`pytest -s`).
The CPU test checks the reference builders themselves (im2col in (ky, kx, c) column order times weights packed like
`_VaeBase._ready` == F.conv2d) so that the GPU tests compare against something known to be right."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import vae_encode_oracle as VE  # noqa: E402
from oracle import vae_oracle as VO  # noqa: E402

gpu = pytest.mark.gpu
f64, bf16 = torch.float64, torch.bfloat16
EPS = 1e-6     # GroupNorm eps (Normalize, autoencoder.py:34-35)


# ---- reference builders (float64, any device) ------------------------------------------------------------------------
def im2col_ref(x, ks=3, up=1, down=False, Kp=None):
    """x [B,C,H,W] -> A [B*Ho*Wo, Kp] with A[(b,y,x), (ky,kx,c)] = the ks x ks window of nearest-upsample(x) (padding
    ks // 2), or with down=True of F.pad(x, (0,1,0,1)) at stride 2; columns >= ks*ks*C are zero."""
    if up != 1:
        x = F.interpolate(x, scale_factor=float(up), mode="nearest")
    if down:
        cols = F.unfold(F.pad(x, (0, 1, 0, 1)), 3, stride=2)
        ks = 3
    else:
        cols = F.unfold(x, ks, padding=ks // 2)
    B, C = x.shape[:2]
    L = cols.shape[-1]
    A = cols.view(B, C, ks * ks, L).permute(0, 3, 2, 1).reshape(B * L, ks * ks * C)
    if Kp is not None and Kp > A.shape[1]:
        A = torch.cat([A, A.new_zeros(A.shape[0], Kp - A.shape[1])], 1)
    return A


def pack_weight(w):
    """Conv weight [Co,Ci,kh,kw] -> [Co, Kp] in (ky, kx, c) order, Ci padded to a multiple of 4 and K to a multiple of 8
    with zeros: the GEMM layout `_VaeBase._ready` builds."""
    co, ci, kh, kw = w.shape
    cp = (ci + 3) // 4 * 4
    wt = F.pad(w.permute(0, 2, 3, 1), (0, cp - ci))
    K = kh * kw * cp
    return F.pad(wt.reshape(co, K), (0, (K + 7) // 8 * 8 - K))


def pad_channels(x, c):
    return F.pad(x, (0, 0, 0, 0, 0, c - x.shape[1]))


def gn_sums_ref(rows, B, C):
    """[B,32,2] (sum, sum of squares) per (image, group) of pixel-major rows [B*P, C], in float64."""
    g = rows.double().view(B, -1, 32, C // 32)
    return torch.stack([g.sum((1, 3)), (g * g).sum((1, 3))], -1).contiguous()


def gn_mean_rstd(sums, n):
    """The mean and rstd `vae_im2col_kernel` derives from the sums (in float64)."""
    m = sums[..., 0] / n
    return m, (sums[..., 1] / n - m * m + EPS).rsqrt()


def to_rows(x):
    """[B,C,H,W] -> [B*H*W, C] pixel-major (the layout every VAE kernel works in)."""
    return x.permute(0, 2, 3, 1).reshape(-1, x.shape[1]).contiguous()


def to_nchw(rows, B, H, W):
    return rows.reshape(B, H, W, -1).permute(0, 3, 1, 2)


def swish(x):
    return x * torch.sigmoid(x)


def bf16_ulp(x):
    """Spacing of bf16 numbers at |x| (8 significant bits), for x in the normal range; 2^-133 below it."""
    _, e = torch.frexp(x.abs().double().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x, dtype=f64), e - 8)


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm()).item()


def max_rel(got, ref):
    """max |got - ref| / max |ref| (the error relative to the output scale)."""
    got, ref = got.double(), ref.double()
    assert torch.isfinite(got).all(), "non-finite output (an element the kernel should have written is still NaN)"
    return ((got - ref).abs().max() / (ref.abs().max() + 1e-300)).item()


def nan_full(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), dtype=dtype, device="cuda")


# ---- CPU: the reference builders -------------------------------------------------------------------------------------
def test_im2col_reference_times_packed_weights_is_conv2d():
    """im2col_ref @ pack_weight(w).T == F.conv2d in every mode the network uses (3x3 pad 1, 1x1, nearest-2x upsample,
    the stride-2 Downsample with (0,1,0,1) padding, RGB padded to 4 channels), float64: rounding only (1e-12)."""
    g = torch.Generator().manual_seed(0)
    B = 2
    for (H, W) in ((6, 10), (7, 5), (1, 1)):
        for ci, co, ks, up, down in ((8, 12, 3, 1, False), (8, 12, 1, 1, False), (8, 12, 3, 2, False),
                                     (8, 12, 3, 1, True), (3, 16, 3, 1, False), (4, 5, 3, 1, False)):
            if up == 2 and (H % 2 or W % 2):
                continue
            Hs, Ws = (2 * H, 2 * W) if down else (H // up, W // up)
            x = torch.randn(B, ci, Hs, Ws, generator=g, dtype=f64)
            w = torch.randn(co, ci, ks, ks, generator=g, dtype=f64)
            bias = torch.randn(co, generator=g, dtype=f64)
            wp = pack_weight(w)
            cp = (ci + 3) // 4 * 4
            assert wp.shape == (co, (ks * ks * cp + 7) // 8 * 8)
            A = im2col_ref(pad_channels(x, cp), ks, up, down, wp.shape[1])
            got = to_nchw(A @ wp.t() + bias, B, H, W)
            if down:
                ref = VE._downsample({"d.weight": w, "d.bias": bias}, "d", x)
            else:
                xu = F.interpolate(x, scale_factor=2.0, mode="nearest") if up == 2 else x
                ref = F.conv2d(xu, w, bias, padding=ks // 2)
            assert got.shape == ref.shape, (got.shape, ref.shape)
            assert max_rel(got, ref) < 1e-12, (H, W, ci, ks, up, down)
    # the sums helpers are GroupNorm's statistics
    x = torch.randn(3, 128, 5, 7, generator=g, dtype=f64) * 2 + 1
    m, rstd = gn_mean_rstd(gn_sums_ref(to_rows(x), 3, 128), 4 * 35)
    xn = (x.view(3, 32, -1) - m[..., None]) * rstd[..., None]
    assert max_rel(xn.view_as(x), F.group_norm(x, 32, eps=EPS)) < 1e-12


# ---- GPU: kernel parity -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ops():
    from maskdit_b200 import ops as o
    return o


@gpu
@pytest.mark.parametrize("H,W", [(8, 8), (48, 80), (5, 7)])
def test_image_to_rows(ops, H, W):
    """NCHW RGB -> pixel-major rows with a zero 4th channel, mirrored along W for flip = 1.  A copy: exact."""
    torch.manual_seed(20)
    B = 2
    x = torch.rand(B, 3, H, W, device="cuda") * 2 - 1
    for flip in (0, 1):
        out = nan_full(B * H * W, 4)
        ops.check(ops.lib().mdt_vae_image_to_rows(ops.ptr(x), ops.ptr(out), B, H, W, flip, ops.stream_ptr()),
                  "mdt_vae_image_to_rows")
        ref = to_rows(pad_channels(x.flip(-1) if flip else x, 4))
        assert torch.equal(out, ref), (H, W, flip)
        assert (out[:, 3] == 0).all()


def gn_stats(ops, x, B, P, C):
    sums = nan_full(B, 32, 2, dtype=f64)
    scratch = nan_full(B * ((P + 255) // 256) * 64)
    ops.check(ops.lib().mdt_vae_gn_stats(ops.ptr(x), ops.ptr(sums), ops.ptr(scratch), B, P, C, ops.stream_ptr()),
              "mdt_vae_gn_stats", 2)
    return sums


def gn_input(B, P, C, r, seed):
    """x [B*P, C]: unit-spread noise with group g offset by r * (-1)^g * (1 + g / 32) and image b by a further b."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    g = torch.arange(32, device="cuda").repeat_interleave(C // 32)
    off = r * (1 - 2 * (g % 2)) * (1 + g / 32.0)
    x = torch.randn(B, P, C, generator=gen, device="cuda") + off + torch.arange(B, device="cuda").view(B, 1, 1)
    return x.reshape(B * P, C).contiguous()


def check_gn_stats(sums, x, B, P, C, what):
    """Mean and rstd derived from the kernel's sums vs float64 mean and var(unbiased=False); returns the errors
    (mean error in units of the group's std, relative rstd error)."""
    n = P * (C // 32)
    assert torch.isfinite(sums).all(), f"{what}: non-finite sums"
    m, rstd = gn_mean_rstd(sums, n)
    g = x.double().view(B, P, 32, C // 32).permute(0, 2, 1, 3).reshape(B, 32, n)
    m_ref, var_ref = g.mean(-1), g.var(-1, unbiased=False)
    rstd_ref = (var_ref + EPS).rsqrt()
    e_m = ((m - m_ref).abs() * rstd_ref).max().item()
    e_r = ((rstd - rstd_ref).abs() / rstd_ref).max().item()
    return e_m, e_r


@gpu
@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("P", [1, 60, 255, 256, 257, 4096])
def test_gn_stats(ops, C, P):
    """GroupNorm(32) sums vs float64, per (image, group), at groups whose mean is 0, 10, 100 and 1000 times their spread.

    Bound: mean and rstd within 1e-4 (mean in units of the group's std, rstd relative).  The partials are fp32 sums of
    x - k over at most 256 pixels x C/32 channels (k: one sample of the group), so each term is O(std) and the fp32
    error is ~2^-24 x sqrt(terms) x std ~ 1e-6 of std; the partials are combined in fp64.  Accumulating x itself in
    fp32 would make the sum of squares ~ (mean^2 + var) x n and lose var to cancellation in q/n - m^2: at
    mean / std = 100 about 2^-24 x 1e4 x sqrt(terms) ~ 1e-3 relative, which this bound catches.  Deterministic: two
    calls agree bit for bit."""
    B = 3
    for r in (0, 10, 100, 1000):
        x = gn_input(B, P, C, r, seed=C + P + r)
        sums = gn_stats(ops, x, B, P, C)
        e_m, e_r = check_gn_stats(sums, x, B, P, C, f"C={C} P={P} r={r}")
        print(f"gn_stats C={C} P={P} mean/std={r}: mean err {e_m:.2e} std, rstd rel err {e_r:.2e} (bound 1e-4)")
        assert e_m <= 1e-4 and e_r <= 1e-4, (C, P, r, e_m, e_r)
        assert torch.equal(gn_stats(ops, x, B, P, C), sums), "not deterministic"


@gpu
def test_gn_stats_c384_rejected_or_right(ops):
    """C = 384 passed the old argument check (`C % 128 || C > 512`) although the partial kernel's 8 slots per group are
    then only 6 written: the reduction read uninitialised shared memory.  With real, full-size buffers, the call must
    either be refused (MdtError) or return the float64 statistics.  A C = 512 call first leaves non-zero values in
    shared memory, so unwritten slots show as wrong sums."""
    from maskdit_b200._lib import MdtError
    B, P, C = 2, 1024, 384
    gn_stats(ops, gn_input(B, P, 512, 100, seed=1), B, P, 512)
    x = gn_input(B, P, C, 0, seed=2)
    try:
        sums = gn_stats(ops, x, B, P, C)
    except MdtError:
        return
    e_m, e_r = check_gn_stats(sums, x, B, P, C, "C=384")
    assert e_m <= 1e-4 and e_r <= 1e-4, ("C = 384 returned wrong statistics", e_m, e_r)


def im2col_cases():
    out = []
    for mode, Cs in (("id", (4, 128)), ("gn", (128, 256, 512)), ("gn_silu", (128, 256, 512))):
        for C in Cs:
            out.append((mode, C))
    return out


@gpu
@pytest.mark.parametrize("mode,C", im2col_cases())
def test_im2col(ops, mode, C):
    """im2col with GroupNorm affine (+ swish) and nearest-2x upsample fused, vs float64 F.group_norm -> swish ->
    F.interpolate -> F.unfold in (ky, kx, c) column order.  ks in {1, 3}, up in {1, 2}, output 8x8 and 6x10 (and 7x5,
    1x1 at up = 1), Kp = ks*ks*C rounded up to 8 and that + 8, B = 2.

    Identity: a bf16 cast of the fp32 source, exact.  GN modes: each element within one bf16 ulp of the bf16-rounded
    float64 value, plus the fp32 evaluation before the rounding: mean, v - mean, * rstd, fma with gamma / beta are ~5
    fp32 roundings (rsqrtf 2 ulp), <= 2^-21 x T with T = (|v| + |mean|) rstd |gamma| + |beta|, and swish (slope <= 1.1,
    __expf and a division) adds ~2^-22 |y|: 2^-20 x 1.1 x T in all.  Fed the kernel's own gn_stats sums (instead of
    float64 ones) the statistics add 1e-4 x (1 + |v - mean| rstd) |gamma| (test_gn_stats's bound).  Columns >= ks*ks*C
    are exactly 0.  The printed ratio to the bound is ~1.00 for a one-ulp flip; more than one ulp occurs only where the
    normalised value nearly cancels to 0, so that the fp32 slack spans several of its ulps."""
    torch.manual_seed(21 + C)
    B = 2
    gn = mode != "id"
    worst = worst_ratio = 0.0
    for ks in (1, 3):
        for up in (1, 2):
            for (H, W) in ((8, 8), (6, 10)) + (((7, 5), (1, 1)) if up == 1 else ()):
                Hs, Ws = H // up, W // up
                K = ks * ks * C
                x = (torch.randn(B, C, Hs, Ws, device="cuda") * 2 + torch.randn(C, 1, 1, device="cuda") * 3)
                rows = to_rows(x)
                x64 = x.double()
                if gn:
                    gamma = 1 + 0.5 * torch.randn(C, device="cuda")
                    beta = torch.randn(C, device="cuda")
                    sums64 = gn_sums_ref(rows, B, C)
                    m, rstd = gn_mean_rstd(sums64, Hs * Ws * (C // 32))
                    bc = lambda t: t.repeat_interleave(C // 32, 1).view(B, C, 1, 1)  # noqa: E731
                    y = F.group_norm(x64, 32, gamma.double(), beta.double(), eps=EPS)
                    if mode == "gn_silu":
                        y = swish(y)
                    T = (x64.abs() + bc(m).abs()) * bc(rstd) * gamma.double().abs().view(1, C, 1, 1) \
                        + beta.double().abs().view(1, C, 1, 1)
                    S = (1 + (x64 - bc(m)).abs() * bc(rstd)) * gamma.double().abs().view(1, C, 1, 1)
                    feeds = (("fp64 sums", sums64, 0.0), ("own sums", gn_stats(ops, rows, B, Hs * Ws, C), 1e-4))
                else:
                    y, feeds = x64, (("identity", None, 0.0),)
                for Kp in sorted({(K + 7) // 8 * 8, (K + 7) // 8 * 8 + 8}):
                    ref = im2col_ref(y, ks, up, Kp=Kp)
                    for what, sums, stat_tol in feeds:
                        A = nan_full(B * H * W, Kp, dtype=bf16)
                        ops.check(ops.lib().mdt_vae_im2col(
                            ops.ptr(rows), ops.ptr(sums), ops.ptr(gamma) if gn else 0, ops.ptr(beta) if gn else 0,
                            int(mode == "gn_silu"), ks, up, ops.ptr(A), B, H, W, C, Kp, ops.stream_ptr()),
                            "mdt_vae_im2col")
                        case = (mode, C, ks, up, H, W, Kp, what)
                        assert torch.equal(A[:, K:], torch.zeros_like(A[:, K:])), case
                        if not gn:
                            assert torch.equal(A, ref.to(bf16)), case
                            continue
                        assert not torch.isnan(A).any(), case
                        rr = ref.to(bf16).double()
                        slack = im2col_ref(2.0 ** -20 * 1.1 * T + 1.1 * stat_tol * S, ks, up, Kp=Kp)
                        err = (A.double() - rr).abs()
                        bound = torch.where(rr == 0, slack, bf16_ulp(rr) + slack)
                        over = err > bound
                        worst = max(worst, (err / bf16_ulp(rr)).max().item())
                        worst_ratio = max(worst_ratio, (err / bound.clamp_min(1e-300)).max().item())
                        assert not over.any(), (case, err[over][:4], rr[over][:4], bound[over][:4])
    print(f"im2col {mode} C={C}: worst error {worst:.2f} bf16 ulp, {worst_ratio:.2f} of its bound")


@gpu
@pytest.mark.parametrize("C", [4, 128, 256, 512])
def test_im2col_down(ops, C):
    """The Downsample window: F.pad(x, (0,1,0,1)) then F.unfold(3, stride=2), (ky, kx, c) columns; a bf16 cast of the
    source, exact.  Source 2x2, 8x8, 6x14, 16x10, B = 2; Kp = 9C rounded up to 8 and that + 8, pad columns 0."""
    torch.manual_seed(22)
    B = 2
    for (H, W) in ((2, 2), (8, 8), (6, 14), (16, 10)):
        x = torch.randn(B, C, H, W, device="cuda")
        rows = to_rows(x)
        K = 9 * C
        for Kp in sorted({(K + 7) // 8 * 8, (K + 7) // 8 * 8 + 8}):
            A = nan_full(B * (H // 2) * (W // 2), Kp, dtype=bf16)
            ops.check(ops.lib().mdt_vae_im2col_down(ops.ptr(rows), ops.ptr(A), B, H, W, C, Kp, ops.stream_ptr()),
                      "mdt_vae_im2col_down")
            assert torch.equal(A, im2col_ref(x.double(), down=True, Kp=Kp).to(bf16)), (C, H, W, Kp)


@gpu
@pytest.mark.parametrize("rows,cols,ld", [(60, 60, 64), (64, 64, 64), (4096, 4096, 4096), (7, 1, 8), (33, 31, 40)])
def test_softmax_rows(ops, rows, cols, ld):
    """softmax(scale * S) per row to bf16, vs float64; scale = 512^-0.5, score spreads from 0.1 to 1e3 after scaling
    (so exp would overflow without the max subtraction).  S[:, cols:ld] is NaN: the kernel must not read it, and must
    write P[:, cols:ld] = 0.

    Bound: 1 bf16 ulp of the float64 probability (half an ulp of rounding, plus the fp32 evaluation: s - max is exact
    to 2^-24 x 2e3 / scale, i.e. ~1e-4 relative after scaling, __expf ~2^-21 relative, the sum and 1 / sum ~1e-6), and
    2^-126 absolute: __expf flushes results below the fp32 normal range to zero."""
    torch.manual_seed(23)
    scale = 512 ** -0.5
    spread = torch.logspace(-1, 3, rows, device="cuda").view(rows, 1) / scale
    S = nan_full(rows, ld)
    S[:, :cols] = (torch.rand(rows, cols, device="cuda") * 2 - 1) * spread
    ref = torch.softmax(scale * S[:, :cols].double(), -1)
    fns = [("ld", lambda P: ops.lib().mdt_vae_softmax_rows_ld(ops.ptr(S), scale, ops.ptr(P), rows, cols, ld,
                                                              ops.stream_ptr()))]
    if cols == ld:
        fns.append(("plain", lambda P: ops.lib().mdt_vae_softmax_rows(ops.ptr(S), scale, ops.ptr(P), rows, cols,
                                                                      ops.stream_ptr())))
    for what, fn in fns:
        P = nan_full(rows, ld, dtype=bf16)
        ops.check(fn(P), "mdt_vae_softmax_rows")
        assert torch.equal(P[:, cols:], torch.zeros_like(P[:, cols:])), what
        got = P[:, :cols].double()
        assert torch.isfinite(got).all(), what
        err = (got - ref).abs()
        ulps = (err / bf16_ulp(ref)).max().item()
        print(f"softmax_rows_{what} {rows}x{cols} ld {ld}: worst {ulps:.2f} bf16 ulp")
        assert (err <= bf16_ulp(ref) + 2.0 ** -126).all(), (what, ulps)


@gpu
@pytest.mark.parametrize("C", [4, 8])
@pytest.mark.parametrize("P", [1, 60, 4096])
def test_post_quant_and_quant_out(ops, C, P):
    """The two 1x1 convolutions with their own kernels, vs float64 einsum: post_quant_conv(z / scale_factor) (NCHW ->
    rows) and quant_conv(rows with ldx = C or 16, NaN beyond C) -> NCHW moments.  B = 3.

    Bound: max-abs 1e-6 of the output scale.  Each output is an fp32 fma chain of C <= 8 terms plus the bias (and the
    1 / scale_factor product): <= (C + 2) x 2^-24 ~ 6e-7 of sum |w v| + |b|, which with these weights is about the
    output's own magnitude and below its scale."""
    torch.manual_seed(24)
    B, sf = 3, 0.18215
    W = torch.randn(C, C, device="cuda") * C ** -0.5
    bias = torch.randn(C, device="cuda") * 0.1
    z = torch.randn(B, C, P, device="cuda")
    out = nan_full(B * P, C)
    ops.check(ops.lib().mdt_vae_post_quant(ops.ptr(z), ops.ptr(W), ops.ptr(bias), sf, ops.ptr(out), B, C, P,
                                           ops.stream_ptr()), "mdt_vae_post_quant")
    ref = torch.einsum("oc,bcp->bpo", W.double(), z.double() / sf) + bias.double()
    e = max_rel(out, ref.reshape(B * P, C))
    print(f"post_quant C={C} P={P}: max-abs {e:.2e} of scale (bound 1e-6)")
    assert e <= 1e-6
    for ldx in (C, 16):
        rows = nan_full(B * P, ldx)
        rows[:, :C] = torch.randn(B * P, C, device="cuda")
        mom = nan_full(B, C, P)
        ops.check(ops.lib().mdt_vae_quant_out(ops.ptr(rows), ldx, ops.ptr(W), ops.ptr(bias), ops.ptr(mom), B, C, P,
                                              ops.stream_ptr()), "mdt_vae_quant_out")
        ref = torch.einsum("oc,bpc->bop", W.double(), rows[:, :C].double().view(B, P, C)) + bias.double().view(C, 1)
        e = max_rel(mom, ref)
        print(f"quant_out C={C} P={P} ldx={ldx}: max-abs {e:.2e} of scale (bound 1e-6)")
        assert e <= 1e-6


@gpu
def test_rows_to_nchw(ops):
    """[B*P, ldx] rows (first C columns valid, the rest NaN) -> [B, C, P]; P = 7 x 9 (not a multiple of 4); exact."""
    torch.manual_seed(25)
    B, P, C, ldx = 3, 63, 3, 8
    x = nan_full(B * P, ldx)
    x[:, :C] = torch.randn(B * P, C, device="cuda")
    out = nan_full(B, C, P)
    ops.check(ops.lib().mdt_vae_rows_to_nchw(ops.ptr(x), ops.ptr(out), B, P, C, ldx, ops.stream_ptr()),
              "mdt_vae_rows_to_nchw")
    assert torch.equal(out, x[:, :C].reshape(B, P, C).permute(0, 2, 1))


# ---- GPU: the GEMM at the VAE's shapes -------------------------------------------------------------------------------
def rb(*shape, scale=1.0):
    return (torch.randn(*shape, device="cuda") * scale).to(bf16)


@gpu
def test_gemm_vae_shapes(ops):
    """The tcgen05 GEMM at shapes only the VAE runs, vs fp32 A.float() @ B.float().t() on the same bf16 operands: 1e-3
    of the output scale for fp32 output (fp32 accumulation), 2^-8 for bf16 output (one rounding).  Elements outside
    the written block (ragged ldo columns, rows around an offset view) must stay NaN."""
    torch.manual_seed(26)
    errs = {}

    def chk(got, ref, tol, what):
        e = max_rel(got, ref)
        errs[what] = e
        assert e <= tol, (what, e, tol)

    # decoder conv_out: N = 3 in an 8-column output (the ragged epilogue), bias, fp32; encoder conv_out: N = 8
    for M, N, K in ((3 * 48 * 80, 3, 9 * 128), (3 * 6 * 10, 8, 9 * 512)):
        A, Bw, bias = rb(M, K), rb(N, K, scale=K ** -0.5), torch.randn(N, device="cuda")
        out = nan_full(M, 8)
        ops.gemm(A, Bw, M, N, K, out=out, ldo=8, bias=bias)
        chk(out[:, :N], A.float() @ Bw.float().t() + bias, 1e-3, f"conv_out N={N}")
        assert torch.isnan(out[:, N:]).all(), f"conv_out N={N}: wrote past N"
    # conv_in: K = Kp = 40 (36 taps x channels + 4 zero columns), N = 128 (encoder) and 512 (decoder)
    for N in (128, 512):
        M = 2 * 64 * 64
        A, Bw = rb(M, 40), rb(N, 40, scale=0.2)
        A[:, 36:] = 0
        Bw[:, 36:] = 0
        bias = torch.randn(N, device="cuda")
        out = nan_full(M, N)
        ops.gemm(A, Bw, M, N, 40, out=out, bias=bias)
        chk(out, A.float() @ Bw.float().t() + bias, 1e-3, f"conv_in N={N}")
    # attention at T = 60 (Tp = 64): scores q k^T into a 64-column buffer, then P V with V at a row offset
    T, Tp, c, B = 60, 64, 512, 3
    q, k = rb(B * T, c), rb(B * T, c)
    v = rb(B * T + Tp - T, c)
    S = nan_full(T, Tp)
    ops.gemm(q[T:2 * T], k[T:2 * T], T, T, c, out=S, ldo=Tp)
    chk(S[:, :T], q[T:2 * T].float() @ k[T:2 * T].float().t(), 1e-3, "scores 60x60x512 ldo 64")
    assert torch.isnan(S[:, T:]).all(), "scores: wrote past N"
    Pm = torch.softmax(torch.randn(T, T, device="cuda") * 3, -1)
    Pb = torch.zeros(T, Tp, device="cuda", dtype=bf16)
    Pb[:, :T] = Pm.to(bf16)
    o = nan_full(B * T, c, dtype=bf16)
    ops.gemm(Pb, v[T:T + Tp], T, c, Tp, b_mn=True, out=o[T:2 * T])
    chk(o[T:2 * T], Pb.float() @ v[T:T + Tp].float(), 2 ** -8, "P V b_mn at row offset")
    assert torch.isnan(o[:T].float()).all() and torch.isnan(o[2 * T:].float()).all(), "P V wrote outside its rows"
    # q / k / v: bf16 output with bias (EPI_STORE, out_fp32 = 0)
    M = B * T
    xn, Wq, bq = rb(M, c), rb(c, c, scale=c ** -0.5), torch.randn(c, device="cuda")
    o16 = nan_full(M, c, dtype=bf16)
    ops.gemm(xn, Wq, M, c, c, out=o16, bias=bq)
    chk(o16, xn.float() @ Wq.float().t() + bq, 2 ** -8, "qkv bf16 + bias")
    # proj_out / conv2: bias + resid into a row-offset view of a larger buffer (_conv's chunk loop, image 1 of 3)
    for (N, K, ldo) in ((512, 512, 512), (256, 9 * 256, 256)):
        m = 6 * 10
        A, Bw, bias = rb(m, K), rb(N, K, scale=K ** -0.5), torch.randn(N, device="cuda")
        resid = torch.randn(3 * m, N, device="cuda")
        out = nan_full(3 * m, ldo)
        ops.gemm(A, Bw, m, N, K, out=out[m:], ldo=ldo, bias=bias, resid=resid[m:], ld_resid=N)
        chk(out[m:2 * m], A.float() @ Bw.float().t() + bias + resid[m:2 * m], 1e-3, f"bias+resid N={N} K={K}")
        assert torch.isnan(out[:m]).all() and torch.isnan(out[2 * m:]).all(), "bias+resid wrote outside its rows"
    print("gemm at VAE shapes, max-abs / scale:", {k: f"{v:.2e}" for k, v in errs.items()})


# ---- GPU: the building blocks of _VaeBase vs the float64 oracle ------------------------------------------------------
def stand_in_state_dict(round_convs):
    sd = {**VE.make_vae_encoder_state_dict(5), **VO.make_vae_state_dict(3)}
    if round_convs:   # the weights the GEMM sees, so that only activation rounding and accumulation order differ
        sd = {k: v.to(bf16).float() if v.ndim == 4 and not k.startswith(("quant_conv", "post_quant_conv")) else v
              for k, v in sd.items()}
    return sd


@pytest.fixture(scope="module")
def vae_rounded():
    from maskdit_b200.vae import AutoencoderKL
    sd = stand_in_state_dict(True)
    vae = AutoencoderKL()
    vae.load_state_dict(sd, strict=True)
    vae = vae.cuda().eval()
    vae._ready()
    return vae, {k: v.double().cuda() for k, v in sd.items()}


# (name, cin, H x W of the source relative to the output, _conv keywords, GroupNorm name)
CONV_MODES = {
    "enc_conv_in": ("encoder.conv_in", 3, {}, None),
    "dec_conv_in": ("decoder.conv_in", 4, {}, None),
    "gn_swish_128": ("encoder.down.0.block.0.conv1", 128, {}, "encoder.down.0.block.0.norm1"),
    "gn_swish_256": ("encoder.down.1.block.1.conv1", 256, {}, "encoder.down.1.block.1.norm1"),
    "gn_swish_512": ("decoder.mid.block_1.conv1", 512, {}, "decoder.mid.block_1.norm1"),
    "nin_128_256": ("encoder.down.1.block.0.nin_shortcut", 128, {"ks": 1}, None),
    "nin_512_256": ("decoder.up.1.block.0.nin_shortcut", 512, {"ks": 1}, None),
    "up_512": ("decoder.up.3.upsample.conv", 512, {"up": 2}, None),
    "up_256": ("decoder.up.1.upsample.conv", 256, {"up": 2}, None),
    "down_128": ("encoder.down.0.downsample.conv", 128, {"down": True}, None),
    "down_256": ("encoder.down.1.downsample.conv", 256, {"down": True}, None),
    "down_512": ("encoder.down.2.downsample.conv", 512, {"down": True}, None),
    "dec_conv_out": ("decoder.conv_out", 128, {}, "decoder.norm_out"),
    "enc_conv_out": ("encoder.conv_out", 512, {}, "encoder.norm_out"),
}


def run_conv(ops, vae, x, name, cin, H, W, kw, norm):
    """vae._conv on the NCHW fp32 input x -> NCHW fp32 [B, cout, H, W] (RGB goes through mdt_vae_image_to_rows)."""
    B = x.shape[0]
    if cin == 3:
        rows = nan_full(x.shape[0] * x.shape[2] * x.shape[3], 4)
        ops.check(ops.lib().mdt_vae_image_to_rows(ops.ptr(x), ops.ptr(rows), B, x.shape[2], x.shape[3], 0,
                                                  ops.stream_ptr()), "mdt_vae_image_to_rows")
        cin = 4
    else:
        rows = to_rows(x)
    y = vae._conv(rows, B, H, W, cin, name, norm=norm, silu=norm is not None, **kw)
    cout = vae._packed[f"{name}.weight"][0].shape[0]
    return to_nchw(y[:, :cout], B, H, W)


def conv_ref(sd, x, name, kw, norm, round_operand):
    """The same layer in float64: f(x) (GroupNorm + swish, nearest upsample or the Downsample pad), optionally rounded
    to bf16 (what the GEMM's A operand holds), then F.conv2d with the (bf16-exact) weights."""
    if norm is not None:
        x = swish(VO._gn(sd, norm, x))
    if kw.get("up", 1) == 2:
        x = F.interpolate(x, scale_factor=2.0, mode="nearest")
    if kw.get("down"):
        x = F.pad(x, (0, 1, 0, 1))
    if round_operand:
        x = x.to(bf16).double()
    ks = kw.get("ks", 3)
    return F.conv2d(x, sd[f"{name}.weight"], sd[f"{name}.bias"], stride=2 if kw.get("down") else 1,
                    padding=0 if kw.get("down") else ks // 2)


@gpu
@pytest.mark.parametrize("mode", list(CONV_MODES))
def test_conv_layer_vs_fp64(ops, vae_rounded, mode):
    """`_VaeBase._conv` in every mode the network uses, H x W in {8x8, 6x10}, B = 3, stand-in weights rounded to bf16.

    Bounds: (1) max-abs <= 1e-3 of scale against the float64 convolution of the bf16-rounded float64 operand: what is
    left is fp32 accumulation (~sqrt(K) 2^-24 relative) and a 1-ulp bf16 flip of a few operand elements (one of K
    terms each off by 2^-7 relative): far below 1e-3, while a wrong border row or column is O(1) there.  (2) rel-L2
    <= 3e-3 against the unrounded float64 layer: bf16 keeps 8 significant bits, so rounding an operand errs by up to
    2^-8 relative (at the bottom of a binade; 2^-9 at the top), rms ~ 2^-8 / sqrt(3) x 0.74 ~ 1.7e-3 over a
    log-uniform mantissa, and a sum of K independent terms has the same relative rms error: ~1.7e-3 (a float64
    emulation that rounds only the operand gives 1.4e-3 to 1.7e-3 on these cases).  (3) The layer run with one and
    with two images per im2col operand (`max_rows`) is bit-identical to the unchunked run."""
    vae, sd = vae_rounded
    name, cin, kw, norm = CONV_MODES[mode]
    torch.manual_seed(27)
    B = 3
    for (H, W) in ((8, 8), (6, 10)):
        up = kw.get("up", 1)
        Hs, Ws = (2 * H, 2 * W) if kw.get("down") else (H // up, W // up)
        if cin == 3:
            x = torch.rand(B, 3, Hs, Ws, device="cuda") * 2 - 1
        else:
            x = torch.randn(B, cin, Hs, Ws, device="cuda") + 0.5 * torch.randn(1, cin, 1, 1, device="cuda")
        vae.max_rows = 1 << 21
        got = run_conv(ops, vae, x, name, cin, H, W, kw, norm)
        x64 = x.double()
        e_max = max_rel(got, conv_ref(sd, x64, name, kw, norm, True))
        e_l2 = rel_l2(got, conv_ref(sd, x64, name, kw, norm, False))
        print(f"conv {mode} {H}x{W}: max-abs {e_max:.2e} of scale vs rounded operand (bound 1e-3), "
              f"rel-L2 {e_l2:.2e} vs fp64 (bound 3e-3)")
        assert e_max <= 1e-3 and e_l2 <= 3e-3, (mode, H, W, e_max, e_l2)
        for per in (1, 2):
            vae.max_rows = per * H * W
            assert torch.equal(run_conv(ops, vae, x, name, cin, H, W, kw, norm), got), (mode, H, W, per)
        vae.max_rows = 1 << 21


@gpu
def test_packed_weights_are_the_reference_layout(vae_rounded):
    """`_VaeBase._ready` packs every convolution weight like pack_weight (the layout the CPU test checks)."""
    vae, sd = vae_rounded
    for name, *_ in CONV_MODES.values():
        wq, K, Kp = vae._packed[f"{name}.weight"]
        assert torch.equal(wq, pack_weight(sd[f"{name}.weight"]).to(bf16)), name


@gpu
def test_resblock_cin_ne_cout_vs_fp64(ops, vae_rounded):
    """`_resblock` 128 -> 256 (conv1, conv2 with the residual in the epilogue, the 1x1 nin_shortcut), B = 3 at 6x10
    and 8x8, vs the float64 oracle.  Three bf16-rounded operands, each ~1.7e-3 relative to its convolution's output
    (test_conv_layer_vs_fp64); conv1's error is partly normalised away by norm2, and the sum of the shortcut and
    conv2 adds two independent errors: a float64 emulation that rounds the three operands gives rel-L2 1.9e-3 and
    max-abs 1.9e-3 of scale (a B200 measured 1.85e-3 and 1.94e-3).  Bounds: rel-L2 <= 3e-3, max-abs <= 4e-3 of
    scale."""
    vae, sd = vae_rounded
    name = "encoder.down.1.block.0"
    torch.manual_seed(28)
    for (H, W) in ((6, 10), (8, 8)):
        B = 3
        x = torch.randn(B, 128, H, W, device="cuda") + 0.5 * torch.randn(1, 128, 1, 1, device="cuda")
        got = to_nchw(vae._resblock(to_rows(x), B, H, W, name, 128, 256), B, H, W)
        ref = VO._resblock(sd, name, x.double())
        e_max, e_l2 = max_rel(got, ref), rel_l2(got, ref)
        print(f"resblock 128->256 {H}x{W}: max-abs {e_max:.2e} of scale (bound 4e-3), rel-L2 {e_l2:.2e} (bound 3e-3)")
        assert e_max <= 4e-3 and e_l2 <= 3e-3, (H, W, e_max, e_l2)


@gpu
@pytest.mark.parametrize("B,H,W", [(3, 6, 10), (2, 8, 8), (1, 16, 16)])
def test_attn_vs_fp64(ops, vae_rounded, B, H, W):
    """`_attn` (GroupNorm, q / k / v, softmax(q k^T / sqrt(512)), P V, proj_out + residual) vs the float64 oracle.
    (3, 6x10) pads T = 60 to 64 columns: image b's P V reads 4 V rows of image b + 1 and relies on exact-zero
    probabilities; each image of a batch must be bit-equal to a B = 1 run on that image.

    bf16 operands in series: the normalised input, q / k / v, P and the attention output each add ~1.7e-3 relative
    (test_conv_layer_vs_fp64) to the attention branch; the residual x dominates the output and dilutes it.  A float64
    emulation that rounds exactly these operands gives, over the three cases, rel-L2 3.7e-4 to 4.8e-4, max-abs
    4.2e-4 to 5.4e-4 of scale, and 1.9e-3 to 2.2e-3 rel-L2 on the branch alone (output - x); on a B200 the kernels
    measured rel-L2 3.7e-4 to 4.8e-4, max-abs 3.7e-4 to 8.1e-4 and branch rel-L2 1.8e-3 to 2.3e-3 (fp32 score
    accumulation and __expf on top of the roundings).  Bounds, at most twice the worst measured value: rel-L2 <= 1e-3,
    max-abs <= 1.5e-3 of scale, branch rel-L2 <= 4.5e-3."""
    vae, sd = vae_rounded
    name = "encoder.mid.attn_1"
    torch.manual_seed(29)
    x = torch.randn(B, 512, H, W, device="cuda") * 2 + torch.randn(1, 512, 1, 1, device="cuda")
    T = H * W
    rows = to_rows(x)
    got = vae._attn(rows, B, H, W, name, 512)
    ref = VO._attn(sd, name, x.double())
    g = to_nchw(got, B, H, W)
    e_max, e_l2 = max_rel(g, ref), rel_l2(g, ref)
    # the attention branch alone (output minus the residual), so the residual cannot hide an error in it
    e_br = rel_l2(g - x.double(), ref - x.double())
    print(f"attn B={B} {H}x{W}: max-abs {e_max:.2e} of scale (bound 1.5e-3), rel-L2 {e_l2:.2e} (bound 1e-3), "
          f"branch rel-L2 {e_br:.2e} (bound 4.5e-3)")
    assert e_max <= 1.5e-3 and e_l2 <= 1e-3 and e_br <= 4.5e-3, (e_max, e_l2, e_br)
    for i in range(B):
        one = vae._attn(rows[i * T:(i + 1) * T].contiguous(), 1, H, W, name, 512)
        assert torch.equal(one, got[i * T:(i + 1) * T]), i


# ---- GPU: end to end at the shapes the goldens miss ------------------------------------------------------------------
@pytest.fixture(scope="module")
def vae_full():
    from maskdit_b200.vae import AutoencoderKL
    sd = stand_in_state_dict(False)
    vae = AutoencoderKL()
    vae.load_state_dict(sd, strict=True)
    return vae.cuda().eval(), sd


@gpu
def test_decode_6x10_vs_fp64_oracle(vae_full):
    """Decode of z [3,4,6,10] (T = 60 in the mid attention, 48x80 images) vs vae_oracle.decode in float64: rel-L2 <=
    1e-2 (the bar of the decode golden); image i bit-equal to a B = 1 decode of z[i]."""
    vae, sd = vae_full
    torch.manual_seed(30)
    z = torch.randn(3, 4, 6, 10, device="cuda")
    img = vae.decode(z)
    ref = VO.decode({k: v.double().cuda() for k, v in sd.items()}, z.double())
    e_l2 = rel_l2(img, ref)
    print(f"decode [3,4,6,10]: rel-L2 {e_l2:.2e} vs fp64 oracle (bound 1e-2)")
    assert img.shape == (3, 3, 48, 80) and e_l2 <= 1e-2
    for i in range(3):
        assert torch.equal(vae.decode(z[i:i + 1]), img[i:i + 1]), i


@gpu
def test_encode_decode_past_2_31_elements(vae_full):
    """Encode at 512x512 with B = 8 and decode of 64x64 latents with B = 8: the top-level im2col operand has
    8 x 512 x 512 = 2.1 M rows x 1152 columns, more than 2^31 elements, and decode's level-1 upsample convolution
    2.1 M rows x 2304 columns (9.7 GB of bf16; peak memory about 15 GB, from the shapes).  Image 7 must be bit-equal
    to a B = 1 run: an index that wraps at 2^31 reads or writes another image's rows."""
    vae, _ = vae_full
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    g = torch.Generator(device="cuda").manual_seed(31)
    x = torch.rand(8, 3, 512, 512, generator=g, device="cuda") * 2 - 1
    m = vae.encode_moments(x)
    assert torch.isfinite(m).all()
    assert torch.equal(vae.encode_moments(x[7:].contiguous()), m[7:])
    del x, m
    z = torch.randn(8, 4, 64, 64, generator=g, device="cuda")
    img = vae.decode(z)
    assert img.shape == (8, 3, 512, 512) and torch.isfinite(img).all()
    assert torch.equal(vae.decode(z[7:].contiguous()), img[7:])
    print(f"encode 512^2 x 8 / decode 64^2 x 8: peak memory {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")
