"""Per-kernel parity (GPU): every C-ABI kernel against a plain PyTorch fp32 reference of the same op fed the SAME
bf16-rounded inputs.  Tolerances are stated per test: fp32-accumulate kernels 1e-3 relative to the output scale,
bf16-output kernels 1 bf16 ulp (2^-8) relative; the integer mask path is bit-exact.  The SD-VAE kernels (`mdt_vae_*`)
and the GEMM at the VAE's shapes are in test_vae_kernels_gpu.py."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ops():
    from maskdit_b200 import ops as o
    return o


def dev():
    return torch.device("cuda")


def close(got, ref, tol, what=""):
    got, ref = got.float(), ref.float()
    scale = ref.abs().max().item() + 1e-12
    err = (got - ref).abs().max().item()
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    assert err <= tol * scale, f"{what}: max_abs {err:.4g} > {tol} * scale {scale:.4g}"


def rb(*shape, scale=1.0):
    return (torch.randn(*shape, device=dev()) * scale).to(torch.bfloat16)


# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [(256, 256, 128), (512, 1152, 1152), (384, 3456, 1152), (300, 200, 1000),
                                   (2, 1152, 256), (1024, 16, 512),
                                   # half-width last column tile, paired unit order: odd panel count / several waves
                                   (1200, 1152, 256), (20000, 1152, 128), (9000, 3456, 64)])
def test_gemm_kk(ops, M, N, K):
    torch.manual_seed(0)
    A, B = rb(M, K), rb(N, K)
    out = torch.empty(M, N, device=dev(), dtype=torch.float32)
    ops.gemm(A, B, M, N, K, out=out)
    close(out, A.float() @ B.float().t(), 1e-3, "gemm KK")


@pytest.mark.parametrize("M,N,K", [(256, 256, 128), (512, 1152, 4608), (256, 512, 16), (300, 1000, 1152),
                                   (1200, 1152, 512)])
def test_gemm_dgrad(ops, M, N, K):
    torch.manual_seed(1)
    A, W = rb(M, K), rb(K, N)
    out = torch.empty(M, N, device=dev(), dtype=torch.float32)
    ops.gemm(A, W, M, N, K, b_mn=True, out=out)
    close(out, A.float() @ W.float(), 1e-3, "gemm K-MN")


@pytest.mark.parametrize("M,N,K", [(3456, 1152, 2048), (512, 512, 8192), (1152, 1000, 256), (16, 512, 4096)])
def test_gemm_wgrad_streamk(ops, M, N, K):
    torch.manual_seed(2)
    A, B = rb(K, M), rb(K, N)
    out = torch.zeros(M, N, device=dev(), dtype=torch.float32)
    ops.gemm(A, B, M, N, K, a_mn=True, b_mn=True, out=out, epi=ops.EPI_ATOMIC)
    close(out, A.float().t() @ B.float(), 1e-3, "gemm MN-MN stream-K")


def test_gemm_epilogues(ops):
    torch.manual_seed(3)
    M, N, K, T = 512, 1152, 1152, 128
    A, B = rb(M, K), rb(N, K, scale=0.05)
    bias = torch.randn(N, device=dev())
    acc = A.float() @ B.float().t() + bias
    R = torch.randn(M, N, device=dev())
    out = torch.empty(M, N, device=dev(), dtype=torch.float32)
    ops.gemm(A, B, M, N, K, out=out, bias=bias, resid=R, ld_resid=N)
    close(out, acc + R, 1e-3, "bias+resid")
    ops.gemm(A, B, M, N, K, out=out, bias=bias, act=ops.ACT_SILU)
    close(out, F.silu(acc), 2e-3, "bias+silu")
    o16 = torch.empty(M, N, device=dev(), dtype=torch.bfloat16)
    aux = torch.empty(M, N, device=dev(), dtype=torch.bfloat16)
    ops.gemm(A, B, M, N, K, out=o16, bias=bias, epi=ops.EPI_GELU, aux=aux, ld_aux=N)
    close(aux, acc, 2 ** -8, "gelu pre")
    close(o16, F.gelu(aux.float(), approximate="tanh"), 2 ** -7, "gelu out")
    gate = torch.randn(M // T, N, device=dev())
    ops.gemm(A, B, M, N, K, out=out, bias=bias, epi=ops.EPI_GATE_RESID, aux=aux, ld_aux=N, resid=R, ld_resid=N,
             gate=gate, ld_gate=N, rows_per_group=T)
    close(aux, acc, 2 ** -8, "gate_resid y")
    close(out, R + gate.repeat_interleave(T, 0) * acc, 1e-3, "gate_resid out")
    h = rb(M, N)
    ops.gemm(A, B, M, N, K, out=o16, epi=ops.EPI_DGELU, aux=h, ld_aux=N)
    hf = h.float().requires_grad_(True)
    F.gelu(hf, approximate="tanh").sum().backward()
    close(o16, (A.float() @ B.float().t()) * hf.grad, 2 ** -7, "dgelu")
    # fused bias gradient: colsum[n] += sum_m of the STORED (bf16-rounded) outputs, incl. a ragged N (1000) and odd M
    for (m2, n2) in ((M, N), (300, 1000)):
        A2, B2, h2 = rb(m2, K), rb(n2, K, scale=0.05), rb(m2, n2)
        o2 = torch.empty(m2, n2, device=dev(), dtype=torch.bfloat16)
        cs = torch.full((n2,), 0.5, device=dev())
        ops.gemm(A2, B2, m2, n2, K, out=o2, epi=ops.EPI_DGELU, aux=h2, ld_aux=n2, colsum=cs)
        close(cs - 0.5, o2.float().sum(0), 1e-4, f"dgelu colsum {m2}x{n2}")


# ---------------------------------------------------------------------------------------------------------
def test_mask_indices_bit_exact(ops):
    """Integer path: bit-exact against the golden vectors (which include forced ties) and torch stable argsort."""
    g = np.load(os.path.join(GOLD, "tables.npz"))
    for L, r in ((256, 0.5), (1024, 0.5), (256, 0.75), (16, 0.5)):
        noise = torch.from_numpy(g[f"mask_noise_{L}_{r}"]).cuda()
        md = ops.mask_indices(noise, int(L * (1 - r)))
        for k in ("mask", "ids_keep", "ids_restore"):
            ref = torch.from_numpy(g[f"mask_{k}_{L}_{r}"]).cuda()
            assert torch.equal(md[k], ref), (L, r, k)
    torch.manual_seed(0)
    noise = torch.rand(64, 1024, device=dev())
    noise[:, 100:200] = noise[:, :100]  # many ties
    md = ops.mask_indices(noise, 512)
    sh = torch.argsort(noise, dim=1, stable=True)
    rs = torch.argsort(sh, dim=1, stable=True)
    assert torch.equal(md["ids_restore"], rs) and torch.equal(md["ids_keep"], sh[:, :512])
    assert torch.equal(md["mask"], (rs >= 512).float())
    # properties (SURVEY §8c): mask.sum = L - T ; ids_restore[ids_keep[i]] = i
    assert torch.equal(md["mask"].sum(1), torch.full((64,), 512.0, device=dev()))
    assert torch.equal(torch.gather(md["ids_restore"], 1, md["ids_keep"]),
                       torch.arange(512, device=dev()).expand(64, -1))


@pytest.mark.parametrize("masked", [True, False])
def test_patch_embed_fwd_bwd(ops, masked):
    torch.manual_seed(4)
    B, C, R, p, D = 3, 4, 32, 2, 1152
    G = R // p
    L = G * G
    x = torch.randn(B, C, R, R, device=dev())
    sigma = torch.rand(B, device=dev()) + 0.1
    W = torch.randn(D, C, p, p, device=dev()) * 0.2
    bias = torch.randn(D, device=dev())
    pos = torch.randn(L, D, device=dev())
    ids = torch.stack([torch.randperm(L, device=dev())[:L // 2] for _ in range(B)]) if masked else None
    out = ops.patch_embed(x, sigma, 0.5, W.reshape(D, -1).contiguous(), bias, pos, ids, p, D)
    c_in = 1 / (0.25 + sigma ** 2).sqrt()
    ref = F.conv2d(x * c_in.view(-1, 1, 1, 1), W, bias, stride=p).flatten(2).transpose(1, 2) + pos
    if masked:
        ref = torch.gather(ref, 1, ids.unsqueeze(-1).expand(-1, -1, D))
    close(out, ref, 1e-5, "patch_embed")
    g = torch.randn_like(out)
    gW = torch.zeros(D, C * p * p, device=dev())
    gb = torch.zeros(D, device=dev())
    ops.patch_embed_bwd(x, sigma, 0.5, ids, g, gW, gb, p)
    Wr = W.clone().requires_grad_(True)
    br = bias.clone().requires_grad_(True)
    ref = F.conv2d(x * c_in.view(-1, 1, 1, 1), Wr, br, stride=p).flatten(2).transpose(1, 2)
    if masked:
        ref = torch.gather(ref, 1, ids.unsqueeze(-1).expand(-1, -1, D))
    (ref * g).sum().backward()
    close(gW, Wr.grad.reshape(D, -1), 1e-3, "patch_embed gW")
    close(gb, br.grad, 1e-3, "patch_embed gb")


def test_timestep_freq(ops):
    g = np.load(os.path.join(GOLD, "tables.npz"))
    t = torch.from_numpy(g["tfreq_in"]).cuda()
    sigma = torch.exp(4 * t)
    out = ops.timestep_freq(sigma.contiguous(), 256)
    close(out, torch.from_numpy(g["tfreq"]).cuda(), 2 ** -8, "timestep_freq vs reference golden")


def test_pointwise(ops):
    torch.manual_seed(5)
    a, b = torch.randn(7, 1152, device=dev()), torch.randn(7, 1152, device=dev())
    o, s = ops.silu(a, b, want_sum=True)
    close(s, a + b, 1e-6)
    close(o, F.silu(a + b), 2 ** -8)
    dy = torch.randn_like(a)
    d32, d16 = ops.silu_bwd(dy, a)
    ar = a.clone().requires_grad_(True)
    (F.silu(ar) * dy).sum().backward()
    close(d32, ar.grad, 1e-5)
    close(d16, ar.grad, 2 ** -8)
    x = torch.randn(1000, 333, device=dev())
    close(ops.cast_bf16(x.reshape(-1)[:333 * 996].contiguous()), x.reshape(-1)[:333 * 996].to(torch.bfloat16), 0)
    xb = rb(1000, 1152)
    out = torch.zeros(1152, device=dev())
    ops.colsum(xb, out)
    close(out, xb.float().sum(0), 1e-4, "colsum bf16")
    xf = torch.randn(700, 513, device=dev())
    out = torch.zeros(513, device=dev())
    ops.colsum(xf, out)
    close(out, xf.sum(0), 1e-4, "colsum f32")


@pytest.mark.parametrize("D,T,B", [(1152, 128, 4), (512, 256, 3), (384, 8, 2)])
def test_ln_modulate_fwd_bwd(ops, D, T, B):
    torch.manual_seed(6)
    M = B * T
    x = torch.randn(M, D, device=dev()) * 2 + 0.3
    mod = torch.randn(B, 3 * D, device=dev()) * 0.5
    shift, scale = mod[:, :D], mod[:, D:2 * D]
    out, mean, rstd = ops.ln_modulate(x, shift, scale, 3 * D, T, M, D)
    xr = x.clone().requires_grad_(True)
    mr = mod.clone().requires_grad_(True)
    ln = F.layer_norm(xr, (D,), eps=1e-6).view(B, T, D)
    ref = (ln * (1 + mr[:, None, D:2 * D]) + mr[:, None, :D]).view(M, D)
    close(out, ref, 2 ** -8, "ln_modulate")
    close(mean, x.mean(1), 1e-5, "mean")
    dxmod = rb(M, D)
    (ref * dxmod.float()).sum().backward()
    g = torch.randn(M, D, device=dev())
    g0 = g.clone()
    dmod = torch.zeros(B, 3 * D, device=dev())
    ops.ln_modulate_bwd(dxmod, x, mean, rstd, scale, 3 * D, T, g, True, dmod[:, :D], dmod[:, D:], 3 * D, M, D)
    close(g - g0, xr.grad, 1e-3, "ln bwd dx (accumulate)")
    close(dmod[:, :D], mr.grad[:, :D], 1e-3, "dshift")
    close(dmod[:, D:2 * D], mr.grad[:, D:2 * D], 1e-3, "dscale")
    g2 = torch.full((M, D), float("nan"), device=dev())
    dmod.zero_()
    ops.ln_modulate_bwd(dxmod, x, mean, rstd, scale, 3 * D, T, g2, False, dmod[:, :D], dmod[:, D:], 3 * D, M, D)
    close(g2, xr.grad, 1e-3, "ln bwd dx (init)")


@pytest.mark.parametrize("D,T,B,fused_gate", [(1152, 128, 4, True), (512, 16, 2, True), (1152, 128, 2, False),
                                              (512, 256, 3, True), (1280, 8, 2, True), (384, 20, 2, True)])
def test_ln_modulate_bwd_gate(ops, D, T, B, fused_gate):
    """Fused LN-modulate backward + gate backward == the two separate kernels == autograd."""
    torch.manual_seed(16)
    M = B * T
    x = torch.randn(M, D, device=dev()) * 2 + 0.3
    mod = torch.randn(B, 3 * D, device=dev()) * 0.5
    shift, scale, gate = mod[:, :D], mod[:, D:2 * D], mod[:, 2 * D:]
    _, mean, rstd = ops.ln_modulate(x, shift, scale, 3 * D, T, M, D)
    dxmod, y = rb(M, D), rb(M, D)
    g0 = torch.randn(M, D, device=dev())
    # separate kernels
    g_a, dmod_a, dbias_a = g0.clone(), torch.zeros(B, 3 * D, device=dev()), torch.zeros(D, device=dev())
    ops.ln_modulate_bwd(dxmod, x, mean, rstd, scale, 3 * D, T, g_a, True, dmod_a[:, :D], dmod_a[:, D:], 3 * D, M, D)
    dy_a = ops.gate_bwd(g_a, y, gate, 3 * D, T, dmod_a[:, 2 * D:], 3 * D, dbias_a, M, D)
    # fused
    g_b, dmod_b, dbias_b = g0.clone(), torch.zeros(B, 3 * D, device=dev()), torch.zeros(D, device=dev())
    gn = (y, gate, 3 * D, dmod_b[:, 2 * D:], 3 * D, dbias_b) if fused_gate else None
    dy_b = ops.ln_modulate_bwd_gate(dxmod, x, mean, rstd, scale, 3 * D, T, g_b, True, dmod_b[:, :D], dmod_b[:, D:],
                                    3 * D, M, D, gate_next=gn)
    close(g_b, g_a, 1e-5, "fused g")
    close(dmod_b[:, :2 * D], dmod_a[:, :2 * D], 1e-4, "fused dshift/dscale")
    if fused_gate:
        close(dy_b, dy_a, 2 ** -8, "fused dy")
        close(dmod_b[:, 2 * D:], dmod_a[:, 2 * D:], 1e-4, "fused dgate")
        close(dbias_b, dbias_a, 1e-4, "fused dbias")
    else:
        assert dy_b is None
    # autograd reference of the LN part, non-accumulating variant
    xr = x.clone().requires_grad_(True)
    ln = F.layer_norm(xr, (D,), eps=1e-6).view(B, T, D)
    ((ln * (1 + scale[:, None, :]) + shift[:, None, :]).view(M, D) * dxmod.float()).sum().backward()
    g_c = torch.full((M, D), float("nan"), device=dev())
    dmod_c = torch.zeros(B, 3 * D, device=dev())
    ops.ln_modulate_bwd_gate(dxmod, x, mean, rstd, scale, 3 * D, T, g_c, False, dmod_c[:, :D], dmod_c[:, D:], 3 * D,
                             M, D)
    close(g_c, xr.grad, 1e-3, "fused ln bwd dx (init)")


@pytest.mark.parametrize("D,T,B", [(1152, 128, 4), (512, 16, 2)])
def test_gate_bwd(ops, D, T, B):
    torch.manual_seed(7)
    M = B * T
    g = torch.randn(M, D, device=dev())
    y = rb(M, D)
    gate = torch.randn(B, 2 * D, device=dev())[:, D:]
    dgate = torch.zeros(B, D, device=dev())
    dbias = torch.zeros(D, device=dev())
    dy = ops.gate_bwd(g, y, gate, 2 * D, T, dgate, D, dbias, M, D)
    ref_dy = g.view(B, T, D) * gate[:, None, :]
    close(dy, ref_dy.reshape(M, D), 2 ** -8, "dy")
    close(dgate, (g.view(B, T, D) * y.float().view(B, T, D)).sum(1), 1e-4, "dgate")
    close(dbias, ref_dy.sum((0, 1)), 1e-4, "dbias")


def attn_ref(qkv, B, T, H, dh):
    q, k, v = qkv.float().view(B, T, 3, H, dh).permute(2, 0, 3, 1, 4).unbind(0)
    att = torch.softmax(q @ k.transpose(-1, -2) * dh ** -0.5, -1)
    return (att @ v).transpose(1, 2).reshape(B * T, H * dh)


@pytest.mark.parametrize("B,T,H,dh", [(2, 128, 16, 72), (2, 256, 16, 32), (3, 8, 6, 64), (1, 200, 4, 72),
                                      (1, 512, 16, 72), (1, 1024, 2, 32), (2, 256, 16, 72), (3, 128, 6, 64),
                                      (5, 128, 16, 32), (2, 512, 4, 32), (1, 512, 6, 64), (1, 1024, 3, 64),
                                      (1, 1024, 2, 72), (3, 256, 5, 64)])
def test_attention_fwd_bwd(ops, B, T, H, dh):
    torch.manual_seed(8)
    qkv = rb(B * T, 3 * H * dh)
    out, lse = ops.attention_fwd(qkv, B, T, H, dh)
    impl_fwd = ops.lib().mdt_attention_last_impl(0)
    qr = qkv.float().requires_grad_(True)
    ref = attn_ref(qr, B, T, H, dh)
    close(out, ref, 2 ** -7, "attention fwd")
    q, k = qkv.float().view(B, T, 3, H, dh)[:, :, 0].transpose(1, 2), qkv.float().view(B, T, 3, H, dh)[:, :, 1].transpose(1, 2)
    close(lse[0], torch.logsumexp(q @ k.transpose(-1, -2) * dh ** -0.5, -1), 1e-3, "lse")
    dout = rb(B * T, H * dh)
    (ref * dout.float()).sum().backward()
    dqkv = ops.attention_bwd(qkv, out, dout, lse, B, T, H, dh)
    impl_bwd = ops.lib().mdt_attention_last_impl(1)
    close(dqkv, qr.grad, 2 ** -7, "attention bwd")
    # which kernel family ran (include/maskdit_b200.h: 0 mma.sync, 1 split-tile TMA, 2 no-swizzle, 3 blocked split-tile,
    # 4 blocked no-swizzle): a tcgen05 kernel for every T that is a multiple of 128, and for the shapes of the
    # BASELINE configs exactly the production kernel - a silently broken tcgen05 path cannot hide behind the fallback.
    print("attention impl", (B, T, H, dh), impl_fwd, impl_bwd)
    if T % 128 == 0:
        # forward at T = 1024 with head_dim > 32: K and V of the whole sequence do not fit one SM's shared memory in
        # the two-pass kernels (no shipped config has that shape); everything else must be a tcgen05 kernel
        assert impl_bwd > 0 and (impl_fwd > 0 or (T == 1024 and dh > 32)), (impl_fwd, impl_bwd)
    else:
        assert (impl_fwd, impl_bwd) == (0, 0)
    production = {(128, 72): (1, 1), (256, 32): (1, 1), (256, 72): (1, 3), (512, 72): (3, 3), (1024, 32): (3, 3),
                  (128, 64): (1, 1), (128, 32): (2, 2)}
    if (T, dh) in production:
        assert (impl_fwd, impl_bwd) == production[(T, dh)], ((T, dh), impl_fwd, impl_bwd)


def test_unmask_fwd_bwd(ops):
    torch.manual_seed(9)
    B, L, T, D = 3, 256, 128, 512
    u = torch.randn(B, T, D, device=dev())
    tok = torch.randn(D, device=dev())
    pos = torch.randn(L, D, device=dev())
    noise = torch.rand(B, L, device=dev())
    md = ops.mask_indices(noise, T)
    out = ops.unmask_tokens(u, tok, pos, md["ids_restore"], B, T, L, D)
    # reference formulation: concat + gather (models/maskdit.py:157-163)
    x_ = torch.cat([u, tok.expand(B, L - T, D)], 1)
    ref = torch.gather(x_, 1, md["ids_restore"].unsqueeze(-1).expand(-1, -1, D)) + pos
    assert torch.equal(out, ref)
    g = torch.randn(B, L, D, device=dev())
    dtok = torch.zeros(D, device=dev())
    du = ops.unmask_tokens_bwd(g, md["ids_restore"], dtok, B, T, L, D)
    close(du.view(B, T, D), torch.gather(g, 1, md["ids_keep"].unsqueeze(-1).expand(-1, -1, D)), 2 ** -8, "du")
    close(dtok, (g * md["mask"].unsqueeze(-1)).sum((0, 1)), 1e-4, "dmask_token")
    out2 = ops.unmask_tokens(u.new_zeros(B, L, D) + 1, None, pos, None, B, L, L, D)
    assert torch.equal(out2, pos.expand(B, L, D) + 1)


@pytest.mark.parametrize("masked", [True, False])
def test_edm_loss_and_grad(ops, masked):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(__file__)))
    from oracle import maskdit_oracle as O
    torch.manual_seed(10)
    B, C, R, p = 4, 4, 32, 2
    L = (R // p) ** 2
    Fo = torch.randn(B, L, p * p * C, device=dev())
    xin, y = torch.randn(B, C, R, R, device=dev()), torch.randn(B, C, R, R, device=dev()) * 0.5
    sigma = torch.tensor([0.05, 0.4, 1.3, 7.0], device=dev())
    gl = torch.rand(B, device=dev())
    mask = ops.mask_indices(torch.rand(B, L, device=dev()), L // 2)["mask"] if masked else None
    loss, Dx, dF = ops.edm_loss(Fo, xin, y, sigma, mask, gl, 0.5, 0.1, p, want_D=True)
    Fr = Fo.clone().requires_grad_(True)
    s4 = sigma.view(-1, 1, 1, 1)
    D = 0.25 / (s4 ** 2 + 0.25) * xin + s4 * 0.5 / (s4 ** 2 + 0.25).sqrt() * O.unpatchify(Fr, p, C)
    w = (s4 ** 2 + 0.25) / (s4 * 0.5) ** 2
    l = w * (D - y) ** 2
    if masked:
        pp = F.avg_pool2d(l.mean(1), p).flatten(1)
        ref = (pp * (1 - mask)).sum(1) / (1 - mask).sum(1)
        tgt = O.patchify(xin, p, C)
        tgt = (tgt - tgt.mean(-1, keepdim=True)) / (tgt.var(-1, keepdim=True) + 1e-6) ** 0.5
        mae = ((O.patchify(D, p, C) - tgt) ** 2).mean(-1)
        ref = ref + 0.1 * (mae * mask).sum(1) / mask.sum(1)
    else:
        ref = l.mean((1, 2, 3))
    close(loss, ref, 1e-4, "loss")
    close(Dx, D, 1e-5, "D")
    (ref * gl).sum().backward()
    close(dF, Fr.grad, 2 ** -7, "dF")
    close(ops.edm_precond_out(Fo, xin, sigma, 0.5, p), D, 1e-5, "precond_out")
    gD = torch.randn_like(xin)
    Fr.grad = None
    D2 = 0.25 / (s4 ** 2 + 0.25) * xin + s4 * 0.5 / (s4 ** 2 + 0.25).sqrt() * O.unpatchify(Fr, p, C)
    (D2 * gD).sum().backward()
    close(ops.edm_precond_out_bwd(gD, sigma, 0.5, p).view_as(Fo), Fr.grad, 2 ** -8, "precond_out_bwd")
    F2 = torch.randn(2 * B, L, p * p * C, device=dev())
    refc = F2[B:] + 1.5 * (F2[:B] - F2[B:])
    refD = 0.25 / (s4 ** 2 + 0.25) * xin + s4 * 0.5 / (s4 ** 2 + 0.25).sqrt() * O.unpatchify(refc, p, C)
    close(ops.cfg_precond_out(F2, xin, sigma, 0.5, 1.5, p), refD, 1e-5, "cfg_precond_out")


def test_heun_and_adamw(ops):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(__file__)))
    from oracle import maskdit_oracle as O
    torch.manual_seed(11)
    n = 4096
    x_hat = torch.randn(n, device=dev(), dtype=torch.float64) * 80
    den = torch.randn(n, device=dev())
    d_cur = torch.empty_like(x_hat)
    x_next = torch.empty_like(x_hat)
    xf = torch.empty(n, device=dev())
    ops.heun_update(0, x_hat, den, d_cur, x_next, xf, 80.0, 57.586)
    dref = (x_hat - den.double()) / 80.0
    assert torch.allclose(d_cur, dref, rtol=1e-14, atol=0)
    xe = x_hat + (57.586 - 80.0) * dref
    assert torch.allclose(x_next, xe, rtol=1e-14, atol=1e-14)
    ops.heun_update(1, x_hat, den, d_cur, x_next, xf, 80.0, 57.586)
    dp = (xe - den.double()) / 57.586
    assert torch.allclose(x_next, x_hat + (57.586 - 80.0) * (0.5 * dref + 0.5 * dp), rtol=1e-13, atol=1e-13)
    # AdamW + EMA vs the oracle restatement of apex FusedAdam(adam_w_mode) + update_ema
    n = 10000
    w = torch.randn(n, device=dev())
    g = torch.randn(n, device=dev()) * 0.01
    m, v = torch.zeros(n, device=dev()), torch.zeros(n, device=dev())
    ema = w.clone()
    w16 = torch.empty(n, device=dev(), dtype=torch.bfloat16)
    wr, mr, vr, er = w.cpu().clone(), m.cpu().clone(), v.cpu().clone(), ema.cpu().clone()
    for step in (1, 2, 3):
        ops.adamw_ema(w, g, m, v, ema, w16, n, 1e-4, step, grad_scale=0.5)
        O.adamw_ema_step(wr, g.cpu() * 0.5, mr, vr, er, step)
    close(w.cpu(), wr, 1e-6, "adamw w")
    close(ema.cpu(), er, 1e-6, "ema")
    close(v.cpu(), vr, 1e-4, "adamw v")
    assert torch.equal(w16, w.to(torch.bfloat16))
    # the bf16-gradient variant (mdt_adamw_ema_g16, after a bf16 all-reduce) on a grid capped at 3 blocks: 3 x 256
    # threads x 4 elements per pass, so the grid-stride loop wraps 4 times over n = 10000
    w = torch.randn(n, device=dev())
    g16 = (torch.randn(n, device=dev()) * 0.01).to(torch.bfloat16)
    m, v = torch.zeros(n, device=dev()), torch.zeros(n, device=dev())
    ema = w.clone()
    wr, mr, vr, er = w.cpu().clone(), m.cpu().clone(), v.cpu().clone(), ema.cpu().clone()
    for step in (1, 2, 3):
        ops.adamw_ema(w, g16, m, v, ema, w16, n, 1e-4, step, grad_scale=0.5, max_blocks=3)
        O.adamw_ema_step(wr, g16.float().cpu() * 0.5, mr, vr, er, step)
    close(w.cpu(), wr, 1e-6, "adamw g16 w")
    close(ema.cpu(), er, 1e-6, "g16 ema")
    close(v.cpu(), vr, 1e-4, "adamw g16 v")
    assert torch.equal(w16, w.to(torch.bfloat16))


def test_sampler_tail_uint8_and_lincomb(ops):
    """sample.py:287: images.add_(1).mul(127.5).clamp_(0, 255).to(uint8).permute(0, 2, 3, 1) — bit-exact; and the fp64
    linear-combination kernel of the ablation sampler."""
    torch.manual_seed(12)
    img = (torch.randn(3, 3, 16, 8, device=dev()) * 0.8)
    img[0, 0, 0, :4] = torch.tensor([-1.0, 1.0, -3.0, 3.0], device=dev())
    got = ops.to_uint8_nhwc(img.contiguous())
    ref = img.clone().add_(1).mul(127.5).clamp_(0, 255).to(torch.uint8).permute(0, 2, 3, 1)
    assert torch.equal(got, ref)
    x, y = torch.randn(1000, device=dev(), dtype=torch.float64), torch.randn(1000, device=dev(), dtype=torch.float64)
    z = torch.randn(1000, device=dev())
    out, o32 = torch.empty_like(x), torch.empty(1000, device=dev())
    ops.lincomb_f64(0.3, x, -1.7, y, 2.5, z, out=out, out_f32=o32, f32_scale=0.5)
    want = 0.3 * x - 1.7 * y + 2.5 * z.double()
    assert torch.allclose(out, want, rtol=1e-14, atol=1e-14) and torch.allclose(o32, (want * 0.5).float(), rtol=1e-6)
    ops.lincomb_f64(2.0, x, out=x)                                   # in place, x only
    assert torch.allclose(x, want * 0 + x)                           # finite, no aliasing fault


def test_attention_strict_mode_refuses_the_mma_sync_fallback():
    """MDT_ATTN_STRICT=1: a shape no tcgen05 kernel accepts (T = 200) is an error instead of a silent mma.sync run; the
    production shapes are unaffected.  (The switch is read once per process: checked in a child process.)"""
    import subprocess
    import sys
    code = (
        "import torch, sys; sys.path.insert(0, %r)\n"
        "from maskdit_b200 import ops\n"
        "from maskdit_b200._lib import MdtError\n"
        "q = torch.randn(2 * 128, 3 * 16 * 72, device='cuda').to(torch.bfloat16)\n"
        "ops.attention_fwd(q, 2, 128, 16, 72)\n"
        "assert ops.lib().mdt_attention_last_impl(0) == 1\n"
        "q = torch.randn(200, 3 * 4 * 72, device='cuda').to(torch.bfloat16)\n"
        "try:\n"
        "    ops.attention_fwd(q, 1, 200, 4, 72)\n"
        "    print('NO_ERROR')\n"
        "except MdtError as e:\n"
        "    print('STRICT_OK', e)\n" % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, MDT_ATTN_STRICT="1"), capture_output=True,
                       text=True, timeout=300)
    assert "STRICT_OK" in r.stdout and "unsupported" in r.stdout, r.stdout + r.stderr
