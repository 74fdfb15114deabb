"""SD-VAE on the B200 kernels.  Decode is the sampler tail of the reference (sample.py:275 `images = vae.decode(z)`,
autoencoder.py:306-453), so that `generate.py` ends in images as `generate_with_net` does; encode is the latent
extraction in front of training (extract_latent.py:77 `encode_moments`, autoencoder.py:212-303,431-434), driven by
`extract_latent.py` at the repository root.

`AutoencoderKL` holds both halves under FrozenAutoencoderKL's keys (a published `autoencoder_kl.pth` loads with
`strict=True`) and provides `encode_moments(x) -> [B, 8, H/8, W/8]` and `decode(z)`.

`AutoencoderKLDecoder` holds `post_quant_conv.*` and `decoder.*` under the reference's state-dict keys (an
`autoencoder_kl.pth` written for `FrozenAutoencoderKL` loads with `strict=False`: the encoder half is ignored) and
`decode(z)` returns the `[B, 3, 8h, 8w]` image the reference's `decode` returns.  Every convolution is the tcgen05 GEMM on
an im2col operand with GroupNorm + swish + nearest upsample (or the stride-2 Downsample window) fused into its
construction (csrc/vae.cu); activations are pixel-major fp32 row matrices.  No PyTorch arithmetic on the path (torch
only lays out the weights once).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .ops import bf16, f32

CH, CH_MULT, NUM_RES_BLOCKS, Z_CH, OUT_CH = 128, (1, 2, 4, 4), 2, 4, 3   # autoencoder.py:466-479 (get_model)
IN_CH = 3


class _Node(nn.Module):
    """Container whose children are created on demand, so parameters can live under the reference's dotted names."""

    def child(self, name):
        if name not in self._modules:
            self.add_module(name, _Node())
        return self._modules[name]


def _resblock_shapes(p, cin, cout):
    """(key, shape) of one ResnetBlock (autoencoder.py:78-115; temb_channels = 0, no conv_shortcut)."""
    out = [(f"{p}.norm1.weight", (cin,)), (f"{p}.norm1.bias", (cin,)), (f"{p}.conv1.weight", (cout, cin, 3, 3)),
           (f"{p}.conv1.bias", (cout,)), (f"{p}.norm2.weight", (cout,)), (f"{p}.norm2.bias", (cout,)),
           (f"{p}.conv2.weight", (cout, cout, 3, 3)), (f"{p}.conv2.bias", (cout,))]
    if cin != cout:
        out.extend([(f"{p}.nin_shortcut.weight", (cout, cin, 1, 1)), (f"{p}.nin_shortcut.bias", (cout,))])
    return out


def _shapes():
    """(key, shape) of post_quant_conv + decoder in the reference's registration order (autoencoder.py:307-377, :424)."""
    out = []

    def res(p, cin, cout):
        out.extend(_resblock_shapes(p, cin, cout))

    out.extend([("post_quant_conv.weight", (Z_CH, 4, 1, 1)), ("post_quant_conv.bias", (Z_CH,))])
    c = CH * CH_MULT[-1]
    out.extend([("decoder.conv_in.weight", (c, Z_CH, 3, 3)), ("decoder.conv_in.bias", (c,))])
    res("decoder.mid.block_1", c, c)
    p = "decoder.mid.attn_1"
    out.extend([(f"{p}.norm.weight", (c,)), (f"{p}.norm.bias", (c,))])
    for n in ("q", "k", "v", "proj_out"):
        out.extend([(f"{p}.{n}.weight", (c, c, 1, 1)), (f"{p}.{n}.bias", (c,))])
    res("decoder.mid.block_2", c, c)
    plan, cur = {}, c
    for lvl in reversed(range(len(CH_MULT))):
        for i in range(NUM_RES_BLOCKS + 1):
            plan[(lvl, i)] = (cur, CH * CH_MULT[lvl])
            cur = CH * CH_MULT[lvl]
        plan[(lvl, "up")] = cur
    for lvl in range(len(CH_MULT)):
        for i in range(NUM_RES_BLOCKS + 1):
            res(f"decoder.up.{lvl}.block.{i}", *plan[(lvl, i)])
        if lvl != 0:
            cu = plan[(lvl, "up")]
            out.extend([(f"decoder.up.{lvl}.upsample.conv.weight", (cu, cu, 3, 3)),
                        (f"decoder.up.{lvl}.upsample.conv.bias", (cu,))])
    out.extend([("decoder.norm_out.weight", (CH,)), ("decoder.norm_out.bias", (CH,)),
                ("decoder.conv_out.weight", (OUT_CH, CH, 3, 3)), ("decoder.conv_out.bias", (OUT_CH,))])
    return out, plan


def _encoder_shapes():
    """(key, shape) of the encoder in the reference's registration order (Encoder.__init__, autoencoder.py:212-278)."""
    out = []

    def res(p, cin, cout):
        out.extend(_resblock_shapes(p, cin, cout))

    out.extend([("encoder.conv_in.weight", (CH, IN_CH, 3, 3)), ("encoder.conv_in.bias", (CH,))])
    plan, cin = {}, CH
    for lvl in range(len(CH_MULT)):
        for i in range(NUM_RES_BLOCKS):
            plan[(lvl, i)] = (cin, CH * CH_MULT[lvl])
            res(f"encoder.down.{lvl}.block.{i}", *plan[(lvl, i)])
            cin = CH * CH_MULT[lvl]
        if lvl != len(CH_MULT) - 1:
            out.extend([(f"encoder.down.{lvl}.downsample.conv.weight", (cin, cin, 3, 3)),
                        (f"encoder.down.{lvl}.downsample.conv.bias", (cin,))])
    res("encoder.mid.block_1", cin, cin)
    p = "encoder.mid.attn_1"
    out.extend([(f"{p}.norm.weight", (cin,)), (f"{p}.norm.bias", (cin,))])
    for n in ("q", "k", "v", "proj_out"):
        out.extend([(f"{p}.{n}.weight", (cin, cin, 1, 1)), (f"{p}.{n}.bias", (cin,))])
    res("encoder.mid.block_2", cin, cin)
    out.extend([("encoder.norm_out.weight", (cin,)), ("encoder.norm_out.bias", (cin,)),
                ("encoder.conv_out.weight", (2 * Z_CH, cin, 3, 3)), ("encoder.conv_out.bias", (2 * Z_CH,))])
    return out, plan


class _VaeBase(nn.Module):
    """Parameters under the reference's dotted names plus the building blocks both halves of the autoencoder run:
    convolution as im2col + tcgen05 GEMM, deterministic GroupNorm statistics, ResnetBlock, single-head AttnBlock."""

    def __init__(self, shapes, scale_factor, max_rows):
        super().__init__()
        self.scale_factor = scale_factor
        self.max_rows = max_rows          # im2col operands are built for at most this many output pixels at a time
        self._keys = [k for k, _ in shapes]
        for k, shp in shapes:
            node, parts = self, k.split(".")
            for part in parts[:-1]:
                node = node.child(part) if isinstance(node, _Node) else self._root_child(part)
            node.register_parameter(parts[-1], nn.Parameter(torch.zeros(shp), requires_grad=False))
        self._packed, self._versions = {}, None

    def _root_child(self, name):
        if name not in self._modules:
            self.add_module(name, _Node())
        return self._modules[name]

    # -- weights ---------------------------------------------------------------------------------------------------
    def _p(self, key):
        node = self
        for part in key.split("."):
            node = node._modules[part] if part in node._modules else node._parameters[part]
        return node

    def _ready(self):
        """(Re)build the GEMM-layout bf16 weights when a parameter changed: conv weight [Co,Ci,kh,kw] -> [Co, (kh,kw,Ci)]
        padded to a multiple of 8 columns (Ci padded to a multiple of 4 with zero channels: the encoder's RGB conv_in).
        The 1x1 quant_conv / post_quant_conv stay fp32 [Co, Ci]: their own kernels apply them."""
        ver = (sum(self._p(k)._version for k in self._keys), self._p(self._keys[0]).data_ptr())
        if self._versions == ver:
            return
        self._packed = {}
        for k in self._keys:
            w = self._p(k)
            if not w.is_cuda:
                raise ops.L.MdtError("maskdit_b200 runs on CUDA (sm_100a) only — there is no CPU fallback")
            if k.endswith(".weight") and w.ndim == 4 and not k.startswith(("post_quant_conv", "quant_conv")):
                co, ci, kh, kw = w.shape
                cp = (ci + 3) // 4 * 4
                K = kh * kw * cp
                Kp = (K + 7) // 8 * 8
                flat = torch.zeros(co, Kp, dtype=f32, device=w.device)
                wt = w.detach().permute(0, 2, 3, 1)
                if cp != ci:
                    wt = torch.cat([wt, wt.new_zeros(co, kh, kw, cp - ci)], dim=3)
                flat[:, :K] = wt.reshape(co, K)
                self._packed[k] = (ops.cast_bf16(flat.contiguous()), K, Kp)
            else:
                self._packed[k] = w.detach().float().contiguous()
        self._versions = ver

    # -- building blocks -------------------------------------------------------------------------------------------
    def _conv(self, x, B, H, W, cin, name, norm=None, silu=False, up=1, resid=None, ks=3, down=False):
        """x [B*(H/up)*(W/up), cin] f32 -> [B*H*W, cout] f32 = conv_ks(f(upsample(x))) + bias (+ resid).
        down: x [B*2H*2W, cin] -> the stride-2 3x3 convolution of F.pad(x, (0,1,0,1)) (Downsample, no norm)."""
        wq, K, Kp = self._packed[f"{name}.weight"]
        bias = self._packed[f"{name}.bias"]
        cout = wq.shape[0]
        ldo = (cout + 7) // 8 * 8
        M = B * H * W
        out = torch.empty(M, ldo, dtype=f32, device=x.device)
        sums = gamma = beta = None
        if norm is not None:
            sums = self._gn_stats(x, B, (H // up) * (W // up), cin)
            gamma, beta = self._packed[f"{norm}.weight"], self._packed[f"{norm}.bias"]
        per = max(1, min(B, self.max_rows // (H * W)))        # images per im2col operand
        A = torch.empty(per * H * W, Kp, dtype=bf16, device=x.device)
        src_rows = 4 * H * W if down else (H // up) * (W // up)
        for b0 in range(0, B, per):
            nb = min(per, B - b0)
            if down:
                ops.check(ops.lib().mdt_vae_im2col_down(ops.ptr(x) + 4 * b0 * src_rows * cin, ops.ptr(A), nb, 2 * H,
                                                        2 * W, cin, Kp, ops.stream_ptr()), "mdt_vae_im2col_down")
            else:
                ops.check(ops.lib().mdt_vae_im2col(ops.ptr(x) + 4 * b0 * src_rows * cin,
                                                   (ops.ptr(sums) + 8 * b0 * 64) if sums is not None else 0,
                                                   ops.ptr(gamma), ops.ptr(beta), int(silu), ks, up, ops.ptr(A), nb, H,
                                                   W, cin, Kp, ops.stream_ptr()), "mdt_vae_im2col")
            m = nb * H * W
            ops.gemm(A, wq, m, cout, Kp, out=out[b0 * H * W:], ldo=ldo, bias=bias,
                     resid=resid[b0 * H * W:] if resid is not None else None, ld_resid=cout)
        return out   # (ldo > cout only for conv_out: the caller reads the first cout columns)

    def _gn_stats(self, x, B, P, C):
        """GroupNorm(32) sums [B,32,2] f64 of x [B*P, C] (deterministic two-pass reduction: the VAE is run-to-run stable)."""
        sums = torch.empty(B, 32, 2, dtype=torch.float64, device=x.device)
        scratch = torch.empty(B * ((P + 255) // 256) * 64, dtype=f32, device=x.device)
        ops.check(ops.lib().mdt_vae_gn_stats(ops.ptr(x), ops.ptr(sums), ops.ptr(scratch), B, P, C, ops.stream_ptr()),
                  "mdt_vae_gn_stats", 2)
        return sums

    def _resblock(self, x, B, H, W, name, cin, cout):
        """ResnetBlock.forward with temb = None (autoencoder.py:117-137)."""
        h = self._conv(x, B, H, W, cin, f"{name}.conv1", norm=f"{name}.norm1", silu=True)
        sc = x
        if cin != cout:   # nin_shortcut: 1x1 convolution of the block input
            sc = self._conv(x, B, H, W, cin, f"{name}.nin_shortcut", ks=1)
        return self._conv(h, B, H, W, cout, f"{name}.conv2", norm=f"{name}.norm2", silu=True, resid=sc)

    def _attn(self, x, B, H, W, name, c):
        """AttnBlock.forward (autoencoder.py:174-198): one head over the H*W positions, head_dim = c.  The score rows are
        padded to Tp = T rounded up to 8 columns (zero probabilities), so any T meets the GEMM's 16-byte row strides."""
        T, M = H * W, B * H * W
        Tp = (T + 7) // 8 * 8
        dev = x.device
        q, k = (torch.empty(M, c, dtype=bf16, device=dev) for _ in range(2))
        v = torch.empty(M + Tp - T, c, dtype=bf16, device=dev)
        if Tp != T:
            v[M:].zero_()   # the last image's P @ V reads Tp - T rows past its own (times zero probabilities)
        sums = self._gn_stats(x, B, T, c)
        xn = torch.empty(M, c, dtype=bf16, device=dev)
        ops.check(ops.lib().mdt_vae_im2col(ops.ptr(x), ops.ptr(sums), ops.ptr(self._packed[f"{name}.norm.weight"]),
                                           ops.ptr(self._packed[f"{name}.norm.bias"]), 0, 1, 1, ops.ptr(xn), B, H, W, c,
                                           c, ops.stream_ptr()), "mdt_vae_im2col")
        for t, n in ((q, "q"), (k, "k"), (v, "v")):
            ops.gemm(xn, self._packed[f"{name}.{n}.weight"][0], M, c, c, out=t, bias=self._packed[f"{name}.{n}.bias"])
        S = torch.empty(T, Tp, dtype=f32, device=dev)
        P = torch.empty(T, Tp, dtype=bf16, device=dev)
        o = torch.empty(M, c, dtype=bf16, device=dev)
        for b in range(B):
            qb, kb, vb = q[b * T:(b + 1) * T], k[b * T:(b + 1) * T], v[b * T:b * T + Tp]
            ops.gemm(qb, kb, T, T, c, out=S, ldo=Tp)                                  # w_ = q k^T
            ops.check(ops.lib().mdt_vae_softmax_rows_ld(ops.ptr(S), float(c) ** -0.5, ops.ptr(P), T, T, Tp,
                                                        ops.stream_ptr()), "mdt_vae_softmax_rows_ld")
            ops.gemm(P, vb, T, c, Tp, b_mn=True, out=o[b * T:(b + 1) * T])            # h_ = softmax(w_) v
        out = torch.empty(M, c, dtype=f32, device=dev)
        ops.gemm(o, self._packed[f"{name}.proj_out.weight"][0], M, c, c, out=out,
                 bias=self._packed[f"{name}.proj_out.bias"], resid=x, ld_resid=c)
        return out

    # -- the two halves ----------------------------------------------------------------------------------------------
    def _decode(self, z):
        """FrozenAutoencoderKL.decode (autoencoder.py:449-453): z [B,4,h,w] -> images [B,3,8h,8w] f32."""
        self._ready()
        z = z.contiguous().float()
        ops._c(z, f32)
        B, C, H, W = z.shape
        x = torch.empty(B * H * W, C, dtype=f32, device=z.device)
        ops.check(ops.lib().mdt_vae_post_quant(ops.ptr(z), ops.ptr(self._packed["post_quant_conv.weight"]),
                                               ops.ptr(self._packed["post_quant_conv.bias"]), self.scale_factor,
                                               ops.ptr(x), B, C, H * W, ops.stream_ptr()), "mdt_vae_post_quant")
        c = CH * CH_MULT[-1]
        h = self._conv(x, B, H, W, C, "decoder.conv_in")
        h = self._resblock(h, B, H, W, "decoder.mid.block_1", c, c)
        h = self._attn(h, B, H, W, "decoder.mid.attn_1", c)
        h = self._resblock(h, B, H, W, "decoder.mid.block_2", c, c)
        for lvl in reversed(range(len(CH_MULT))):
            for i in range(NUM_RES_BLOCKS + 1):
                cin, cout = self._plan[(lvl, i)]
                h = self._resblock(h, B, H, W, f"decoder.up.{lvl}.block.{i}", cin, cout)
            if lvl != 0:
                H, W = 2 * H, 2 * W
                cu = self._plan[(lvl, "up")]
                h = self._conv(h, B, H, W, cu, f"decoder.up.{lvl}.upsample.conv", up=2)
        y = self._conv(h, B, H, W, CH, "decoder.conv_out", norm="decoder.norm_out", silu=True)   # [M, 8], 3 valid
        img = torch.empty(B, OUT_CH, H, W, dtype=f32, device=z.device)
        ops.check(ops.lib().mdt_vae_rows_to_nchw(ops.ptr(y), ops.ptr(img), B, H * W, OUT_CH, y.shape[1],
                                                 ops.stream_ptr()), "mdt_vae_rows_to_nchw")
        return img


class AutoencoderKLDecoder(_VaeBase):
    def __init__(self, scale_factor=0.18215, max_rows=1 << 21):
        shapes, plan = _shapes()
        super().__init__(shapes, scale_factor, max_rows)
        self._plan = plan

    # -- reference interface ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def decode(self, z):
        """FrozenAutoencoderKL.decode (autoencoder.py:449-453): z [B,4,h,w] -> images [B,3,8h,8w] f32."""
        return self._decode(z)

    def forward(self, inputs, fn="decode"):
        if fn != "decode":
            raise NotImplementedError("only the decode half of the autoencoder is on the sampling path")
        return self.decode(inputs)


def get_model(pretrained_path=None, scale_factor=0.18215, device="cuda"):
    """autoencoder.get_model (autoencoder.py:466-479) for the decode half: loads `decoder.*` / `post_quant_conv.*` from a
    FrozenAutoencoderKL checkpoint (encoder / quant_conv entries are ignored)."""
    m = AutoencoderKLDecoder(scale_factor)
    if pretrained_path is not None:
        sd = torch.load(pretrained_path, map_location="cpu", weights_only=True)
        own = set(m.state_dict().keys())
        missing = own - set(sd.keys())
        if missing:
            raise KeyError(f"checkpoint lacks decoder tensors: {sorted(missing)[:4]} ...")
        m.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=True)
    return m.to(device).eval()


class AutoencoderKL(_VaeBase):
    """FrozenAutoencoderKL (autoencoder.py:415-463) with both halves: `encoder.*`, `decoder.*`, `quant_conv.*`,
    `post_quant_conv.*` in the reference's registration order, so a published `autoencoder_kl.pth` loads with
    `strict=True`.  `encode_moments(x)` is what extract_latent.py stores for training; `decode(z)` is bit-identical to
    `AutoencoderKLDecoder.decode`."""

    def __init__(self, scale_factor=0.18215, max_rows=1 << 21):
        dec, plan = _shapes()
        enc, enc_plan = _encoder_shapes()
        pq = [kv for kv in dec if kv[0].startswith("post_quant_conv.")]
        dec = [kv for kv in dec if not kv[0].startswith("post_quant_conv.")]
        quant = [("quant_conv.weight", (2 * Z_CH, 2 * Z_CH, 1, 1)), ("quant_conv.bias", (2 * Z_CH,))]
        super().__init__(enc + dec + quant + pq, scale_factor, max_rows)
        self._plan, self._enc_plan = plan, enc_plan

    @torch.no_grad()
    def encode_moments(self, x, flip=False):
        """FrozenAutoencoderKL.encode_moments (autoencoder.py:431-434): x [B,3,H,W] f32 in [-1,1], H and W multiples of 8
        -> moments [B,8,H/8,W/8] f32 (mean, logvar).  flip=True encodes x mirrored along W (`x.flip(-1)`) without a
        copy."""
        if x.ndim != 4 or x.shape[1] != IN_CH or x.shape[2] % 8 or x.shape[3] % 8 or x.shape[0] == 0:
            raise ops.L.MdtError(f"encode_moments takes [B,3,H,W] with H and W multiples of 8, got {tuple(x.shape)}")
        if not x.is_cuda or x.dtype != f32:
            raise ops.L.MdtError("encode_moments takes a CUDA float32 tensor [B,3,H,W] (there is no CPU fallback)")
        self._ready()
        x = x.contiguous()
        B, _, H, W = x.shape
        rows = torch.empty(B * H * W, 4, dtype=f32, device=x.device)
        ops.check(ops.lib().mdt_vae_image_to_rows(ops.ptr(x), ops.ptr(rows), B, H, W, int(bool(flip)),
                                                  ops.stream_ptr()), "mdt_vae_image_to_rows")
        h = self._conv(rows, B, H, W, 4, "encoder.conv_in")
        for lvl in range(len(CH_MULT)):
            for i in range(NUM_RES_BLOCKS):
                cin, cout = self._enc_plan[(lvl, i)]
                h = self._resblock(h, B, H, W, f"encoder.down.{lvl}.block.{i}", cin, cout)
            if lvl != len(CH_MULT) - 1:
                H, W = H // 2, W // 2
                h = self._conv(h, B, H, W, cout, f"encoder.down.{lvl}.downsample.conv", down=True)
        c = CH * CH_MULT[-1]
        h = self._resblock(h, B, H, W, "encoder.mid.block_1", c, c)
        h = self._attn(h, B, H, W, "encoder.mid.attn_1", c)
        h = self._resblock(h, B, H, W, "encoder.mid.block_2", c, c)
        y = self._conv(h, B, H, W, c, "encoder.conv_out", norm="encoder.norm_out", silu=True)      # [M, 8]
        moments = torch.empty(B, 2 * Z_CH, H, W, dtype=f32, device=x.device)
        ops.check(ops.lib().mdt_vae_quant_out(ops.ptr(y), y.shape[1], ops.ptr(self._packed["quant_conv.weight"]),
                                              ops.ptr(self._packed["quant_conv.bias"]), ops.ptr(moments), B, 2 * Z_CH,
                                              H * W, ops.stream_ptr()), "mdt_vae_quant_out")
        return moments

    @torch.no_grad()
    def decode(self, z):
        """FrozenAutoencoderKL.decode (autoencoder.py:449-453): z [B,4,h,w] -> images [B,3,8h,8w] f32."""
        return self._decode(z)

    def forward(self, inputs, fn):
        """FrozenAutoencoderKL.forward (autoencoder.py:455-463) for 'encode_moments' and 'decode'.  The reference's
        'encode' (moments -> sampled latent) is not here: training samples latents from the stored moments."""
        if fn == "encode_moments":
            return self.encode_moments(inputs)
        if fn == "decode":
            return self.decode(inputs)
        raise NotImplementedError(f"AutoencoderKL.forward: fn={fn!r} (supported: 'encode_moments', 'decode')")


def get_autoencoder(pretrained_path=None, device="cuda", scale_factor=0.18215):
    """autoencoder.get_model (autoencoder.py:466-479) with both halves: loads a FrozenAutoencoderKL checkpoint
    (`autoencoder_kl.pth`) with `strict=True`.  Without a path the weights stay zero (load a state dict afterwards)."""
    m = AutoencoderKL(scale_factor)
    if pretrained_path is not None:
        sd = torch.load(pretrained_path, map_location="cpu", weights_only=True)
        m.load_state_dict(sd, strict=True)
    return m.to(device).eval()
