"""TEST INFRASTRUCTURE ONLY — CPU fp32 restatement of the reference's SD-VAE ENCODE path (autoencoder.py:212-303,
:431-434), the `encode_moments` that extract_latent.py runs on every image batch to build the training LMDB.
The product path (`maskdit_b200/vae.py`) never imports it; it is pinned against the unmodified reference `Encoder` +
`quant_conv` by tests/golden/make_golden_vae_encode.py + tests/test_vae_encode.py.

Parameters are a flat dict keyed like `FrozenAutoencoderKL.state_dict()` (`encoder.*`, `quant_conv.*`).  The decoder
half lives in oracle/vae_oracle.py, whose building blocks this module reuses.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from .vae_oracle import CH, CH_MULT, NUM_RES_BLOCKS, Z_CH, _attn, _conv, _gn, _resblock, _swish

IN_CH = 3


def encoder_param_shapes():
    """Key -> shape of `encoder` (Encoder.__init__, autoencoder.py:212-278) then `quant_conv` (:424), in registration
    order."""
    out = {"encoder.conv_in.weight": (CH, IN_CH, 3, 3), "encoder.conv_in.bias": (CH,)}

    def res(p, cin, cout):
        out[f"{p}.norm1.weight"], out[f"{p}.norm1.bias"] = (cin,), (cin,)
        out[f"{p}.conv1.weight"], out[f"{p}.conv1.bias"] = (cout, cin, 3, 3), (cout,)
        out[f"{p}.norm2.weight"], out[f"{p}.norm2.bias"] = (cout,), (cout,)
        out[f"{p}.conv2.weight"], out[f"{p}.conv2.bias"] = (cout, cout, 3, 3), (cout,)
        if cin != cout:
            out[f"{p}.nin_shortcut.weight"], out[f"{p}.nin_shortcut.bias"] = (cout, cin, 1, 1), (cout,)

    in_ch_mult = (1,) + tuple(CH_MULT)
    for lvl in range(len(CH_MULT)):
        block_in, block_out = CH * in_ch_mult[lvl], CH * CH_MULT[lvl]
        for i in range(NUM_RES_BLOCKS):
            res(f"encoder.down.{lvl}.block.{i}", block_in, block_out)
            block_in = block_out
        if lvl != len(CH_MULT) - 1:
            out[f"encoder.down.{lvl}.downsample.conv.weight"] = (block_in, block_in, 3, 3)
            out[f"encoder.down.{lvl}.downsample.conv.bias"] = (block_in,)
    res("encoder.mid.block_1", block_in, block_in)
    p = "encoder.mid.attn_1"
    out[f"{p}.norm.weight"], out[f"{p}.norm.bias"] = (block_in,), (block_in,)
    for n in ("q", "k", "v", "proj_out"):
        out[f"{p}.{n}.weight"], out[f"{p}.{n}.bias"] = (block_in, block_in, 1, 1), (block_in,)
    res("encoder.mid.block_2", block_in, block_in)
    out["encoder.norm_out.weight"], out["encoder.norm_out.bias"] = (block_in,), (block_in,)
    out["encoder.conv_out.weight"], out["encoder.conv_out.bias"] = (2 * Z_CH, block_in, 3, 3), (2 * Z_CH,)
    out["quant_conv.weight"], out["quant_conv.bias"] = (2 * Z_CH, 2 * Z_CH, 1, 1), (2 * Z_CH,)
    return out


def make_vae_encoder_state_dict(seed=5):
    """Deterministic stand-in weights for `encoder.*` + `quant_conv.*`, drawn like vae_oracle.make_vae_state_dict:
    conv weights N(0, 1/fan_in), GroupNorm scales 1 + 0.1 N(0,1), biases 0.05 N(0,1)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shp in encoder_param_shapes().items():
        if k.endswith("weight") and len(shp) == 4:
            fan_in = shp[1] * shp[2] * shp[3]
            sd[k] = torch.randn(shp, generator=g) * fan_in ** -0.5
        elif k.endswith("weight"):
            sd[k] = 1 + 0.1 * torch.randn(shp, generator=g)
        else:
            sd[k] = 0.05 * torch.randn(shp, generator=g)
    return sd


def _downsample(sd, p, x):
    """Downsample.forward with a convolution (autoencoder.py:56-75): asymmetric zero pad, 3x3 stride 2."""
    x = F.pad(x, (0, 1, 0, 1), mode="constant", value=0)
    return F.conv2d(x, sd[f"{p}.weight"], sd[f"{p}.bias"], stride=2)


def encode_moments(sd, x):
    """FrozenAutoencoderKL.encode_moments (autoencoder.py:431-434) + Encoder.forward (:280-303).
    x [B,3,H,W] -> moments [B,8,H/8,W/8] (mean, logvar)."""
    h = _conv(sd, "encoder.conv_in", x, 1)
    for lvl in range(len(CH_MULT)):
        for i in range(NUM_RES_BLOCKS):
            h = _resblock(sd, f"encoder.down.{lvl}.block.{i}", h)
        if lvl != len(CH_MULT) - 1:
            h = _downsample(sd, f"encoder.down.{lvl}.downsample.conv", h)
    h = _resblock(sd, "encoder.mid.block_1", h)
    h = _attn(sd, "encoder.mid.attn_1", h)
    h = _resblock(sd, "encoder.mid.block_2", h)
    h = _conv(sd, "encoder.conv_out", _swish(_gn(sd, "encoder.norm_out", h)), 1)
    return _conv(sd, "quant_conv", h, 0)


def center_crop_synthetic(w, h, seed):
    """A smooth colour gradient plus seeded noise, uint8 [h, w, 3]: the input of the center_crop golden (numpy's PCG64
    stream is platform-independent, so the images are regenerated instead of stored)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([255 * xx / max(1, w - 1), 255 * yy / max(1, h - 1), 127.5 + 0 * xx], axis=-1)
    return np.clip(base + rng.normal(0, 40, (h, w, 3)), 0, 255).astype(np.uint8)
