"""Generate the SD-VAE encode golden vectors by executing the UNMODIFIED reference (a checkout of the original MaskDiT)
on CPU fp32: its `Encoder` + quant_conv (autoencoder.py) and its image preprocessing `center_crop_arr`
(train_utils/datasets.py).

    MDT_REFERENCE_DIR=<checkout of Anima-Lab/MaskDiT> python tests/golden/make_golden_vae_encode.py
Writes tests/golden/vae_encode.npz and tests/golden/center_crop.npz (small) and nothing else; the other fixtures come
from make_golden.py.  Weights are NOT stored: they are oracle.vae_encode_oracle.make_vae_encoder_state_dict(5) and
oracle.vae_oracle.make_vae_state_dict(3), deterministic on CPU.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
if not os.path.isdir(os.environ.get("MDT_REFERENCE_DIR", "")):
    sys.exit("set MDT_REFERENCE_DIR to a checkout of the original MaskDiT (autoencoder.py, train_utils/datasets.py)")
sys.path.insert(0, os.environ["MDT_REFERENCE_DIR"])


def vae_encode_case(name):
    """SD-VAE encode_moments (autoencoder.py:431-434; extract_latent.py:77) by the unmodified reference `Encoder` + a
    Conv2d(8, 8, 1) holding quant_conv, with the stand-in weights of
    oracle.vae_encode_oracle.make_vae_encoder_state_dict: case A x [2,3,64,64], case B x [1,3,48,80] (mid attention over
    6 x 10 = 60 positions).  Also stores the FrozenAutoencoderKL state-dict key list (from the real class, loading a
    checkpoint of every tensor) and the rel-L2 that PyTorch's CPU bf16 autocast of the same modules reaches."""
    import io
    import contextlib
    import tempfile
    import autoencoder as ra
    from oracle import vae_oracle as VO
    from oracle import vae_encode_oracle as VE
    ddconfig = dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=[1, 2, 4, 4],
                    num_res_blocks=2, attn_resolutions=[], dropout=0.0)           # autoencoder.py:467-477
    sd = VE.make_vae_encoder_state_dict(5)
    with contextlib.redirect_stdout(io.StringIO()):
        enc = ra.Encoder(**ddconfig).eval()
        full = {**{f"encoder.{k}": v for k, v in enc.state_dict().items()},
                **{f"decoder.{k}": v for k, v in ra.Decoder(**ddconfig).state_dict().items()}}
        full.update({k: v for k, v in VO.make_vae_state_dict(3).items()})
        full.update({k: v for k, v in sd.items() if k.startswith("quant_conv.")})
        with tempfile.TemporaryDirectory() as td:
            ck = os.path.join(td, "autoencoder_kl.pth")
            torch.save(full, ck)
            keys = list(ra.get_model(ck).state_dict().keys())                    # strict load asserts the key set
    esd = {k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}
    assert list(esd.keys()) == list(enc.state_dict().keys())          # same keys in the same registration order
    enc.load_state_dict(esd, strict=True)
    qc = torch.nn.Conv2d(8, 8, 1)
    qc.load_state_dict({"weight": sd["quant_conv.weight"], "bias": sd["quant_conv.bias"]})
    n_enc = sum(p.numel() for p in enc.parameters())
    g = torch.Generator().manual_seed(41)
    xa = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
    xb = torch.rand(1, 3, 48, 80, generator=g) * 2 - 1
    out = dict(keys=np.array(keys), n_encoder_params=np.int64(n_enc))

    def rel(a, b):
        return np.float64(((a.double() - b.double()).norm() / b.double().norm()).item())

    with torch.no_grad():
        for case, x in (("a", xa), ("b", xb)):
            m = qc(enc(x))                                                       # FrozenAutoencoderKL.encode_moments
            with torch.autocast("cpu", dtype=torch.bfloat16):
                mb = qc(enc(x)).float()
            out[f"x_{case}"], out[f"moments_{case}"] = x.numpy(), m.numpy()
            out[f"autocast_rel_{case}"] = rel(mb, m)
            out[f"autocast_rel_mean_{case}"] = rel(mb[:, :4], m[:, :4])
            out[f"autocast_rel_logvar_{case}"] = rel(mb[:, 4:], m[:, 4:])
            print(name, case, "moments", tuple(m.shape), "|m|", m.abs().mean().item(), "bf16 autocast rel-L2",
                  out[f"autocast_rel_{case}"], "(mean", out[f"autocast_rel_mean_{case}"], "logvar",
                  out[f"autocast_rel_logvar_{case}"], ")")
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **out)


def center_crop_case(name):
    """The reference's center_crop_arr (train_utils/datasets.py:19-37) on two seeded synthetic RGB images: 700x530 -> 64
    (three BOX halvings, then BICUBIC down) and 50x37 -> 64 (BICUBIC up).  The images are regenerated from their seeds
    by the test (numpy's PCG64 stream is platform-independent), so only the crops are stored."""
    import types
    from PIL import Image
    sys.modules.setdefault("lmdb", types.ModuleType("lmdb"))   # datasets.py imports lmdb at the top; unused here
    import train_utils.datasets as rd
    from oracle.vae_encode_oracle import center_crop_synthetic
    out = {}
    for case, (w, h, seed) in (("box", (700, 530, 1)), ("up", (50, 37, 2))):
        arr = center_crop_synthetic(w, h, seed)
        out[f"crop_{case}"] = np.asarray(rd.center_crop_arr(Image.fromarray(arr), 64))
        out[f"size_{case}"] = np.array([w, h, seed], dtype=np.int64)
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **out)
    print(name, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    vae_encode_case("vae_encode")
    center_crop_case("center_crop")
