"""SD-VAE encode (`vae.AutoencoderKL.encode_moments`) and the latent-extraction data path (`data.MdbWriter`,
`data.center_crop_arr`, `extract_latent.py`).

CPU: the encoder oracle (oracle/vae_encode_oracle.py) against goldens produced by the UNMODIFIED reference Encoder +
quant_conv (tests/golden/make_golden_vae_encode.py), the state-dict layout, the reference's center crop, the streaming
LMDB writer and input validation.  GPU: the tcgen05 encode path against the same goldens, determinism, the fused
horizontal flip, decode parity with `AutoencoderKLDecoder`, full-size runs and `extract_latent.main` end to end."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from maskdit_b200 import data as D  # noqa: E402
from oracle import vae_encode_oracle as VE  # noqa: E402
from oracle import vae_oracle as VO  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def load(name):
    return {k: v for k, v in np.load(os.path.join(GOLD, name + ".npz")).items()}


def rel_l2(a, b):
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / b.norm()).item()


def full_state_dict():
    """Stand-in weights for every AutoencoderKL tensor: the encoder golden's encoder / quant_conv, the decoder golden's
    decoder / post_quant_conv."""
    return {**VE.make_vae_encoder_state_dict(5), **VO.make_vae_state_dict(3)}


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_encoder_oracle_matches_reference():
    g = load("vae_encode")
    sd = VE.make_vae_encoder_state_dict(5)
    n_enc = sum(int(np.prod(s)) for k, s in VE.encoder_param_shapes().items() if k.startswith("encoder."))
    assert n_enc == int(g["n_encoder_params"])
    with torch.no_grad():
        for case in ("a", "b"):
            m = VE.encode_moments(sd, torch.from_numpy(g[f"x_{case}"]))
            assert m.shape == g[f"moments_{case}"].shape
            np.testing.assert_allclose(m.numpy(), g[f"moments_{case}"], rtol=1e-4, atol=1e-4)


def test_autoencoder_state_dict_keys_match_reference():
    from maskdit_b200.vae import AutoencoderKL, AutoencoderKLDecoder
    g = load("vae_encode")
    keys = list(AutoencoderKL().state_dict().keys())
    assert keys == [str(k) for k in g["keys"]]
    # the oracle's weights load with strict=True; the decoder-only module keeps exactly the decoder half
    AutoencoderKL().load_state_dict(full_state_dict(), strict=True)
    assert set(AutoencoderKLDecoder().state_dict()) == {k for k in keys if k.startswith(("decoder.", "post_quant_conv."))}


def test_center_crop_matches_reference():
    """Exact equality with the reference's center_crop_arr run by the same Pillow.  (Pillow's resampling is integer
    fixed-point arithmetic, so another Pillow release may round single pixels differently: if this starts failing after
    a Pillow upgrade, the fair bound is max |diff| <= 1.)"""
    from PIL import Image
    g = load("center_crop")
    for case in ("box", "up"):
        w, h, seed = (int(v) for v in g[f"size_{case}"])
        out = np.asarray(D.center_crop_arr(Image.fromarray(VE.center_crop_synthetic(w, h, seed)), 64))
        assert out.shape == (64, 64, 3) and out.dtype == np.uint8
        assert np.array_equal(out, g[f"crop_{case}"]), (case, np.abs(out.astype(int) - g[f"crop_{case}"]).max())


def test_mdb_writer_streams_in_index_order(tmp_path):
    """Values put in index order (z-0, z-1, ..., z-10, ...: not key order), inline and overflow values mixed, deep
    enough for branch pages; everything reads back through MdbReader and ImageNetLatentDataset / batches."""
    rng = np.random.default_rng(4)
    n, R = 300, 4
    moments = rng.standard_normal((n, 8, R, R)).astype(np.float32)          # 512 B: inline leaf values
    big = rng.standard_normal((n // 10, 8, 32, 32)).astype(np.float32)     # 32 KB: overflow pages
    labels = rng.integers(0, 10, n)
    root = tmp_path / "lat"
    with D.MdbWriter(str(root / "train")) as w:
        for i in range(n):
            w.put(f"z-{i}".encode(), moments[i].astype("<f4").tobytes())
            w.put(f"y-{i}".encode(), str(int(labels[i])).encode())
            if i % 10 == 0:
                w.put(f"big-{i // 10}".encode(), big[i // 10].tobytes())
        w.put(b"length", str(n).encode())
        with pytest.raises(KeyError):
            w.put(b"length", b"0")
    rd = D.MdbReader(str(root / "train"))
    assert rd.entries == 2 * n + n // 10 + 1 and rd.depth >= 2
    for j in range(n // 10):
        assert bytes(rd.get(f"big-{j}".encode())) == big[j].tobytes()
    assert rd.get(b"z-300") is None
    rd.close()
    ds = D.ImageNetLatentDataset(str(root), resolution=R, num_classes=10)
    assert len(ds) == n
    for i in (0, 1, 9, 10, 11, 100, 299):
        z, y = ds.raw(i)
        assert np.array_equal(z, moments[i]) and y == labels[i]
    zb, yb = next(D.batches(ds, 7, pin=False))
    assert torch.equal(zb, torch.from_numpy(moments[:7])) and torch.equal(yb.argmax(1), torch.from_numpy(labels[:7]))


def test_encode_rejects_cpu_and_bad_shapes():
    from maskdit_b200._lib import MdtError
    from maskdit_b200.vae import AutoencoderKL
    vae = AutoencoderKL()
    with pytest.raises(MdtError):
        vae.encode_moments(torch.zeros(1, 3, 64, 64))
    dev = "cuda" if torch.cuda.is_available() else "cpu"     # the shape is checked before the device
    for shape in ((1, 3, 60, 64), (1, 3, 64, 36), (1, 4, 64, 64), (3, 64, 64)):
        with pytest.raises(MdtError, match="multiples of 8"):
            vae.encode_moments(torch.zeros(shape, device=dev))
    with pytest.raises(NotImplementedError):
        vae(torch.zeros(1, 3, 64, 64), "encode")


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _vae(max_rows=1 << 21):
    from maskdit_b200.vae import AutoencoderKL
    vae = AutoencoderKL(max_rows=max_rows)
    vae.load_state_dict(full_state_dict(), strict=True)
    return vae.cuda().eval()


@pytest.mark.gpu
def test_encode_vs_reference_golden_and_deterministic():
    g = load("vae_encode")
    vae = _vae()
    for case in ("a", "b"):
        x = torch.from_numpy(g[f"x_{case}"]).cuda()
        ref = g[f"moments_{case}"]
        m = vae.encode_moments(x)
        assert m.shape == ref.shape and torch.isfinite(m).all()
        r, rm, rv = rel_l2(m, ref), rel_l2(m[:, :4], ref[:, :4]), rel_l2(m[:, 4:], ref[:, 4:])
        print(f"VAE encode case {case} {tuple(x.shape)}: rel-L2 {r:.3e} (mean {rm:.3e}, logvar {rv:.3e}); "
              f"reference under CPU bf16 autocast: {float(g[f'autocast_rel_{case}']):.3e} "
              f"(mean {float(g[f'autocast_rel_mean_{case}']):.3e}, logvar {float(g[f'autocast_rel_logvar_{case}']):.3e})")
        assert r <= 1e-2, r
        # no atomics on the path: a rerun, and chunked im2col operands (several GEMM launches per convolution), agree
        # bit for bit
        assert torch.equal(vae.encode_moments(x), m)
        vae.max_rows = 2048
        assert torch.equal(vae.encode_moments(x), m)
        vae.max_rows = 1 << 21
        # the fused horizontal flip is the flip of the input
        assert torch.equal(vae.encode_moments(x, flip=True), vae.encode_moments(x.flip(-1).contiguous()))
        assert torch.equal(vae(x, "encode_moments"), m)


@pytest.mark.gpu
def test_autoencoder_decode_is_decoder_decode():
    from maskdit_b200.vae import AutoencoderKLDecoder
    g = load("vae_decode")
    dec = AutoencoderKLDecoder()
    dec.load_state_dict(VO.make_vae_state_dict(3), strict=True)
    dec = dec.cuda().eval()
    vae = _vae()
    z = torch.from_numpy(g["z"]).cuda()
    img = vae.decode(z)
    assert torch.equal(img, dec.decode(z))
    assert torch.equal(vae(z, "decode"), img)
    assert rel_l2(img, g["images"]) <= 1e-2


@pytest.mark.gpu
def test_encode_full_size():
    """256x256 at B = 4 (image 0 bit-equal to a B = 1 run: rows are independent) and 512x512 at B = 1 (mid attention
    over T = 4096 positions), stand-in weights."""
    vae = _vae()
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.rand(4, 3, 256, 256, generator=g, device="cuda") * 2 - 1
    m = vae.encode_moments(x)
    assert m.shape == (4, 8, 32, 32) and torch.isfinite(m).all()
    assert torch.equal(vae.encode_moments(x[:1].contiguous())[0], m[0])
    x = torch.rand(1, 3, 512, 512, generator=g, device="cuda") * 2 - 1
    m = vae.encode_moments(x)
    assert m.shape == (1, 8, 64, 64) and torch.isfinite(m).all()


@pytest.mark.gpu
def test_extract_latent_end_to_end(tmp_path):
    """A tiny ImageFolder (7 images of mixed sizes, 3 classes) -> extract_latent.main at resolution 64, batch 3 (one
    ragged batch), --xflip -> the LMDB reads back through ImageNetLatentDataset / batches with the ImageFolder targets
    twice and every z-{i} equal to encode_moments of the same preprocessed batch (flipped for the second half)."""
    from PIL import Image
    import extract_latent as X
    rng = np.random.default_rng(12)
    sizes = [(90, 70), (64, 64), (150, 200), (33, 47), (300, 128), (128, 300), (65, 80)]
    for i, (w, h) in enumerate(sizes):
        d = tmp_path / "imgs" / "train" / f"class_{'abc'[i % 3]}"
        d.mkdir(parents=True, exist_ok=True)
        Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(d / f"img{i}.png")
    ck = tmp_path / "autoencoder_kl.pth"
    torch.save(full_state_dict(), ck)
    argv = ["--data_dir", str(tmp_path / "imgs"), "--ckpt", str(ck), "--resolution", "64", "--batch_size", "3",
            "--split", "train", "--xflip", "--outdir", str(tmp_path / "out"), "--num_workers", "0"]
    target = X.main(argv)
    assert target == os.path.join(str(tmp_path / "out"), "imagenet_64_latent_lmdb", "train")
    ds = D.ImageNetLatentDataset(os.path.dirname(target), resolution=8, num_classes=3)
    assert len(ds) == 14
    dataset, loader = X.make_loader(X.parse_args(argv))
    targets = [t for _, t in dataset.samples]
    vae = _vae()
    want = []
    for flip in (False, True):
        for img, _ in loader:
            want.extend(vae.encode_moments(img.cuda(), flip=flip).cpu().numpy())
    for i in range(14):
        z, y = ds.raw(i)
        assert y == targets[i % 7], i
        assert np.array_equal(z, want[i]), i
    zb, yb = next(D.batches(ds, 14, pin=False))
    assert zb.shape == (14, 8, 8, 8) and yb.argmax(1).tolist() == targets * 2
