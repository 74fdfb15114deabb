"""Generate golden vectors by executing the UNMODIFIED reference (a checkout of the original MaskDiT) on CPU fp32.

    MDT_REFERENCE_DIR=<checkout of Anima-Lab/MaskDiT> python tests/golden/make_golden.py
Writes tests/golden/*.npz (small).  Weights are NOT stored: both the reference module and the oracle are loaded
from oracle.maskdit_oracle.make_state_dict(cfg, seed) which is deterministic on CPU.

Random draws of EDMLoss / get_mask are reproduced by re-seeding the CPU generator and drawing in the reference's
order (loss.py:35 randn[B,1,1,1]; loss.py:39 randn_like(images); maskdit.py:102 rand[B,L]) and are stored.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import maskdit_oracle as O  # noqa: E402
from oracle import timm_standin  # noqa: E402

timm_standin.install()
if not os.path.isdir(os.environ.get("MDT_REFERENCE_DIR", "")):
    sys.exit("set MDT_REFERENCE_DIR to a checkout of the original MaskDiT (models/maskdit.py, train_utils/loss.py, ...)")
sys.path.insert(0, os.environ["MDT_REFERENCE_DIR"])
import models.maskdit as rm  # noqa: E402
import sample as rs  # noqa: E402
import train_utils.loss as rl  # noqa: E402

torch.set_grad_enabled(True)
GRAD_KEYS_FULL = [
    "model.mask_token", "model.final_layer.linear.bias", "model.final_layer.linear.weight",
    "model.x_embedder.proj.bias", "model.t_embedder.mlp.0.bias", "model.t_embedder.mlp.2.bias",
    "model.decoder_layer.linear.bias", "model.blocks.0.attn.qkv.bias", "model.blocks.0.mlp.fc1.bias",
    "model.blocks.0.adaLN_modulation.1.bias", "model.decoder_blocks.7.adaLN_modulation.1.bias",
    "model.final_layer.adaLN_modulation.1.bias", "model.decoder_blocks.0.attn.proj.bias",
]


class Wrap:
    """EDMLoss needs `net.module` (loss.py:47,52) — i.e. a DDP-like wrapper."""

    def __init__(self, m):
        self.module = m
        self.model = m.model  # unwrap_model (helper.py:61-68) only unwraps real DDP; loss.py:57 then reads .model
        self.training = m.training

    def __call__(self, *a, **k):
        return self.module(*a, **k)


def build_ref(cfg: O.Cfg, seed=1):
    net = rm.Precond_models["edm"](img_resolution=cfg.img_resolution, img_channels=cfg.img_channels,
                                   num_classes=cfg.num_classes, model_type=cfg.model_type,
                                   use_decoder=cfg.use_decoder, mae_loss_coef=cfg.mae_loss_coef, pad_cls_token=False)
    sd = O.make_state_dict(cfg, seed)
    missing = net.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    assert set(net.state_dict().keys()) == set(O.param_shapes(cfg).keys())
    return net


def inputs(cfg, B, seed):
    g = torch.Generator().manual_seed(seed)
    images = torch.randn(B, cfg.img_channels, cfg.img_resolution, cfg.img_resolution, generator=g) * 0.5
    if not cfg.num_classes:
        return images, None
    cls = torch.randint(0, cfg.num_classes, (B,), generator=g)
    labels = torch.eye(cfg.num_classes)[cls]
    if B > 1:
        labels[-1] = 0  # one dropped label row (train.py:209)
    return images, labels


def train_case(name, cfg, B, mask_ratio, with_grads):
    net = build_ref(cfg).train()
    images, labels = inputs(cfg, B, seed=7)
    loss_fn = rl.Losses["edm"]()
    torch.manual_seed(123)
    loss = loss_fn(net=Wrap(net), images=images, labels=labels, mask_ratio=mask_ratio,
                   mae_loss_coef=cfg.mae_loss_coef)
    # reproduce the draws
    torch.manual_seed(123)
    rnd_normal = torch.randn([B, 1, 1, 1])
    noise_unit = torch.randn_like(images)
    mnoise = torch.rand(B, cfg.num_patches) if mask_ratio > 0 else None
    out = dict(images=images.numpy(), **({"labels": labels.numpy()} if labels is not None else {}),
               rnd_normal=rnd_normal.numpy(),
               noise_unit=noise_unit.numpy(), loss=loss.detach().numpy(), mask_ratio=np.float32(mask_ratio))
    sigma = (rnd_normal * 1.2 - 1.2).exp()
    if mask_ratio > 0:
        out["mask_noise"] = mnoise.numpy()
        md = O.mask_from_noise(mnoise, mask_ratio)
        # net output with the same mask injected must reproduce the loss path's D
        res = net(images + noise_unit * sigma, sigma, labels, mask_ratio=mask_ratio, mask_dict=md)
        # and the reference's own unstable argsort must agree with the stable rule on tie-free noise
        torch.manual_seed(5)
        ref_md = rm.get_mask(B, cfg.num_patches, mask_ratio, "cpu")
        torch.manual_seed(5)
        chk = O.mask_from_noise(torch.rand(B, cfg.num_patches), mask_ratio)
        for k in ("mask", "ids_keep", "ids_restore"):
            assert torch.equal(ref_md[k], chk[k]), k
        out.update(mask=md["mask"].numpy(), ids_keep=md["ids_keep"].numpy(), ids_restore=md["ids_restore"].numpy())
    else:
        res = net(images + noise_unit * sigma, sigma, labels)
    out["D"] = res["x"].detach().numpy()
    if with_grads:
        net.zero_grad()
        loss.mean().backward()
        for k, p in net.named_parameters():
            if p.grad is None:
                continue
            g = p.grad
            out[f"gnorm/{k}"] = np.float64(g.double().norm().item())
            if k in GRAD_KEYS_FULL:
                out[f"grad/{k}"] = g.numpy()
            elif g.ndim >= 2:
                out[f"gslice/{k}"] = g.reshape(g.shape[0], -1)[:4, :8].numpy().copy()
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **out)
    print(name, "loss", loss.detach().numpy())


def eval_case(name, cfg, B, num_steps=18):
    net = build_ref(cfg).eval()
    images, labels = inputs(cfg, B, seed=11)
    sigma = torch.tensor([0.3, 2.5][:B] if B <= 2 else np.linspace(0.1, 5, B), dtype=torch.float32)
    with torch.no_grad():
        plain = net(images, sigma, labels)["x"]
        s0 = torch.tensor(1.7, dtype=torch.float64)  # 0-d fp64 sigma, as the sampler passes it (sample.py:56)
        cfgout = net(images, s0, labels, 1.5)["x"]
        rnd = rs.StackedRandomGenerator("cpu", list(range(B)))
        latents = rnd.randn([B, cfg.img_channels, cfg.img_resolution, cfg.img_resolution])
        sig_seen = []
        orig_forward = net.forward

        def spy(x, sigma, *a, **k):
            sig_seen.append(float(sigma))
            return orig_forward(x, sigma, *a, **k)

        net.forward = spy
        z = rs.edm_sampler(net, latents, labels, cfg_scale=1.5, randn_like=rnd.randn_like, num_steps=num_steps)
        net.forward = orig_forward
    assert len(sig_seen) == 2 * num_steps - 1
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), images=images.numpy(), labels=labels.numpy(),
                        sigma=sigma.numpy(), D_plain=plain.numpy(), D_cfg=cfgout.numpy(), latents=latents.numpy(),
                        z=z.numpy(), sampler_sigmas=np.array(sig_seen),
                        **({} if num_steps == 18 else {"num_steps": np.int64(num_steps)}))  # (s2_eval predates the key)
    print(name, "sampler |z|", z.abs().mean().item())


def churn_case(name, cfg, B):
    """Sampler with stochastic churn (sample.py:50-53), no guidance: pins gamma / t_hat / noise injection."""
    net = build_ref(cfg).eval()
    _, labels = inputs(cfg, B, seed=13)
    kw = dict(num_steps=8, S_churn=30.0, S_min=0.05, S_max=50.0, S_noise=1.003)
    with torch.no_grad():
        rnd = rs.StackedRandomGenerator("cpu", list(range(B)))
        latents = rnd.randn([B, cfg.img_channels, cfg.img_resolution, cfg.img_resolution])
        noises, sig_seen = [], []

        def randn_like(x):
            n = rnd.randn_like(x)
            noises.append(n.numpy().copy())
            return n

        orig_forward = net.forward

        def spy(x, sigma, *a, **k):
            sig_seen.append(float(sigma))
            return orig_forward(x, sigma, *a, **k)

        net.forward = spy
        z = rs.edm_sampler(net, latents, labels, randn_like=randn_like, **kw)
        net.forward = orig_forward
    assert len(sig_seen) == 15 and len(noises) == 8
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), labels=labels.numpy(), latents=latents.numpy(),
                        noises=np.stack(noises), z=z.numpy(), sampler_sigmas=np.array(sig_seen),
                        **{k: np.float64(v) for k, v in kw.items()})
    print(name, "sampler |z|", z.abs().mean().item(), "sigmas", sig_seen[:4])


def table_case():
    out = {}
    for D, g in ((1152, 16), (512, 16), (384, 4), (512, 4), (1152, 32)):
        out[f"pos_{D}_{g}"] = rm.get_2d_sincos_pos_embed(D, g).astype(np.float32)[:: max(1, g * g // 16)]
    t = torch.tensor([-1.5, -0.3, 0.0, 0.4, 1.1])
    out["tfreq_in"] = t.numpy()
    out["tfreq"] = rm.TimestepEmbedder.timestep_embedding(t, 256).numpy()
    # mask path incl. exact ties (duplicates in the noise row): stable argsort is the contract
    torch.manual_seed(3)
    for L, r in ((256, 0.5), (1024, 0.5), (256, 0.75), (16, 0.5)):
        noise = torch.rand(4, L)
        noise[1, ::7] = noise[1, 3]  # force ties
        md = O.mask_from_noise(noise, r)
        out[f"mask_noise_{L}_{r}"] = noise.numpy()
        for k, v in md.items():
            out[f"mask_{k}_{L}_{r}"] = v.numpy()
    np.savez_compressed(os.path.join(HERE, "tables.npz"), **out)
    print("tables ok")


def front_case(name):
    """Step front of the training loop (train.py:206-209 + loss.py:35-39) executed with the reference's own functions:
    utils.sample on VAE moments, label dropout, sigma draw, noise injection; all draws recorded."""
    import utils as ru
    B, C, R, ncls = 6, 4, 8, 10
    g = torch.Generator().manual_seed(21)
    moments = torch.randn(B, 2 * C, R, R, generator=g)
    moments[0, C:] = 25.0      # logvar above the clamp (20)
    moments[1, C:] = -40.0     # below the clamp (-30)
    labels = torch.eye(ncls)[torch.randint(0, ncls, (B,), generator=g)]
    drop_prob = 0.4
    torch.manual_seed(77)
    x = ru.sample(moments)                                                  # train.py:206
    y = labels * (torch.rand([B, 1]) >= drop_prob)                         # train.py:209
    rnd_normal = torch.randn([B, 1, 1, 1])                                 # loss.py:35
    sigma = (rnd_normal * 1.2 - 1.2).exp()                                 # loss.py:36
    n = torch.randn_like(x) * sigma                                        # loss.py:39
    torch.manual_seed(77)                                                  # reproduce the draws
    eps = torch.randn(B, C, R, R)
    drop_u = torch.rand([B, 1])
    rn2 = torch.randn([B, 1, 1, 1])
    noise_unit = torch.randn(B, C, R, R)
    assert torch.equal(rn2, rnd_normal)
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), moments=moments.numpy(), labels=labels.numpy(),
                        eps=eps.numpy(), drop_u=drop_u.reshape(B).numpy(), drop_prob=np.float32(drop_prob),
                        rnd_normal=rnd_normal.reshape(B).numpy(), noise_unit=noise_unit.numpy(), y=x.numpy(),
                        yn=(x + n).numpy(), sigma=sigma.reshape(B).numpy(), labels_out=y.numpy())
    print(name, "dropped rows", int((y.sum(1) == 0).sum()))


def ablation_case(name, cfg, B):
    """ablation_sampler (sample.py:73-188) for every discretization / schedule / scaling family, both solvers, with
    churn on one of them; 5 steps each."""
    net = build_ref(cfg).eval()
    _, labels = inputs(cfg, B, seed=17)
    combos = [dict(solver="heun", discretization="edm", schedule="linear", scaling="none"),
              dict(solver="euler", discretization="vp", schedule="vp", scaling="vp"),
              dict(solver="heun", discretization="ve", schedule="ve", scaling="none"),
              dict(solver="heun", discretization="iddpm", schedule="linear", scaling="none", alpha=0.75,
                   S_churn=10.0, S_min=0.05, S_max=50.0, S_noise=1.003),
              dict(solver="heun", discretization="vp", schedule="linear", scaling="vp")]
    out = dict(labels=labels.numpy(), n=np.int64(len(combos)))
    with torch.no_grad():
        for ci, kw in enumerate(combos):
            rnd = rs.StackedRandomGenerator("cpu", list(range(B)))
            latents = rnd.randn([B, cfg.img_channels, cfg.img_resolution, cfg.img_resolution])
            noises, sig_seen = [], []

            def randn_like(x):
                nz = rnd.randn_like(x)
                noises.append(nz.numpy().copy())
                return nz

            orig_forward = net.forward

            def spy(x, sigma, *a, **k):
                sig_seen.append(float(sigma))
                return orig_forward(x, sigma, *a, **k)

            net.forward = spy
            z = rs.ablation_sampler(net, latents, labels, cfg_scale=1.5 if ci % 2 == 0 else None,
                                    randn_like=randn_like, num_steps=5, **kw)
            net.forward = orig_forward
            out[f"latents{ci}"], out[f"z{ci}"] = latents.numpy(), z.numpy()
            out[f"noises{ci}"], out[f"sigmas{ci}"] = np.stack(noises), np.array(sig_seen)
            out[f"kw{ci}"] = np.array(repr(kw))
            print(name, ci, kw["discretization"], "evals", len(sig_seen), "|z|", z.abs().mean().item())
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **out)


def vae_case(name):
    """SD-VAE decode (autoencoder.py:449-453; the sampler tail, sample.py:275,287) by the unmodified reference module
    with the stand-in weights of oracle.vae_oracle.make_vae_state_dict: 8x8 latents -> 64x64 images."""
    import io
    import contextlib
    import tempfile
    import autoencoder as ra
    from oracle import vae_oracle as VO
    sd = VO.make_vae_state_dict(3)
    with contextlib.redirect_stdout(io.StringIO()):
        dec = ra.Decoder(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
                         ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0).eval()
    dsd = {k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}
    assert list(dsd.keys()) == list(dec.state_dict().keys())          # same keys in the same registration order
    dec.load_state_dict(dsd, strict=True)
    pq = torch.nn.Conv2d(4, 4, 1)
    pq.load_state_dict({"weight": sd["post_quant_conv.weight"], "bias": sd["post_quant_conv.bias"]})
    g = torch.Generator().manual_seed(31)
    z = torch.randn(2, 4, 8, 8, generator=g) * 0.18215 * 4.0
    with torch.no_grad():
        img = dec(pq((1.0 / 0.18215) * z))                               # FrozenAutoencoderKL.decode, :449-453
        u8 = img.clone().add_(1).mul(127.5).clamp_(0, 255).to(torch.uint8).permute(0, 2, 3, 1)   # sample.py:287
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), z=z.numpy(), images=img.numpy(), u8=u8.numpy())
    print(name, "image range", img.min().item(), img.max().item(), "mean |img|", img.abs().mean().item())


def round2_cases():
    """Round 2: goldens that reach the PRODUCTION kernels (VERDICT r1 weak #1): XL/2 at R=32 has T=128 kept tokens,
    so B=2 gives M=256 token rows (2-CTA GEMM tiles) and the split-tile tcgen05 attention forward/backward
    (head_dim 72 / 32); the eval/CFG case runs T=256, head_dim 72; R=64 runs the blocked T=512 / L=1024 kernels."""
    xl = O.Cfg(model_type="DiT-XL/2", img_resolution=32, num_classes=1000)
    train_case("xl2_c1_grads", xl, B=2, mask_ratio=0.5, with_grads=True)
    eval_case("xl2_eval", xl, B=2, num_steps=3)
    xl64 = O.Cfg(model_type="DiT-XL/2", img_resolution=64, num_classes=1000)
    train_case("xl2_r64_grads", xl64, B=1, mask_ratio=0.5, with_grads=True)
    round2_small()


def round2_small():
    # class-UNconditional net (num_classes = 0: no y_embedder, labels None) with 30 % masking: T = int(256 * 0.7) = 179 kept
    # tokens - an odd token count (no tcgen05 attention tile fits: the mma.sync kernels) and odd GEMM M, batch 3
    train_case("s2_uncond_mask30", O.Cfg(model_type="DiT-S/2", img_resolution=32, num_classes=0), B=3, mask_ratio=0.3,
               with_grads=True)
    vae_case("vae_decode")
    front_case("step_front")
    ablation_case("s2_ablation", O.Cfg(model_type="DiT-S/2", img_resolution=8, num_classes=10), B=2)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "round2":
        round2_cases()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "round2_small":
        round2_small()
        sys.exit(0)
    small = O.Cfg(model_type="DiT-S/2", img_resolution=8, num_classes=10)
    train_case("s2_train_mask", small, B=2, mask_ratio=0.5, with_grads=True)
    train_case("s2_train_nomask", small, B=2, mask_ratio=0.0, with_grads=True)
    eval_case("s2_eval", small, B=2)
    table_case()
    churn_case("s2_sampler_churn", small, B=2)
    # another geometry: patch 4 (16 latents per side -> 16 patches), 12 heads of 64, three of four patches masked
    b4 = O.Cfg(model_type="DiT-B/4", img_resolution=16, num_classes=7)
    train_case("b4_train_mask75", b4, B=3, mask_ratio=0.75, with_grads=True)
    xl = O.Cfg(model_type="DiT-XL/2", img_resolution=32, num_classes=1000)
    train_case("xl2_c1_fwd", xl, B=2, mask_ratio=0.5, with_grads=False)
    round2_cases()
