"""Encode an ImageFolder of images into the latent LMDB that `train.py` reads (the twin of the reference's
extract_latent.py, on the B200 kernels).

    python extract_latent.py --data_dir <root> --split train --resolution 256 --ckpt assets/vae/autoencoder_kl.pth \
        --outdir <out> [--xflip]

Images are read from `<data_dir>/<split>` in `torchvision.datasets.ImageFolder` order (the sample order and class
indices of the reference's `imagenet_lmdb_dataset`), center-cropped to `resolution` (`data.center_crop_arr`), scaled to
[-1, 1] and encoded with `vae.AutoencoderKL.encode_moments` on the GPU.  The result is
`<outdir>/<data_name>_<resolution>_latent_lmdb/<split>/data.mdb` with `z-{i}` (raw little-endian fp32 moments
[8, resolution/8, resolution/8]), `y-{i}` (decimal class index) and `length`; with `--xflip` the horizontally mirrored
images follow at indices N..2N-1.  Moments are streamed to disk as they are produced (`data.MdbWriter`).
"""
from __future__ import annotations

import argparse
import functools
import os
import time

import numpy as np
import torch

from maskdit_b200.data import MdbWriter, center_crop_arr
from maskdit_b200.vae import get_autoencoder


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--data_name", default="imagenet", type=str)
    p.add_argument("--data_dir", default="../datasets", type=str)
    p.add_argument("--ckpt", default="assets/vae/autoencoder_kl.pth", type=str, help="checkpoint path")
    p.add_argument("--resolution", default=512, type=int)
    p.add_argument("--batch_size", default=128, type=int)
    p.add_argument("--split", default="train", type=str)
    p.add_argument("--xflip", action="store_true")
    p.add_argument("--outdir", type=str, default="../data/imagenet512-latent", help="output directory")
    p.add_argument("--num_workers", default=8, type=int, help="DataLoader worker processes for decoding and cropping")
    args = p.parse_args(argv)
    if args.split not in ("train", "val"):
        p.error("--split must be 'train' or 'val'")
    if args.resolution % 8:
        p.error("--resolution must be a multiple of 8")
    return args


def make_loader(args):
    import torchvision.datasets as datasets
    import torchvision.transforms as transforms
    transform = transforms.Compose([
        transforms.Lambda(functools.partial(center_crop_arr, image_size=args.resolution)),
        transforms.ToTensor(),
        transforms.Normalize(mean=[0.5, 0.5, 0.5], std=[0.5, 0.5, 0.5]),
    ])
    dataset = datasets.ImageFolder(f"{args.data_dir}/{args.split}", transform=transform)
    loader = torch.utils.data.DataLoader(dataset, batch_size=args.batch_size, shuffle=False, drop_last=False,
                                         num_workers=args.num_workers, pin_memory=torch.cuda.is_available(),
                                         persistent_workers=args.num_workers > 0)
    return dataset, loader


def main(argv=None):
    args = parse_args(argv)
    dataset, loader = make_loader(args)
    print(f"data size: {len(dataset)}")
    model = get_autoencoder(args.ckpt, device="cuda")
    print(f"loaded vae weights from {args.ckpt}")
    target = os.path.join(args.outdir, f"{args.data_name}_{args.resolution}_latent_lmdb", args.split)
    idx = 0
    with MdbWriter(target) as db:
        for flip in ((False, True) if args.xflip else (False,)):
            begin = time.time()
            for img, label in loader:
                assert img.min() >= -1 and img.max() <= 1
                moments = model.encode_moments(img.cuda(non_blocking=True), flip=flip)
                assert moments.shape[-1] == args.resolution // 8
                moments = moments.cpu().numpy().astype("<f4", copy=False)
                for moment, lb in zip(moments, label.numpy()):
                    db.put(f"z-{idx}".encode(), np.ascontiguousarray(moment).tobytes())
                    db.put(f"y-{idx}".encode(), str(int(lb)).encode())
                    idx += 1
                if idx % 5120 < len(label):
                    print(f"saved {idx} latents, {time.time() - begin:.1f}s for this pass so far")
        db.put(b"length", str(idx).encode())
    print(f"[finished] saved {idx} latents to {target}")
    return target


if __name__ == "__main__":
    main()
