"""SD-VAE encode throughput on the GPU: `vae.AutoencoderKL.encode_moments` vs the fp32 restatement of the reference
encoder (oracle/vae_encode_oracle.py) run by PyTorch under bf16 autocast with channels_last (cuDNN convolutions), on
the same inputs, timed in alternating windows.

    python tools/bench_vae_encode.py [--sizes 256x32,512x8] [--ckpt autoencoder_kl.pth] [--out result.json]

Per size (resolution x batch) it reports images/s, algorithmic FLOPs per image (counted below from the convolution
shapes), achieved TF/s, im2col operand bytes written per image, kernel launches and peak memory of one call, and the
split of GPU time between im2col and GEMM kernels (torch.profiler, in a pass of its own after the timed windows).
Stand-in weights unless --ckpt.  Prints one JSON object; --out also writes it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from maskdit_b200 import _lib as L  # noqa: E402
from maskdit_b200 import vae as V  # noqa: E402
from oracle import vae_encode_oracle as VE  # noqa: E402
from oracle import vae_oracle as VO  # noqa: E402


def encoder_counts(H, W):
    """(FLOPs, im2col operand bytes) of one image's encode_moments at H x W, from the layer shapes (multiply-add = 2)."""
    flops = 0
    a_bytes = 0

    def conv(h, w, cin, cout, ks):
        nonlocal flops, a_bytes
        K = ks * ks * ((cin + 3) // 4 * 4)
        flops += 2 * h * w * cout * ks * ks * cin
        a_bytes += h * w * ((K + 7) // 8 * 8) * 2                 # bf16 im2col operand
    conv(H, W, 3, V.CH, 3)
    _, plan = V._encoder_shapes()
    c = V.CH
    for lvl in range(len(V.CH_MULT)):
        for i in range(V.NUM_RES_BLOCKS):
            cin, cout = plan[(lvl, i)]
            conv(H, W, cin, cout, 3)
            conv(H, W, cout, cout, 3)
            if cin != cout:
                conv(H, W, cin, cout, 1)
            c = cout
        if lvl != len(V.CH_MULT) - 1:
            H, W = H // 2, W // 2
            conv(H, W, c, c, 3)
    for _ in range(2):                                             # mid.block_1, mid.block_2
        conv(H, W, c, c, 3)
        conv(H, W, c, c, 3)
    T = H * W
    a_bytes += T * c * 2                                           # normalised input of q / k / v (one operand)
    flops += 4 * 2 * T * c * c + 2 * 2 * T * T * c                 # q, k, v, proj_out; q k^T and P v
    conv(H, W, c, 2 * V.Z_CH, 3)                                   # conv_out
    flops += 2 * T * (2 * V.Z_CH) ** 2                             # quant_conv
    return flops, a_bytes


def timed(fn, seconds):
    """Calls of `fn` in a window of at least `seconds` (CUDA events); returns seconds per call."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    n = max(2, int(seconds / max(1e-6, e0.elapsed_time(e1) / 1e3)) + 1)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3 / n


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clk = (s.strip() for s in q.stdout.strip().split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:                                          # noqa: BLE001 - reported, not fatal
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


def kernel_split(fn):
    """GPU time of one call by kernel family, from torch.profiler (a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    fam = {"im2col": 0.0, "gemm": 0.0, "other": 0.0}
    top = {}
    for ev in prof.key_averages():
        t = ev.self_device_time_total if hasattr(ev, "self_device_time_total") else ev.self_cuda_time_total
        if t <= 0:
            continue
        k = "im2col" if "im2col" in ev.key else "gemm" if "gemm" in ev.key.lower() else "other"
        fam[k] += t / 1e3
        top[ev.key[:80]] = round(t / 1e3, 3)
    tot = sum(fam.values())
    return {"ms": {k: round(v, 3) for k, v in fam.items()}, "share": {k: round(v / tot, 3) for k, v in fam.items()},
            "top_kernels_ms": dict(sorted(top.items(), key=lambda kv: -kv[1])[:8])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="256x32,512x8", help="comma-separated RESOLUTIONxBATCH")
    ap.add_argument("--ckpt", default=None)
    ap.add_argument("--seconds", type=float, default=1.5, help="length of each timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternating (ours, cuDNN) window pairs per size")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_vae_encode needs a CUDA device")
    torch.backends.cudnn.benchmark = True
    if args.ckpt:
        sd = torch.load(args.ckpt, map_location="cpu", weights_only=True)
    else:
        sd = {**VE.make_vae_encoder_state_dict(5), **VO.make_vae_state_dict(3)}
    vae = V.AutoencoderKL()
    vae.load_state_dict(sd, strict=True)
    vae = vae.cuda().eval()
    osd = {k: (v.cuda().to(memory_format=torch.channels_last) if v.ndim == 4 else v.cuda())
           for k, v in sd.items() if k.startswith(("encoder.", "quant_conv."))}

    def cudnn(x):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return VE.encode_moments(osd, x)

    result = {"what": "SD-VAE encode_moments, stand-in weights" if not args.ckpt else "SD-VAE encode_moments",
              "card": card(), "torch": torch.__version__, "cudnn": torch.backends.cudnn.version(), "sizes": []}
    for spec in args.sizes.split(","):
        res, B = (int(v) for v in spec.lower().split("x"))
        g = torch.Generator(device="cuda").manual_seed(res + B)
        x = torch.rand(B, 3, res, res, generator=g, device="cuda") * 2 - 1
        xc = x.contiguous(memory_format=torch.channels_last)
        ours = lambda: vae.encode_moments(x)                      # noqa: E731
        ref = lambda: cudnn(xc)                                   # noqa: E731
        ours()                                                    # packs the weights once
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        l0 = L.LAUNCHES
        m = ours()
        torch.cuda.synchronize()
        launches = L.LAUNCHES - l0
        peak = torch.cuda.max_memory_allocated()
        mr = ref().float()
        agree = ((m.double() - mr.double()).norm() / mr.double().norm()).item()
        t_ours, t_ref = [], []
        for _ in range(args.rounds):
            t_ours.append(timed(ours, args.seconds))
            t_ref.append(timed(ref, args.seconds))
        flops, a_bytes = encoder_counts(res, res)
        to, tr = min(t_ours), min(t_ref)
        row = {"resolution": res, "batch": B, "img_per_s": round(B / to, 2), "ms_per_call": round(to * 1e3, 3),
               "ms_per_call_all_windows": [round(t * 1e3, 3) for t in t_ours],
               "tflop_per_image": round(flops / 1e12, 4), "achieved_tflops": round(flops * B / to / 1e12, 1),
               "im2col_operand_bytes_per_image": a_bytes, "launches_per_call": launches,
               "peak_memory_gb": round(peak / 1e9, 2),
               "cudnn_bf16_autocast": {"img_per_s": round(B / tr, 2), "ms_per_call": round(tr * 1e3, 3),
                                       "ms_per_call_all_windows": [round(t * 1e3, 3) for t in t_ref],
                                       "achieved_tflops": round(flops * B / tr / 1e12, 1)},
               "speedup_vs_cudnn": round(tr / to, 3), "rel_l2_ours_vs_cudnn_bf16": agree}
        row["kernel_split"] = kernel_split(ours)
        result["sizes"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del x, xc
        torch.cuda.empty_cache()
    result["card_after"] = card()
    result["time"] = time.strftime("%Y-%m-%d %H:%M:%S")
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
