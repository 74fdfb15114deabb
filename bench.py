#!/usr/bin/env python
"""Benchmark of the MaskDiT hot path on B200 (contract: see the task statement; one JSON line on rank 0).

  python bench.py --gpus N --steps K --warmup W                 # B200 arm: MaskDiT-XL/2 ImageNet-256 train step
  python bench.py --impl reference --gpus N --steps K --warmup W  # reference arm: the CPU path of the same workload
  python bench.py --workload sampler                            # EDM sampler, 18 steps, CFG 1.5, batch 64
  python bench.py ... --dump-outputs DIR                        # + what the last timed step computed, as DIR/*.npy

A "step" = EDMLoss forward + hand-written backward + (N>1: one NCCL all-reduce of the flat fp32 gradient) +
fused AdamW + EMA, on synthetic latents of BASELINE.json's shape with random-init XL/2 weights (the reference's
zero-initialised tensors are randomised, SURVEY.md §3.3 — otherwise the net is the identity).  For the sampler
workload a "step" is one whole 18-step sampler run.
`value`  : samples/s, inputs resident in HBM.      `e2e.value`: same, inputs copied from pinned host memory
every step and the loss read back to the host every step.

Weights, inputs and the step's random draws are seeded, so the same arguments give the same inputs in every run and
`--dump-outputs` of two builds can be compared array for array (up to floating-point summation order).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_SAMPLE = {256: 392.72e9, 512: 1680.98e9}   # SURVEY.md §8(d): 3 x forward matmul FLOPs, no recompute
SAMPLER_FLOP_PER_IMAGE = 17.608e12                   # 251.55 GF x 2 (CFG) x 35 evals


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return dict(burst=p["bf16_tflops"], sustained=p["bf16_tflops_sustained"], hbm=p["hbm_gbs"], src="measured")
    except Exception:
        return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (profiling guide's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.path = gpu_index, None, f"/tmp/mdt_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1])), mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def randomise_zero_init(net, seed=1):
    """SURVEY §8(d): overwrite the adaLN-Zero / zero-init tensors with N(0, 0.02) so every block is active."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for k, p in net.named_parameters():
            if p.requires_grad and float(p.abs().sum()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)


DUMP_SAMPLE = 1 << 20   # elements drawn from each parameter-sized output: 4 MB per array in float32


def sampled(named, n=DUMP_SAMPLE, seed=0):
    """A fixed, seeded sample of n elements (with replacement, in index order) of the concatenation of the tensors in
    `named` (registration order of the module, so the sample does not depend on how the library lays them out)."""
    sizes = torch.tensor([t.numel() for _, t in named])
    ends = sizes.cumsum(0)
    idx = torch.randint(0, int(ends[-1]), (n,), generator=torch.Generator().manual_seed(seed)).sort().values
    owner = torch.searchsorted(ends, idx, right=True)
    parts = []
    for j, (_, t) in enumerate(named):
        local = idx[owner == j] - (ends[j] - sizes[j])
        if len(local):
            parts.append(t.detach().reshape(-1)[local.to(t.device)].float().cpu())
    return torch.cat(parts).numpy()


def write_outputs(d, arrays):
    """DIR/<name>.npy for every array (float32 / float64 only)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(d, name + ".npy"), a)


def make_batches(n, B, R, ncls, seed=0):
    """Synthetic latents ~ N(0, sigma_data^2) and one-hot labels with 10 % dropped rows (train.py:209), pinned."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        x = (torch.randn(B, 4, R, R, generator=g) * 0.5).pin_memory()
        y = torch.nn.functional.one_hot(torch.randint(0, ncls, (B,), generator=g), ncls).float()
        y = (y * (torch.rand(B, 1, generator=g) >= 0.1)).pin_memory()
        out.append((x, y))
    return out


# ---------------------------------------------------------------------------------------------------------------
def pin_to_one_socket():
    """CPU baseline stability (VERDICT r1: the CPU arm moved 13x between runs): bind this process to the physical cores
    of socket 0 (one hardware thread per core) and size torch's pool to match.  Returns (threads, description)."""
    try:
        cores = {}
        for c in sorted(os.sched_getaffinity(0)):
            base = f"/sys/devices/system/cpu/cpu{c}/topology/"
            pkg = int(open(base + "physical_package_id").read())
            core = int(open(base + "core_id").read())
            cores.setdefault(pkg, {}).setdefault(core, c)     # first hardware thread of every physical core
        pkg0 = min(cores)
        cpus = sorted(cores[pkg0].values())
        os.sched_setaffinity(0, cpus)
        torch.set_num_threads(len(cpus))
        return len(cpus), f"pinned to the {len(cpus)} physical cores of socket {pkg0} (of {len(cores)} sockets)"
    except Exception as e:  # no sysfs topology: leave the affinity alone
        return torch.get_num_threads(), f"unpinned ({type(e).__name__})"


def cpu_reference_train(B, steps, warmup, R=32):
    """The reference's algorithm on the host CPU (oracle port, fp32, AdamW(wd=0)): samples/s.  Checker code timed as a
    BASELINE only — never on the product path.  SURVEY 8(d): full train step at B=8, 1 warm-up + 3 timed."""
    from oracle import maskdit_oracle as O
    cfg = O.Cfg(model_type="DiT-XL/2", img_resolution=R, num_classes=1000)
    sd = {k: v.requires_grad_(not k.endswith("pos_embed")) for k, v in O.make_state_dict(cfg, 1).items()}
    m = {k: torch.zeros_like(v) for k, v in sd.items() if v.requires_grad}
    v2 = {k: torch.zeros_like(v) for k, v in sd.items() if v.requires_grad}
    g = torch.Generator().manual_seed(0)
    times = []
    for it in range(warmup + steps):
        x = torch.randn(B, 4, R, R, generator=g) * 0.5
        y = torch.nn.functional.one_hot(torch.randint(0, 1000, (B,), generator=g), 1000).float()
        t0 = time.perf_counter()
        md = O.mask_from_noise(torch.rand(B, cfg.num_patches, generator=g), 0.5)
        loss, _ = O.edm_loss(sd, cfg, x, y, torch.randn(B, 1, 1, 1, generator=g), torch.randn(x.shape, generator=g),
                             md, 0.1)
        loss.mean().backward()
        with torch.no_grad():
            for k in m:
                O.adamw_ema_step(sd[k], sd[k].grad, m[k], v2[k], None, it + 1)
                sd[k].grad = None
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return B * len(times) / sum(times), sum(times)


def cpu_reference_eval(R=32):
    """SURVEY 8(d) (i) config 1: XL/2 masked forward at B=2, fp32; (iii) sampler at B=2, CFG 1.5: three network
    evaluations are timed and scaled to the 35 of an 18-step run (the sampler is 35 identical evaluations + axpys)."""
    from oracle import maskdit_oracle as O
    cfg = O.Cfg(model_type="DiT-XL/2", img_resolution=R, num_classes=1000)
    sd = O.make_state_dict(cfg, 1)
    g = torch.Generator().manual_seed(0)
    B = 2
    x = torch.randn(B, 4, R, R, generator=g) * 0.5
    y = torch.nn.functional.one_hot(torch.randint(0, 1000, (B,), generator=g), 1000).float()
    md = O.mask_from_noise(torch.rand(B, cfg.num_patches, generator=g), 0.5)
    with torch.no_grad():
        O.edm_loss(sd, cfg, x, y, torch.randn(B, 1, 1, 1, generator=g), torch.randn(x.shape, generator=g), md, 0.1)
        t0 = time.perf_counter()
        for _ in range(2):
            O.edm_loss(sd, cfg, x, y, torch.randn(B, 1, 1, 1, generator=g), torch.randn(x.shape, generator=g), md, 0.1)
        fwd = 2 * B / (time.perf_counter() - t0)
        t0 = time.perf_counter()
        for s_ in (80.0, 10.0, 0.5):
            O.edm_precond(sd, cfg, x, torch.tensor(s_, dtype=torch.float64), y, cfg_scale=1.5, training=False)
        per_eval = (time.perf_counter() - t0) / 3
    return fwd, B / (35 * per_eval)


REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def have_unmodified_reference():
    return os.path.exists(os.path.join(REF_DIR, "models", "maskdit.py"))


def cpu_reference_train_unmodified(B, steps, warmup, R=32):
    """The UNMODIFIED reference (`models/maskdit.py` + `train_utils/loss.py`, staged from `MDT_REFERENCE_DIR` into the
    git-ignored baseline/_ref/ by `__graft_entry__.build()`), imported through the timm stand-in, fp32, PyTorch CPU backend,
    `torch.optim.AdamW(weight_decay=0)` in place of apex FusedAdam, the net wrapped to expose `.module` as the loss
    expects (loss.py:47) - BASELINE.md section 3.  Zero-initialised tensors randomised N(0, 0.02) like the GPU run."""
    from oracle import timm_standin
    timm_standin.install()
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import models.maskdit as rm
    import train_utils.loss as rl
    torch.manual_seed(0)
    net = rm.Precond_models["edm"](img_resolution=R, img_channels=4, num_classes=1000, model_type="DiT-XL/2",
                                   use_decoder=True, mae_loss_coef=0.1, pad_cls_token=False).train()
    randomise_zero_init(net)

    class Wrap:
        def __init__(self, m):
            self.module, self.model, self.training = m, m.model, True

        def __call__(self, *a, **k):
            return self.module(*a, **k)

    wrap, loss_fn = Wrap(net), rl.Losses["edm"]()
    opt = torch.optim.AdamW([p for p in net.parameters() if p.requires_grad], lr=1e-4, weight_decay=0)
    g = torch.Generator().manual_seed(0)
    times = []
    for it in range(warmup + steps):
        x = torch.randn(B, 4, R, R, generator=g) * 0.5
        y = torch.nn.functional.one_hot(torch.randint(0, 1000, (B,), generator=g), 1000).float()
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = loss_fn(net=wrap, images=x, labels=y, mask_ratio=0.5, mae_loss_coef=0.1)
        loss.mean().backward()
        opt.step()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return B * len(times) / sum(times), sum(times)


def cpu_baseline_record(steps, warmup, R=32, B=8, extras=False, prefer_unmodified=False):
    threads, how = pin_to_one_socket()
    if prefer_unmodified and have_unmodified_reference():
        sps, secs = cpu_reference_train_unmodified(B, steps, warmup, R=R)
        extra = {}
        if extras:
            fwd, ips = cpu_reference_eval(R)
            extra = {"c1_forward_b2": {"value": fwd, "unit": "samples/s", "kind": "port"},
                     "c5_sampler_b2_scaled": {"value": ips, "unit": "img/s", "kind": "port",
                                              "how": "3 CFG network evaluations at B=2 timed, scaled to the 35 of an 18-step run"}}
        return sps, secs, {**extra, "value": sps, "unit": "samples/s", "cores": threads, "kind": "reference", "same_config": False,
                           "sample": f"{steps} timed steps (+{warmup} warm-up) of batch {B} (SURVEY 8d): the UNMODIFIED "
                                     f"reference modules (models/maskdit.py + train_utils/loss.py staged in baseline/_ref, "
                                     f"timm stand-in), EDM loss fwd + bwd + torch AdamW(wd=0), torch CPU fp32, {threads} "
                                     f"threads {how}; host has {os.cpu_count()} logical CPUs; {secs:.1f} s timed"}
    sps, secs = cpu_reference_train(B, steps, warmup, R=R)
    extra = {}
    if extras:
        fwd, ips = cpu_reference_eval(R)
        extra = {"c1_forward_b2": {"value": fwd, "unit": "samples/s"},
                 "c5_sampler_b2_scaled": {"value": ips, "unit": "img/s",
                                          "how": "3 CFG network evaluations at B=2 timed, scaled to the 35 of an 18-step run"}}
    return sps, secs, {**extra, "value": sps, "unit": "samples/s", "cores": threads, "kind": "port", "same_config": False,
                       "sample": f"{steps} timed steps (+{warmup} warm-up) of batch {B} (SURVEY 8d), EDM loss fwd + bwd + "
                                 f"AdamW, torch CPU fp32, {threads} threads {how}; host has {os.cpu_count()} logical "
                                 f"CPUs; {secs:.1f} s timed.  No unmodified reference staged in baseline/_ref: the "
                                 "oracle port (pinned to the unmodified reference by tests/golden) is what runs"}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    R = 64 if args.workload == "train512" else 32
    B = 8 if R == 32 else 2
    sps, secs, rec = cpu_baseline_record(args.steps, max(1, min(args.warmup, 2)), R=R, B=B, prefer_unmodified=True)
    line = {"impl": "reference", "metric": "train_samples_per_sec", "value": sps, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"MaskDiT-XL/2 ImageNet-{256 if R == 32 else 512} train step ({R}x{R}x4 latents, "
                                   "mask 0.5) on host CPU", "batch_per_step": B, "same_config": False},
            "cpu_baseline": rec,
            "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def gemm_traffic():
    """DRAM read+write bytes per GEMM launch from the committed `ncu --set full` capture (never a constant in code)."""
    for name in ("r02_gemm_ncu_full_v2.json", "r02_gemm_ncu_full.json", "r01_gemm_ncu_full_v3.json"):
        f = os.path.join(ROOT, "profiles", name)
        try:
            d = json.load(open(f))
            rows = d["launches"] if isinstance(d, dict) else d
            vals = [r["dram_bytes"] if "dram_bytes" in r else 1e6 * (r["dram_read_MB"] + r["dram_write_MB"])
                    for r in rows if "dram_bytes" in r or "dram_read_MB" in r]
            if vals:
                return sum(vals) / len(vals), f"profiles/{name} (mean of {len(vals)} launches inside a step)"
        except Exception:
            continue
    return None, "no ncu --set full capture found under profiles/"


# ---------------------------------------------------------------------------------------------------------------
def build_xl2(R, dev):
    from maskdit_b200.maskdit import Precond_models
    torch.manual_seed(0)
    net = Precond_models["edm"](img_resolution=R, img_channels=4, num_classes=1000, model_type="DiT-XL/2",
                                use_decoder=True, mae_loss_coef=0.1, pad_cls_token=False)
    randomise_zero_init(net)
    return net.to(dev)


class Env:
    def __init__(self, dev, world, rank):
        self.dev, self.world, self.rank = dev, world, rank

    def sync_all(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world == 1:
            return ms
        import torch.distributed as dist
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, K):
        """K calls of fn bracketed by barrier + synchronize on both sides, CUDA events on the launching stream, max
        over ranks (ms)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.sync_all()
        e0.record()
        for i in range(K):
            fn(i)
        e1.record()
        self.sync_all()
        return self.max_over_ranks(e0.elapsed_time(e1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="train256", choices=["train256", "train512", "sampler"])
    ap.add_argument("--batch-per-gpu", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true",
                    help="skip the sub-records (BASELINE configs 3-5: 128/GPU, 64x64x4 latents, sampler)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step of the headline workload computed "
                         "as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"

    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    PK = peaks()
    env = Env(dev, world, rank)

    R = 64 if args.workload == "train512" else 32
    net = build_xl2(R, dev)
    if args.workload == "sampler":
        line = bench_sampler(args, net, env, PK, dump=args.dump_outputs)
    else:
        line = bench_train(args, net, env, R, PK, args.batch_per_gpu or (256 if R == 32 else 128), args.steps,
                           args.warmup, full=True, dump=args.dump_outputs)
        if args.workload == "train256" and not args.no_sub and args.batch_per_gpu is None:
            # BASELINE.json configs 3, 4, 5 next to the headline (config 2), same process, same box, same clocks
            # (a sub-record that fails - symmetrically on every rank, e.g. out of memory - must not cost the headline)
            sub = {}

            def guarded(name, fn):
                try:
                    sub[name] = fn()
                except Exception as e:  # noqa: BLE001
                    sub[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
                    torch.cuda.empty_cache()

            guarded("c3_global1024_at_8gpu",
                    lambda: bench_train(args, net, env, 32, PK, 128, max(5, args.steps // 2), 3, full=False))
            guarded("c5_sampler", lambda: bench_sampler(args, net, env, PK, iters=2, warm=1))
            del net
            torch.cuda.empty_cache()

            def c4():
                net64 = None
                try:
                    net64 = build_xl2(64, dev)
                    return bench_train(args, net64, env, 64, PK, 128, max(4, args.steps // 4), 3, full=False)
                finally:
                    net64 = None
                    torch.cuda.empty_cache()

            guarded("c4_512px", c4)
            line["sub"] = sub
        if world > 1 and not args.no_sub and args.workload == "train256" and args.batch_per_gpu is None:
            # the same step with the fp32 gradient exchange (DDP's arithmetic) next to the default bf16 exchange buffer
            os.environ["MDT_GRAD_AR"] = "fp32"
            try:
                net2 = build_xl2(32, dev)
                line.setdefault("sub", {})["c2_fp32_grad_exchange"] = bench_train(args, net2, env, 32, PK, 256,
                                                                               max(5, args.steps // 2), 3, full=False)
                del net2
            except Exception as e:  # noqa: BLE001
                line.setdefault("sub", {})["c2_fp32_grad_exchange"] = {"error": f"{type(e).__name__}: {e}"[:300]}
            del os.environ["MDT_GRAD_AR"]
            torch.cuda.empty_cache()
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            _, _, line["cpu_baseline"] = cpu_baseline_record(3, 1, R=R, B=8 if R == 32 else 2, extras=(R == 32),
                                                             prefer_unmodified=True)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_train(args, net, env, R, PK, B, steps, warmup, full, dump=None):
    """One training-step measurement.  full=True: the headline record (resident + e2e + per-launch GEMM timing +
    clocks); full=False: a compact sub-record (resident inputs only).  dump: directory that receives what the last
    timed (resident) step returned to its caller - the per-sample loss and the updated weights, EMA weights and
    gradients (a seeded sample of each) - taken before any later step changes them."""
    import copy

    from maskdit_b200 import _lib
    from maskdit_b200.train_step import TrainStep
    dev, world, rank = env.dev, env.world, env.rank
    net.train()
    ema = copy.deepcopy(net).eval()
    ts = TrainStep(net, ema, lr=1e-4, global_batch=B * world, overlap=os.environ.get("MDT_OVERLAP", "0") == "1")
    pool = make_batches(4, B, R, 1000, seed=rank)
    resident = [(x.to(dev), y.to(dev)) for x, y in pool]
    h2d = pool[0][0].numel() * 4 + pool[0][1].numel() * 4
    loss_host = torch.zeros(1).pin_memory()
    last = {}

    def step_resident(i):
        x, y = resident[i % len(resident)]
        last["loss"] = ts.step(x, y, 0.5, 0.1)

    def step_e2e(i):
        xh, yh = pool[i % len(pool)]
        x, y = xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True)
        loss = ts.step(x, y, 0.5, 0.1)
        loss_host.copy_(loss.mean().reshape(1), non_blocking=True)   # D2H read of the step's result

    for i in range(warmup):
        step_resident(i)
    clocks = ClockSampler(torch.cuda.current_device())
    if rank == 0 and full:
        clocks.start()
    n0 = _lib.LAUNCHES
    ms = env.timed(step_resident, steps)
    launches = _lib.LAUNCHES - n0
    clk = clocks.stop() if (rank == 0 and full) else None
    if dump and rank == 0:
        trainable = [(k, p) for k, p in net.named_parameters() if p.requires_grad]
        write_outputs(dump, {
            "loss": last["loss"].float().cpu().numpy(),
            "weights_sample": sampled(trainable),
            "ema_weights_sample": sampled([(k, p) for k, p in ema.named_parameters() if p.requires_grad]),
            "grads_sample": sampled([(k, p.grad) for k, p in trainable])})
    ms_step = ms / steps
    sps = B * world * steps / (ms / 1e3)
    flop = FLOP_PER_SAMPLE[256 if R == 32 else 512]
    step_tf = sps / world * flop / 1e12
    workload = (f"MaskDiT-XL/2 ImageNet-{256 if R == 32 else 512} training step ({R}x{R}x4 latents, bf16 GEMM operands / "
                f"fp32 accumulate+residual, mask_ratio 0.5, EDM+MAE loss, AdamW+EMA)")
    if not full:
        rec = {"metric": "train_samples_per_sec", "value": sps, "unit": "samples/s", "n_gpus": world, "steps": steps,
               "warmup": warmup, "ms_per_step": ms_step, "gpu_launches": launches,
               "config": {"workload": workload, "batch_per_gpu": B, "global_batch": B * world,
                          "grad_allreduce": ts.describe_collective()},
               "roofline": {"bound": "tensor", "step_achieved": step_tf, "peak": PK["sustained"], "unit": "TFLOP/s",
                            "step_frac": step_tf / PK["sustained"], "peak_source": f"{PK['src']} sustained bf16"}}
        ts.close()
        del ts, ema, resident
        torch.cuda.empty_cache()
        return rec
    for i in range(2):
        step_e2e(i)
    ms_e2e = env.timed(step_e2e, steps)
    final_loss = float(loss_host.item())

    # dominant kernel (the tcgen05 GEMM family) timed per launch with CUDA events inside real steps: the library brackets
    # every mdt_gemm_bf16 launch - the C++ step driver's own - with an event pair on the launching stream
    # (mdt_gemm_profile_enable); three steps, per launch the median of the three.
    import ctypes
    L = _lib.lib()
    runs = []
    for i in range(3):
        L.mdt_gemm_profile_enable(1)
        step_resident(i)
        torch.cuda.synchronize()
        L.mdt_gemm_profile_enable(0)
        n = L.mdt_gemm_profile_read(None, None, 0)
        ms_buf, fl_buf = (ctypes.c_float * n)(), (ctypes.c_double * n)()
        assert L.mdt_gemm_profile_read(ms_buf, fl_buf, n) == n
        runs.append(list(zip(list(fl_buf), list(ms_buf))))
    prof = runs[0]
    assert all(len(r) == len(prof) for r in runs)
    gemm_ms = sum(sorted(r[j][1] for r in runs)[1] for j in range(len(prof)))
    gemm_flops = sum(f for f, _ in prof)
    sps_e2e = B * world * steps / (ms_e2e / 1e3)
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, traffic_src = gemm_traffic() if (R == 32 and B == 256) else (None, "no capture for this configuration")
    line = {
        "metric": "train_samples_per_sec", "value": sps, "unit": "samples/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload, "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                   "grad_allreduce": ts.describe_collective(),
                   "l2_policy": "per-step working set (activations > 40 GB) far exceeds the 126 MB L2; no flush needed",
                   "final_loss": final_loss},
        "clocks": clk,
        "e2e": {"value": sps_e2e, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all GEMM launches of one step)",
                     "achieved": achieved, "peak": PK["sustained"], "unit": "TFLOP/s",
                     "frac": achieved / PK["sustained"], "peak_source": f"{PK['src']} sustained bf16",
                     "traffic": traffic, "traffic_source": traffic_src,
                     "launches_per_step": len(prof), "share_of_step": gemm_ms / ms_step,
                     "step_achieved": step_tf, "step_frac": step_tf / PK["sustained"]},
    }
    ts.close()
    del ts, ema, resident
    torch.cuda.empty_cache()
    return line


def bench_sampler(args, net, env, PK, iters=None, warm=None, dump=None):
    """`iters` sampler runs timed (default: --steps); dump: directory that receives the final latents of the last one."""
    from maskdit_b200 import _lib
    from maskdit_b200.sampler import edm_sampler
    dev, world, rank = env.dev, env.world, env.rank
    B = (args.batch_per_gpu if args.workload == "sampler" else None) or 64
    net.eval()
    g = torch.Generator().manual_seed(rank)
    lat_h = torch.randn(B, 4, 32, 32, generator=g).pin_memory()
    lab_h = torch.nn.functional.one_hot(torch.randint(0, 1000, (B,), generator=g), 1000).float().pin_memory()
    out_h = torch.zeros(B, 4, 32, 32, dtype=torch.float64).pin_memory()

    def run(i):
        with torch.no_grad():
            z = edm_sampler(net, lat_h.to(dev, non_blocking=True), lab_h.to(dev, non_blocking=True), cfg_scale=1.5,
                            num_steps=18)
            out_h.copy_(z, non_blocking=True)

    W = warm if warm is not None else max(1, args.warmup // 3)
    for i in range(W):
        run(i)
    K = iters if iters is not None else args.steps
    clocks = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        clocks.start()
    n0 = _lib.LAUNCHES
    ms = env.timed(run, K)
    if dump and rank == 0:
        write_outputs(dump, {"latents": out_h.numpy()})
    ips = B * world * K / (ms / 1e3)
    ach = ips / world * SAMPLER_FLOP_PER_IMAGE / 1e12
    return {"metric": "edm_sampler_imgs_per_sec", "value": ips, "unit": "img/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "EDM sampler 18 steps (35 net evals), CFG 1.5, 32x32x4 latents, MaskDiT-XL/2",
                       "batch_per_gpu": B, "parallelism": f"replicas x{world}"},
            "clocks": clocks.stop() if rank == 0 else None,
            "e2e": {"value": ips, "unit": "img/s", "h2d_bytes_per_step": lat_h.numel() * 4 + lab_h.numel() * 4,
                    "d2h_bytes_per_step": out_h.numel() * 8},
            "gpu_launches": _lib.LAUNCHES - n0,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": PK["sustained"], "unit": "TFLOP/s",
                         "frac": ach / PK["sustained"], "peak_source": f"{PK['src']} sustained bf16",
                         "traffic": None}}


if __name__ == "__main__":
    main()
