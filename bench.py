#!/usr/bin/env python
"""Benchmark of the hot path: images/sec of the full training step (BASELINE.json `metric`).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K ...   # the reference arithmetic on the box's host cores
    python bench.py ... --dump-outputs DIR                    # + what the last timed step returned, as DIR/*.npy

--steps K is the number of timed steps of each GPU-timed loop (device-resident, end to end, eager peer). The inputs
(seeded weights, synthetic batches, host random stream) are the same on every run with the same arguments, so the
dumped outputs of two builds can be compared array for array.

Workload (BASELINE.json configs[1]): FLUX-VAE config ch=128, ch_mult=1,2,4,4, z=16, 256x256 synthetic images,
one step = Encoder -> clamp -> reg -> Decoder -> GradNorm -> LPIPS(eval) + 0.1*mean(z^2) (+ pooled L1 at the reference's
HEAD weight 0.0) -> backward -> gradient all-reduce -> AdamW (vae_trainer.py:530-708), bf16 storage / fp32 accumulate.
One process per GPU (torchrun for N > 1), weak scaling: per-GPU batch fixed.

Printed JSON (one line, rank 0): see the contract in the task statement. `value` = device-resident inputs, CUDA-event
timed, max over ranks; `e2e` = the same step through the public Trainer API with pinned host batches (H2D inside the timed
region) and a device->host read of the loss every step; `roofline` = achieved tensor throughput of the dominant kernel
(vqb::conv_gemm_kernel, fwd + dgrad launches) from CUDA events around every launch of an extra profiled step;
`cpu_baseline` = the CPU oracle (port of the reference arithmetic) on this box's host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "vqgan-training_b200")
sys.path.insert(0, PKG)
sys.path.insert(1, ROOT)
os.environ.setdefault("VQB_OFFLINE", "1")
os.environ.setdefault("WANDB_MODE", "disabled")

import warnings

warnings.simplefilter("ignore")

import torch
import torch.distributed as dist

CFG = dict(vae_ch=128, vae_ch_mult="1,2,4,4", vae_z_channels=16, vae_num_res_blocks=2, resolution=256)
# BASELINE.json configs[1..4] -> bench modes. tflop = algorithmic conv FLOPs per image of one training step
# (SURVEY.md §8a / BASELINE.md §3: fwd + dgrad + wgrad of the VAE, 2 LPIPS VGG forwards + 1 dgrad, + D passes).
CONFIGS = {
    "lpips": dict(idx=1, tflop=2.780, gan=False, vq=False, hr=False, res=256, batch=32,
                  what="Encoder->clamp->Decoder->GradNorm->LPIPS(eval)+0.1*mean(z^2)"),
    "gan": dict(idx=2, tflop=3.107, gan=True, vq=False, hr=False, res=256, batch=32,
                what="Encoder->clamp->Decoder->GradNorm->LPIPS(eval)+0.1*mean(z^2)+PatchD hinge+LeCam (D step every step)"),
    "vq": dict(idx=3, tflop=3.107, gan=True, vq=True, hr=False, res=256, batch=32,
               what="Encoder->clamp->VQ(8192x16 argmin+commitment)->Decoder->GradNorm->LPIPS(eval)+PatchD hinge+LeCam"),
    "hr512": dict(idx=4, tflop=9.98, gan=True, vq=False, hr=True, res=512, batch=8,
                  what="Encoder@256^2->clamp->HR Decoder->512^2->GradNorm->LPIPS(eval)@512^2+PatchD hinge+LeCam@512^2"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
    return 1400.0, "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_threads():
    """Threads for the CPU arm: every core up to 32 (batch-1 convolutions of this size stop scaling — and with 100+
    threads get slower — beyond that; measured 0.007 img/s at 128 threads vs 0.12 img/s at 8 on the survey box)."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("VQB_CPU_THREADS", "32"))))


def cpu_step_runner(batch=1, threads=None):
    """The reference arithmetic on host cores: oracle restatement (fp32, torch CPU) of one training step incl. AdamW."""
    from oracle import lpips_oracle as LP
    from oracle import seeded
    from oracle import step_oracle as SO
    from oracle import vae_oracle as VO

    if threads:
        torch.set_num_threads(threads)
    cfg = VO.VAEConfig(resolution=256, ch=128, ch_mult=(1, 2, 4, 4), num_res_blocks=2, z_channels=16)
    g = torch.Generator().manual_seed(42)
    vsd = {}
    for k, shp in VO.state_dict_shapes(cfg).items():
        fan = max(1, int(torch.tensor(shp[1:]).prod())) if len(shp) == 4 else 1
        if len(shp) == 4:
            v = torch.randn(shp, generator=g) * (1.0 / fan) ** 0.5
        elif k.endswith("weight"):
            v = torch.ones(shp)
        else:
            v = torch.zeros(shp)
        vsd[k] = v.requires_grad_(True)
    lsd = {}
    for k, shp in LP.lpips_state_dict_shapes().items():
        if "scaling" in k:
            continue
        fan = max(1, int(torch.tensor(shp[1:]).prod())) if len(shp) == 4 else 1
        lsd[k] = (torch.randn(shp, generator=g) * (2.0 / fan) ** 0.5) if len(shp) == 4 and "lin" not in k else \
            (torch.rand(shp, generator=g) / fan if len(shp) == 4 else torch.zeros(shp))
    opt = torch.optim.AdamW([p for p in vsd.values()], lr=1e-5 / 128, weight_decay=1e-3, betas=(0.9, 0.95))
    real = torch.rand(batch, 3, 256, 256, generator=g) * 2 - 1

    def step():
        opt.zero_grad(set_to_none=True)
        SO.generator_step(vsd, lsd, None, real, cfg, do_clamp=True, do_ganloss=False)
        opt.step()

    return step, batch


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU arithmetic (oracle port; the Python reference tree itself cannot travel to
    the GPU box) on this box's host cores, same metric/unit/config. Rank 0 only."""
    if rank != 0:
        return
    threads = cpu_threads()
    step, b = cpu_step_runner(batch=1, threads=threads)
    t0 = time.perf_counter()
    step()  # first warm-up step (also tells us how long one step takes on this host)
    first = time.perf_counter() - t0
    # honour --steps / --warmup as long as the whole arm stays within ~3 minutes of CPU time (a step is ~3-9 s on the
    # pool's hosts); otherwise a bounded sample, stated in `cpu_baseline.sample`
    budget = 170.0
    w = max(1, min(args.warmup, int(30.0 / max(first, 1e-3)) or 1))
    for _ in range(w - 1):
        step()
    k = max(1, min(args.steps, int((budget - w * first) / max(first, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(k):
        step()
    dt = (time.perf_counter() - t0) / k
    val = b / dt
    line = {"metric": "images/sec", "value": val, "unit": "images/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": k, "warmup": w, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "FLUX-VAE ch=128 mult 1,2,4,4 z=16 256x256 train step (VAE+LPIPS+z-loss+AdamW)",
                       "per_gpu_batch": b, "note": "CPU oracle port of the reference arithmetic, batch 1 per step"},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": threads, "kind": "port",
                             "sample": f"{k} timed training steps at batch 1 (fwd+bwd+AdamW), torch CPU fp32"},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit_json(line)


def profile_conv_kernels(tr, batch_dev):
    """One extra (untimed) step with CUDA events around every conv_gemm / wgrad_gemm launch on the launching stream."""
    import ops

    rec = {"conv": [], "wgrad": []}
    orig_conv, orig_wgrad = ops.run_conv_gemm, ops.run_wgrad

    def is_fat(g):  # fat-pixel first/last layer: 64-wide K runs carrying 3 real taps x 8 channels (3 real) each
        return g.C == 64 and len(g.taps) == 3 and len(g.views) == 1 and g.views[0].sw == 8

    def flops_conv(g, Cout):
        if is_fat(g):
            return 2.0 * g.N * g.Ho * g.Wo * Cout * 27
        return 2.0 * g.N * g.Ho * g.Wo * Cout * g.C * len(g.taps)

    def conv_wrap(g, a, wp, Cout, out, out_strides, *aa, **kk):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig_conv(g, a, wp, Cout, out, out_strides, *aa, **kk)
        e1.record()
        sig = ("conv", g.N, g.Ho, g.Wo, g.C, Cout, len(g.taps), len(g.views))
        if os.environ.get("VQB_KERNEL_TABLE", "0") == "2":  # split rows by epilogue variant
            sig += ("".join(c for c, k in (("b", "bias"), ("r", "res"), ("m", "mask"), ("s", "stats"))
                            if kk.get(k) is not None) + ("R" if kk.get("relu") else ""),)
        rec["conv"].append((e0, e1, flops_conv(g, Cout), sig))
        return r

    def wgrad_wrap(g, x, dy, weight_shape, Cout_pad, **kk):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig_wgrad(g, x, dy, weight_shape, Cout_pad, **kk)
        e1.record()
        Cout, Cin, KH, KW = weight_shape
        if is_fat(g):  # 3 real channels x 9 taps, not the padded 64 x 3
            Cin, KH, KW = 3, 3, 3
        rec["wgrad"].append((e0, e1, 2.0 * g.N * g.Ho * g.Wo * Cout * Cin * KH * KW,
                             ("wgrad", g.N, g.Ho, g.Wo, g.C, Cout, len(g.taps), len(g.views))))
        return r

    ops.run_conv_gemm, ops.run_wgrad = conv_wrap, wgrad_wrap
    try:
        tr.step(batch_dev)
        torch.cuda.synchronize()
    finally:
        ops.run_conv_gemm, ops.run_wgrad = orig_conv, orig_wgrad
    out = {}
    table = {}
    for k, lst in rec.items():
        for e0, e1, f, sig in lst:
            t = table.setdefault(sig, [0, 0.0, 0.0])
            t[0] += 1
            t[1] += e0.elapsed_time(e1)
            t[2] += f
    if os.environ.get("VQB_KERNEL_TABLE", "0") in ("1", "2"):
        sys.stderr.write("kind N Ho Wo C Cout taps views | launches total_ms TFLOP/s\n")
        for sig, (cnt, ms_, fl_) in sorted(table.items(), key=lambda kv: -kv[1][1]):
            sys.stderr.write(f"{sig} | {cnt} {ms_:.3f} {fl_ / (ms_ * 1e-3) / 1e12 if ms_ > 0 else 0:.1f}\n")
    for k, lst in rec.items():
        ms = sum(e0.elapsed_time(e1) for e0, e1, _, _ in lst)
        fl = sum(f for _, _, f, _ in lst)
        out[k] = {"launches": len(lst), "ms": ms, "tflops": fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0,
                  "flops_per_launch": fl / max(1, len(lst)), "ms_per_launch": ms / max(1, len(lst))}
    return out


DUMP_BYTES = 64_000_000


def host_outputs(out, prefix=""):
    """What Trainer.step returned, flattened to {name: float32/float64 numpy array} on the host (nested dicts become
    `outer.inner`). Copy before the next step: a CUDA-graph replay reuses the same output buffers."""
    import numpy as np

    arrs = {}
    for k, v in out.items():
        name = prefix + k
        if isinstance(v, dict):
            arrs.update(host_outputs(v, name + "."))
        elif torch.is_tensor(v):
            v = v.detach()
            arrs[name] = v.cpu().numpy() if v.dtype == torch.float64 else v.float().cpu().numpy()
        else:
            arrs[name] = np.asarray(v, dtype=np.float64)
    return arrs


def dump_outputs(arrs, outdir):
    """Writes each array as outdir/<name>.npy, DUMP_BYTES in all (1 KiB per file kept for the .npy header). Smallest
    arrays first, each gets an equal share of what is left; an array larger than its share is replaced by a fixed sample
    of its flattened elements (seed 0, sorted positions), so two runs with the same arguments write comparable files."""
    import numpy as np

    os.makedirs(outdir, exist_ok=True)
    left = DUMP_BYTES - 1024 * len(arrs)
    for i, (name, a) in enumerate(sorted(arrs.items(), key=lambda kv: kv[1].nbytes)):
        keep = max(1, left // (len(arrs) - i) // a.itemsize)
        if a.size > keep:
            idx = np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))
            sys.stderr.write(f"dump-outputs: {name} {a.shape}: fixed sample of {keep} of {a.size} elements\n")
            a = a.reshape(-1)[idx]
        np.save(os.path.join(outdir, name + ".npy"), a)
        left -= a.nbytes


_JSON_OUT = None


def emit_json(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def eager_b200_leg(cfg, B, world, rank, device, steps, warmup):
    """The kernel-for-kernel bar (SURVEY.md §8d "Reference beside it (2)"): the reference's arithmetic executed by stock
    PyTorch eager (cuDNN / ATen) on this same B200, with the reference's own precision mix — TF32 encoder / LPIPS / D
    (vae_trainer.py:18-19), bf16-autocast decoder (:453,623), fp32 GroupNorm — fused AdamW, and the gradient all-reduce
    the reference intends for N > 1. The reference tree is plain Python without packaging (`pip install /root/reference`
    fails: no setup.py / pyproject.toml) and may not be copied, so its modules are represented by the oracle
    restatement (oracle/*.py, pinned to the reference by tests/golden)."""
    from oracle import lpips_oracle as LP
    from oracle import step_oracle as SO
    from oracle import vae_oracle as VO

    vcfg = VO.VAEConfig(resolution=256, ch=128, ch_mult=(1, 2, 4, 4), num_res_blocks=2, z_channels=16,
                        decoder_also_perform_hr=cfg["hr"])
    g = torch.Generator().manual_seed(42)

    def init(shapes, skip=()):
        sd = {}
        for k, shp in shapes.items():
            if any(t in k for t in skip):
                continue
            if len(shp) == 4:
                fan = max(1, shp[1] * shp[2] * shp[3])
                v = (torch.rand(shp, generator=g) / fan) if ("lin" in k) else torch.randn(shp, generator=g) * (2.0 / fan) ** 0.5
            elif k.endswith("weight"):
                v = torch.ones(shp)
            else:
                v = torch.zeros(shp)
            sd[k] = v.to(device)
        return sd

    vsd = {k: v.requires_grad_(True) for k, v in init(VO.state_dict_shapes(vcfg)).items()}
    lsd = init(LP.lpips_state_dict_shapes(), skip=("scaling",))
    dsd = None
    if cfg["gan"]:
        dsd = {k: v.requires_grad_(True) for k, v in init(LP.patchd_state_dict_shapes(), skip=("scaling",)).items()}
    named = list(vsd.items())
    opt_g = torch.optim.AdamW([{"params": [v for k, v in named if "conv_in" not in k], "lr": 1e-5 / 128},
                               {"params": [v for k, v in named if "conv_in" in k], "lr": 1e-4}],
                              weight_decay=1e-3, betas=(0.9, 0.95), fused=True)
    opt_d = torch.optim.AdamW(list(dsd.values()), lr=2e-4, weight_decay=1e-3, betas=(0.9, 0.95), fused=True) if dsd else None
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    R = cfg["res"]

    def allreduce(params):
        if world > 1:
            gs = [p.grad for p in params if p.grad is not None]
            flat = torch.cat([x.reshape(-1) for x in gs])
            dist.all_reduce(flat, op=dist.ReduceOp.AVG)
            torch._foreach_copy_(gs, [v.view_as(x) for v, x in zip(flat.split([x.numel() for x in gs]), gs)])

    def avg_fn(n):
        if world > 1:
            t = torch.tensor(n, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.AVG)
            return t.item()
        return n

    def step(real_hr):
        real_enc = torch.nn.functional.interpolate(real_hr, size=(256, 256), mode="area") if R != 256 else real_hr
        if dsd is not None:  # discriminator pass (vae_trainer.py:629-659) on the detached reconstruction
            with torch.no_grad():
                z = VO.encoder_forward(vsd, real_enc, vcfg).clamp(-8.0, 8.0)
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    rec = VO.decoder_forward(vsd, VO.reg(z), vcfg)
            opt_d.zero_grad(set_to_none=True)
            SO.discriminator_step(dsd, real_hr, rec.float(), "hinge", True, (0.0, 0.0))
            allreduce(list(dsd.values()))
            opt_d.step()
            for v in dsd.values():
                v.requires_grad_(False)
        opt_g.zero_grad(set_to_none=True)
        if R != 256:
            o = _eager_generator_step_hr(SO, VO, LP, vsd, lsd, dsd, real_hr, real_enc, vcfg, avg_fn)
        else:
            o = SO.generator_step(vsd, lsd, dsd, real_hr, vcfg, do_clamp=True, do_ganloss=cfg["gan"], disc_type="hinge",
                                  avg_fn=avg_fn, amp_decoder=True)
        if dsd is not None:
            for v in dsd.values():
                v.requires_grad_(True)
        allreduce([v for _, v in named])
        opt_g.step()
        return o["loss"]

    tried = []
    b = B
    while b >= 1:
        try:
            gen = torch.Generator(device=device).manual_seed(1)
            batches = [torch.rand(b, 3, R, R, device=device, generator=gen) * 2 - 1 for _ in range(2)]
            for i in range(max(2, min(warmup, 3))):
                step(batches[i % 2])
            torch.cuda.synchronize()
            k = steps
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(k):
                loss = step(batches[i % 2])
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / k
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
            return {"value": world * b / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms, "per_gpu_batch": b,
                    "steps": k, "last_loss": float(loss), "tried_batches": tried + [b],
                    "impl": "reference arithmetic (oracle restatement of ae.py/utils.py/vae_trainer.py:530-708) in stock "
                            "PyTorch eager on this GPU: cuDNN convs, TF32 encoder/LPIPS/D, bf16-autocast decoder, fp32 "
                            "GroupNorm, fused AdamW, cudnn.benchmark=True",
                    "peak_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30}
        except torch.OutOfMemoryError:
            tried.append(b)
            if world > 1:
                return {"unavailable": f"eager path out of memory at per-GPU batch {b} (no retry under NCCL)"}
            opt_g.zero_grad(set_to_none=True)
            torch.cuda.empty_cache()
            b //= 2
    return {"unavailable": "eager path out of memory at every batch size", "tried_batches": tried}


def _eager_generator_step_hr(SO, VO, LP, vsd, lsd, dsd, real_hr, real_enc, vcfg, avg_fn):
    """configs[4]: encoder on the 256^2 area-resized image, HR decoder to 512^2, losses against the 512^2 image."""
    from oracle import loss_oracle as LO

    z = VO.encoder_forward(vsd, real_enc, vcfg).clamp(-8.0, 8.0)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        recon = VO.decoder_forward(vsd, VO.reg(z), vcfg)
    percep = LP.lpips_forward(lsd, LO.gradnorm(recon, 1.0, avg_fn), real_hr).mean()
    vae_loss, _ = LO.vae_loss_function(real_hr, LO.gradnorm(recon, 0.001, avg_fn), z, do_pool=True, do_recon=False,
                                       recon_weight=0.0)
    loss = percep + vae_loss
    if dsd is not None:
        loss = loss + LO.gan_gen_loss(LP.patchd_forward(dsd, LO.gradnorm(recon, 1.0, avg_fn)), "hinge")
    loss.backward()
    return {"loss": loss.detach()}


def load_traffic_table():
    """Measured DRAM traffic of the dominant conv shapes (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per
    launch) next to their algorithmic bytes: profiles/r02_ncu_traffic.json when present, else the round-1 capture."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return name, json.load(f)
        except Exception:
            continue
    return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=str, default=os.environ.get("VQB_BENCH_CONFIG", "lpips"), choices=sorted(CONFIGS),
                    help="lpips = BASELINE configs[1] (the metric's config), gan = [2], vq = [3], hr512 = [4]")
    ap.add_argument("--batch", type=int, default=int(os.environ.get("VQB_BENCH_BATCH", "0")), help="per-GPU batch")
    ap.add_argument("--gan", action="store_true", help="alias of --config gan")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the PyTorch-eager-on-B200 peer leg")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of as one CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0, 64 MB at most)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.gan and args.config == "lpips":
        args.config = "gan"
    cfg = CONFIGS[args.config]

    # The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner from C at
    # communicator creation), so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to a
    # private duplicate of the original stdout.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import native
    import vae_trainer as vt

    assert torch.cuda.is_available(), "bench.py needs a CUDA (sm_100a) device: there is no CPU path"
    torch.cuda.set_device(local_rank)
    device = f"cuda:{local_rank}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    W = max(3, args.warmup)
    PREP = 0 if args.no_graph else 5  # 3 eager steps + the CUDA-graph capture + one replay, before the W warm-up steps
    K = args.steps
    B, R = (args.batch or cfg["batch"]), cfg["res"]

    tr = vt.Trainer(device, vae_resolution=256, vae_ch=CFG["vae_ch"], vae_ch_mult=CFG["vae_ch_mult"],
                    vae_num_res_blocks=CFG["vae_num_res_blocks"], vae_z_channels=CFG["vae_z_channels"], do_clamp=True,
                    do_ganloss=cfg["gan"], disc_type="hinge", use_lecam=cfg["gan"], max_steps=100000, lpips_eval=True,
                    use_vq=cfg["vq"], decoder_also_perform_hr=cfg["hr"], cuda_graph=False if args.no_graph else None)
    loader = vt.SyntheticLoader(B, R, seed=42 + rank, n_distinct=4)
    host_batches = loader.batches
    dev_batches = [b.to(device) for b in host_batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- graph preparation (untimed) + warm-up
    for i in range(PREP + W):
        tr.step(dev_batches[i % len(dev_batches)])
    barrier()

    # ---------------- timed: device-resident inputs
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = native.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(K):
        out = tr.step(dev_batches[i % len(dev_batches)])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / K
    launches = (native.launch_count() - l0)
    dumped = host_outputs(out) if args.dump_outputs and rank == 0 else None
    graphed = tr.graph_launches_per_step is not None
    if graphed:  # replays do not pass through the C entry points: kernels per replay (counted at capture) x replays
        launches = tr.graph_launches_per_step * K
    clocks = sampler.stop() if rank == 0 else None

    # ---------------- timed: end to end (pinned host batch -> H2D inside, loss read back every step)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    last_loss = 0.0
    for i in range(K):
        o = tr.step(host_batches[i % len(host_batches)])
        last_loss = float(o["overall_vae_loss"])  # device -> host read of the step's result
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3) / K

    t = torch.tensor([ms, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    # every rank runs the profiled extra step (it contains the NCCL collectives of a normal step); rank 0 reports it.
    # It runs eagerly (per-launch CUDA events need the python wrappers), with the same kernels the graph replays.
    tr._graph_wanted = False
    prof = profile_conv_kernels(tr, dev_batches[0])
    peak_mem = torch.cuda.max_memory_allocated() / 2 ** 30

    # ---------------- the PyTorch-eager-on-B200 peer (same step, same batch, same GPUs), after freeing our own state
    eager = None
    if not args.no_eager:
        tr._graph = None
        del tr, out, o, dev_batches, loader
        import gc

        gc.collect()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        try:
            eager = eager_b200_leg(cfg, B, world, rank, device, K, W)
        except Exception as e:  # the peer must never take the product line down
            eager = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}

    if rank == 0:
        peak, peak_src = load_peaks()
        value = world * B / (ms * 1e-3)
        e2e = world * B / (ms_e2e * 1e-3)
        tname, ttab = load_traffic_table()
        conv_traffic = None
        if ttab is not None:
            conv_traffic = ttab.get("conv_gemm_bytes_per_launch", ttab.get("conv_gemm"))
        tflop = cfg["tflop"]
        line = {
            "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"FLUX-VAE ch=128 ch_mult=1,2,4,4 z=16 {R}x{R}: {cfg['what']} fwd+bwd+grad all-reduce+"
                                   f"AdamW+weight re-pack (BASELINE.json configs[{cfg['idx']}]); LPIPS in eval mode "
                                   "(the reference trains with its Dropout(0.5) live; `Trainer(lpips_eval=False)` "
                                   "reproduces that)",
                       "name": args.config, "cuda_graph": graphed, "graph_prep_steps": PREP, "per_gpu_batch": B, "global_batch": world * B, "parallelism": f"dp{world}",
                       "l2": "no explicit flush: per-step working set (activations ~0.9 GB/image) >> 126 MB L2",
                       "tflop_per_image": tflop},
            "e2e": {"value": e2e, "unit": "images/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": B * 3 * R * R * 4,
                    "d2h_bytes_per_step": 4, "last_loss": last_loss},
            "gpu_launches": launches,
            "clocks": clocks,
            "peak_mem_gib": peak_mem,
            "achieved_step_tflops_per_gpu": tflop * B / (ms * 1e-3),
            "step_frac_of_peak": tflop * B / (ms * 1e-3) / peak,
            "roofline": {"kernel": "vqb::conv_gemm_kernel (tcgen05 implicit-GEMM conv, fwd+dgrad launches of one step)",
                         "bound": "tensor", "achieved": prof["conv"]["tflops"], "peak": peak, "unit": "TFLOP/s",
                         "frac": prof["conv"]["tflops"] / peak, "traffic": conv_traffic, "traffic_source": tname,
                         "traffic_per_shape": (ttab or {}).get("per_shape"), "peak_source": peak_src,
                         "launches_per_step": prof["conv"]["launches"], "ms_per_step": prof["conv"]["ms"],
                         "alg_flops_per_launch": prof["conv"]["flops_per_launch"],
                         "avg_launch_ms": prof["conv"]["ms_per_launch"]},
            "roofline_wgrad": {"kernel": "vqb::wgrad_gemm_kernel (+ split reduction)", "bound": "tensor",
                               "achieved": prof["wgrad"]["tflops"], "peak": peak, "unit": "TFLOP/s",
                               "frac": prof["wgrad"]["tflops"] / peak, "launches_per_step": prof["wgrad"]["launches"],
                               "ms_per_step": prof["wgrad"]["ms"]},
        }
        if eager is not None:
            line["eager_b200"] = eager
            if "value" in eager:
                line["vs_eager_b200"] = value / eager["value"]
        if world == 1 and not args.no_cpu_baseline:
            threads = cpu_threads()
            step, b = cpu_step_runner(batch=1, threads=threads)
            t0 = time.perf_counter()
            step()
            first = time.perf_counter() - t0
            n = 2 if first < 15 else 1
            t0 = time.perf_counter()
            for _ in range(n):
                step()
            dt = (time.perf_counter() - t0) / n
            line["cpu_baseline"] = {"value": b / dt, "unit": "images/s", "cores": threads, "kind": "port",
                                    "sample": f"{n} training steps at batch 1 of the configs[1] workload (oracle port "
                                              f"of the reference arithmetic, torch CPU fp32, {threads} threads); the "
                                              "reference tree is unpackaged Python and cannot be installed/travel"}
        emit_json(line)
        if dumped is not None:
            dump_outputs(dumped, args.dump_outputs)
    # release the captured step (its graph holds NCCL work) before tearing the process group down: with a live graph
    # destroy_process_group() hung until the launcher's timeout (N=2, round 2)
    tr = None
    import gc

    gc.collect()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
