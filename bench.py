#!/usr/bin/env python
"""Headline benchmark: images/sec of the ViT-B/16 patch-skip inference forward (BASELINE.json
configs[1]: bf16, batch 256 per B200, st=0.9, mt=0.5, synthetic inputs, random-init weights).

    python bench.py --gpus N --steps K --warmup W            # this implementation (libpsv.so)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)

One "step" = one forward of one batch of 256 images per GPU through the whole hot path
(embed -> 12 x [compressor/mask/compaction, LN, QKV, attention, proj, LN, MLP, scatter] -> head).
Batches are sharded across ranks with no data-path collective (weak scaling: 256 images per
GPU).  Rank 0 prints ONE JSON line; see DESIGN.md "Measurement" for every field.
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
PKG = os.path.join(ROOT, "vit-pruning_b200")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "images/sec ViT-B/16 patch-skip inference"
UNIT = "images/s"
BATCH_PER_GPU = 256
MT, ST = 0.5, 0.9


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="psv", choices=["psv", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="images per GPU per step")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--profile", default="natural", choices=["natural", "trained", "dense"],
                    help="skip profile: natural = compressor decisions of the random-init weights at mt=0.5 (the headline); "
                         "trained = each layer's mlp_layer.2.bias shifted so the per-layer skip ratio matches the reference's "
                         "logged trained profile (27.9 %% mean skip, SURVEY.md 6); dense = mt=0 (every token active)")
    ap.add_argument("--kv-mode", default="active", choices=["active", "all"],
                    help="'all' = query-only pruning variant (psv_set_kv_mode, reference recap/convprad4.py); not the headline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true",
                    help="skip the free-running bf16-vs-fp32 agreement leg (2048 images) of the default 1-GPU run")
    ap.add_argument("--no-extra-profiles", action="store_true",
                    help="skip the dense / trained profile legs that the default 1-GPU run adds under roofline.profiles")
    ap.add_argument("--config", type=int, default=2, choices=[2, 4, 5],
                    help="BASELINE.json config: 2 (default; also config 3 under torchrun) = ViT-B/16 patch-skip inference; "
                         "4 = DeiT-S/16 with the similarity skip criterion, batch 512; 5 = compressor-MLP training step")
    ap.add_argument("--cpu-sample", type=int, default=128, help="images in the CPU-baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step (rank 0) as "
                         "DIR/<name>.npy, float32 or float64; inputs and weights are seeded, so two builds run with the "
                         "same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 60 * 10 ** 6          # all arrays of --dump-outputs together (under 64 MB with the .npy headers)


def dump_outputs(out_dir, arrays):
    """arrays: name -> tensor / ndarray.  float64 is kept, everything else is written as float32.  If the arrays
    together exceed DUMP_BYTES, each is cut to the same fixed seeded sample of its flattened elements in every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v.cpu() if hasattr(v, "cpu") else v) for k, v in arrays.items()}
    arrays = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = a.size * DUMP_BYTES // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML in a thread of this process (what nvidia-smi
    reads; a sample every ~5 ms, no process start-up, so even a 70 ms timed region gets a dozen samples), with the
    nvidia-smi CLI (`-lms 100`) as the fallback when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.samples, self.stop_flag, self.max_mhz = None, [], False, None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.index])
            except Exception:
                pass
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._pump_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump_nvml(self):
        n = self.nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                r = int(get_reasons(self.handle))
                watts = float(n.nvmlDeviceGetPowerUsage(self.handle)) / 1e3
                self.samples.append((time.time(), mhz, [k for k, b in bits.items() if r & b], watts))
            except Exception:
                pass
            time.sleep(0.005)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            rows = [x for x in self.samples if t0 <= x[0] <= t1] or self.samples
            sm = [x[1] for x in rows]
            reasons = sorted({r for x in rows for r in x[2]})
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml",
                    "power_w": statistics.median([x[3] for x in rows]) if rows else None}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [l for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for (_, l) in self.lines]
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_forward_rate(n_images, threads, repeats=1, warmup=1, kind="randn", kv_all=False):
    """The reference's CPU path (oracle port, reference order: per-image loop, fp32, torch ops on
    the host cores) on a bounded sample of the workload.  Returns (img/s, seconds per pass)."""
    import torch
    import synth
    from oracle import vit_skip_oracle as O
    torch.set_num_threads(threads)
    geom = synth.VIT_B16
    sd = synth.make_state_dict(geom, seed=42)
    x = synth.make_pixels(n_images, geom, seed=1234, kind=kind)
    best = None
    with torch.no_grad():
        for i in range(warmup + repeats):
            t0 = time.perf_counter()
            O.forward(sd, x, MT, ST, kv_all=kv_all)
            dt = time.perf_counter() - t0
            if i >= warmup:
                best = dt if best is None else min(best, dt)
    return n_images / best, best


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.cpu_sample
    t_all0 = time.perf_counter()
    import torch
    import synth
    from oracle import vit_skip_oracle as O
    torch.set_num_threads(threads)
    geom = synth.VIT_B16
    sd = synth.make_state_dict(geom, seed=42)
    x = synth.make_pixels(n, geom, seed=1234)
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            r = O.forward(sd, x, MT, ST, kv_all=(args.kv_mode == "all"))
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_all0 > 240 and len(times) >= 1:
                break
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": r.logits, "n_active": r.masks.sum(-1)})
    total = sum(times)
    value = n * len(times) / total
    sample = f"{n} of the {args.batch} images of one step per pass, fp32, per-image loop (reference order), {len(times)} timed passes"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "batch_per_gpu": args.batch, "st": ST, "mt": MT,
                   "note": "CPU path does not use the GPUs; value is host-only throughput"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# per-layer skip ratios of the reference's trained compressor (CIFAR-100, st=0.9, mt=0.7), SURVEY.md section 6
TRAINED_SKIP = [0, 0, 0, 0, 0, .254, .656, .824, .838, .700, .076, 0]


def workload_name(args):
    prof = {"natural": "natural random-init skip profile", "dense": "dense (mt=0)",
            "trained": "reference's trained per-layer skip profile (27.9 % mean) imposed by shifting mlp_layer.2.bias"}[args.profile]
    return (f"ViT-B/16 224px patch-skip inference, {args.precision}, batch {args.batch} per B200, "
            f"st={ST} mt={0.0 if args.profile == 'dense' else MT}, {prof}, C=100"
            + (", query-only pruning (skipped tokens stay keys/values)" if getattr(args, "kv_mode", "active") == "all" else ""))


def calibrate_trained_profile(eng, sd, geom, pix, mt):
    """Shift each layer's compressor output bias so that the fraction of skipped patch tokens on `pix` equals
    TRAINED_SKIP[l] (layer by layer on the running hidden state), reload the weights, return the state dict."""
    import math
    import torch
    logit_mt = math.log(mt / (1.0 - mt))
    hidden = eng.embed(pix)
    for l in range(geom.layers):
        probe = hidden.clone()
        _, scores, _ = eng.layer_forward(l, probe, mt)
        z = torch.logit(scores.float().flatten().clamp(1e-7, 1 - 1e-7))
        target_active = 1.0 - TRAINED_SKIP[l]
        if target_active >= 1.0:
            delta = float(logit_mt - z.min()) + 1.0
        else:
            kth = max(1, int(round((1.0 - target_active) * z.numel())))
            delta = float(logit_mt - torch.kthvalue(z, kth).values) + 1e-6
        key = f"encoder.layer.{l}.mlp_layer.2.bias"
        sd[key] = sd[key] + delta
        eng.load_state_dict(sd)
        eng.layer_forward(l, hidden, mt)
    return sd


# --------------------------------------------------------------------------------------------- GPU arm
def gemm_flops_of_layer(T, D, F):
    return 2.0 * T * D * (3 * D) + 2.0 * T * D * D + 2.0 * T * D * F + 2.0 * T * F * D


class Runner:
    """Common plumbing of the GPU arms: ranks, barrier, device-side timing with the max over ranks."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, sampler=None):
        """W untimed warm-up calls of fn(i), then exactly `steps` calls between a barrier + synchronize on both sides,
        CUDA events on the current stream, max over ranks.  Returns (ms total, clocks or None)."""
        torch = self.torch
        for i in range(warmup):
            fn(i)
        self.barrier()
        if sampler is not None and self.rank == 0:
            sampler.start()
            time.sleep(0.05 if sampler.nvml is not None else 0.3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        w0 = time.time()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        w1 = time.time()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        clocks = sampler.stop(w0, w1) if (sampler is not None and self.rank == 0) else None
        return ms, clocks

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def graph_timeline(eng, pix, outs, mt, reps, plain_ms):
    """In-graph duration of every kernel of one forward: psv_profile_begin makes psv_forward capture a graph with an
    external event-record node between consecutive kernels; the deltas of `reps` replays are averaged per launch.  The
    event nodes themselves cost time (the timeline of a forward is longer than its plain replay): that overhead,
    (timeline sum - plain replay time) / launches, is subtracted from every launch ("corrected")."""
    import torch
    runs = []
    for r in range(reps):
        eng.profile_begin()
        eng.forward(pix[r % len(pix)], mt, want_n_active=True, use_graph=True, out=outs[r % len(outs)])
        torch.cuda.synchronize()
        runs.append(eng.profile_end(capacity=2048))
    n = len(runs[0])
    recs = [(runs[0][i][0], sum(x[i][1] for x in runs) / len(runs)) for i in range(n)]      # (kind, ms)
    total = sum(t for _, t in recs)
    overhead = max(0.0, (total - plain_ms) / max(1, n))
    by = {}
    for k, t in recs:
        a = by.setdefault(k, [0, 0.0])
        a[0] += 1
        a[1] += max(t - overhead, 0.0)
    return {"launches": n, "timeline_ms": total, "plain_replay_ms": plain_ms, "event_overhead_ms_per_launch": overhead,
            "by_kind": by}


def run_profile(R, eng, geom, args, peaks, mt, pix, steps, warmup, sampler=None):
    """Times `steps` graph-replayed forwards (two resident batches alternated) and derives the skip-scaled roofline."""
    import numpy as np
    import torch
    import synth
    B = pix[0].shape[0]
    outs = [dict(logits=torch.empty(B, geom.classes, device="cuda"),
                 n_active=torch.empty(geom.layers, B, dtype=torch.int32, device="cuda")) for _ in pix]

    def step(i):
        return eng.forward(pix[i % len(pix)], mt, want_n_active=True, use_graph=True, out=outs[i % len(outs)])

    ms, clocks = R.timed(step, steps, warmup, sampler)
    value = R.world * B * steps / (ms / 1e3)
    n_active = np.stack([o["n_active"].cpu().numpy() for o in outs], 0)           # [rot, L, B]
    flops_img = float(np.mean([synth.algorithmic_flops_per_image(n_active[i], geom, args.kv_mode == "all")
                               for i in range(len(outs))]))
    active_frac = float((n_active.mean() - 1) / (geom.tokens - 1))
    sus, burst = peaks["bf16_tflops_sustained"], peaks["bf16_tflops"]
    whole = {
        "images_per_s": value, "ms_per_step": ms / steps, "steps": steps,
        "algorithmic_gflop_per_image": flops_img / 1e9, "active_patch_fraction": active_frac,
        "skip_scaled_roofline_images_per_s": R.world * sus * 1e12 / flops_img,
        "frac_of_skip_scaled_roofline": value * flops_img / (R.world * sus * 1e12),
        "frac_of_skip_scaled_roofline_burst_peak": value * flops_img / (R.world * burst * 1e12),
        "achieved_tflops_per_gpu": value * flops_img / R.world / 1e12,
        "timed_region_ms": ms, "clocks": clocks,
    }
    return whole, outs, n_active, ms / steps, eng.last_launch_count


def free_running_parity(geom, B, n_batches=8):
    """Free-running bf16 engine (its own skip decisions, CUDA graph) against the fp32 parity engine (fp32 FFMA kernels;
    tests pin it to the CPU oracle: masks bit-exact outside the 1e-4 band, logits 1e-4) on n_batches x B fresh images.
    Reported, not a gate: with random-init compressors ~1 % of the decisions sit close enough to the threshold to flip
    under bf16 operands, and an image with a flipped decision leaves the 2e-2 logit tolerance."""
    import torch
    import psv_native
    import synth
    sd = synth.make_state_dict(geom, seed=42)
    e16 = psv_native.Engine(geom, "bf16", max_batch=B)
    e32 = psv_native.Engine(geom, "fp32", max_batch=B)
    e16.load_state_dict(sd)
    e32.load_state_dict(sd)
    agree = top1 = top1_dec = decided = clean = imgs = 0
    total_dec = 0
    worst_clean = 0.0
    for i in range(n_batches):
        x = synth.make_pixels(B, geom, seed=9000 + i).cuda()
        a = e16.forward(x, MT, want_masks=True, use_graph=True)
        b = e32.forward(x, MT, want_masks=True)
        torch.cuda.synchronize()
        same = a["masks"] == b["masks"]
        agree += int(same.sum()); total_dec += same.numel()
        la, lb = a["logits"], b["logits"]
        hit = la.argmax(1) == lb.argmax(1)
        top2 = lb.topk(2, dim=1).values
        dec = (top2[:, 0] - top2[:, 1]) > 4e-2
        cl = same.all(0).all(1)
        top1 += int(hit.sum()); decided += int(dec.sum()); top1_dec += int(hit[dec].sum()); clean += int(cl.sum()); imgs += B
        if cl.any():
            worst_clean = max(worst_clean, float((la - lb)[cl].abs().max()))
    e16.close()
    e32.close()
    return {"images": imgs, "reference": "fp32 parity engine of this library, free running (pinned to the CPU oracle by tests/)",
            "mask_agreement": agree / total_dec, "images_with_every_decision_equal": clean,
            "logits_max_abs_err_on_those": worst_clean,
            "top1_agreement_raw": top1 / imgs, "top1_agreement_margin_gt_4e-2": top1_dec / max(1, decided),
            "images_with_margin_gt_4e-2": decided}


def quantised_u8_images(pix):
    """The same randn images as raw uint8 HWC: u8 = round(clip(x, -4, 4) / 8 * 255 + 127.5); with mean 0.5 / std 0.125
    the fused input pipeline maps them back to x (step 0.031, clipped at +-4)."""
    import torch
    u = torch.clamp(pix, -4.0, 4.0) * (0.125 * 255.0) + 127.5
    return torch.round(u).clamp_(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def run_psv_arm(args):
    import numpy as np
    import torch
    import psv_native
    import synth

    R = Runner()
    world, rank = R.world, R.rank
    geom = synth.VIT_B16
    B = args.batch
    mt = 0.0 if args.profile == "dense" else MT
    peaks = load_peaks()
    warmup = max(args.warmup, 3)

    sd = synth.make_state_dict(geom, seed=42)
    eng = psv_native.Engine(geom, args.precision, max_batch=B)
    eng.load_state_dict(sd)
    eng.set_kv_mode(args.kv_mode)
    if args.profile == "trained":
        calibrate_trained_profile(eng, sd, geom, synth.make_pixels(B, geom, seed=1234 + 17 * rank).cuda(), mt)
    # two different resident batches per rank (fp32 pixel_values as the reference's loader yields);
    # 154 MB each > 126 MB L2, alternated between steps
    n_rot = 2
    host_f32 = [synth.make_pixels(B, geom, seed=1234 + 17 * rank + 1000 * i) for i in range(n_rot)]
    pix = [p.cuda() for p in host_f32]

    sampler = ClockSampler(R.local)
    whole, outs, n_active, ms_step, launches_per_step = run_profile(R, eng, geom, args, peaks, mt, pix, args.steps, warmup,
                                                                    sampler)
    if args.dump_outputs and rank == 0:          # before the legs below reuse the output buffers
        last = outs[(args.steps - 1) % len(outs)]
        dump_outputs(args.dump_outputs, {"logits": last["logits"], "n_active": last["n_active"]})
    value, clocks = whole["images_per_s"], whole.pop("clocks")
    flops_img, active_frac = whole["algorithmic_gflop_per_image"] * 1e9, whole["active_patch_fraction"]

    # ---- e2e: the same metric through the C ABI with HOST buffers, every step: H2D of the step's images from pinned
    #      host memory + D2H of its logits and n_active, inside the timed region.  The images travel as what a camera /
    #      decoder delivers -- raw uint8 HWC (psv_set_u8_input: rescale + normalise fused into the patch embedding) --
    #      and are the SAME randn images as the device-resident leg, quantised to 8 bits.
    d2h = B * geom.classes * 4 + geom.layers * B * 4
    host_logits2 = [torch.empty(B, geom.classes).pin_memory() for _ in range(2)]
    host_nact2 = [torch.empty(geom.layers, B, dtype=torch.int32).pin_memory() for _ in range(2)]

    def host_loop(host_batches):
        def run(n):
            for i in range(n):
                eng.forward_host_submit(i & 1, host_batches[i % len(host_batches)], mt, host_logits2[i & 1], host_nact2[i & 1])
                if i >= 1:
                    eng.forward_host_wait((i - 1) & 1)
            eng.forward_host_wait((n - 1) & 1)
        return run

    def time_host_loop(host_batches, steps):
        run = host_loop(host_batches)
        run(3)
        R.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(steps)
        e1.record()                              # after the host has seen the last step's logits
        R.barrier()
        t = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([t], device="cuda", dtype=torch.float64)
            R.dist.all_reduce(tt, op=R.dist.ReduceOp.MAX)
            t = float(tt.item())
        return t

    def h2d_alone_gbs(host_batch, reps=6):
        """all ranks copy their step input at the same time, nothing else running: the host-side ceiling at this N"""
        dst = torch.empty_like(host_batch, device="cuda")
        dst.copy_(host_batch, non_blocking=True)
        R.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dst.copy_(host_batch, non_blocking=True)
        e1.record()
        R.barrier()
        t = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([t], device="cuda", dtype=torch.float64)
            R.dist.all_reduce(tt, op=R.dist.ReduceOp.MAX)
            t = float(tt.item())
        return host_batch.numel() * host_batch.element_size() * reps / (t / 1e3) / 1e9

    e2e = None
    e2e_fp32 = None
    if True:
        eng.set_u8_input(geom.image, geom.image, mean=(0.5, 0.5, 0.5), std=(0.125, 0.125, 0.125))
        host_u8 = [quantised_u8_images(p).pin_memory() for p in host_f32]
        u8_ms = time_host_loop(host_u8, args.steps)
        u8_active = float((np.mean([h.float().mean().item() for h in host_nact2]) - 1.0) / geom.patches)
        h2d = host_u8[0].numel()
        e2e = {"value": world * B * args.steps / (u8_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": u8_ms / args.steps,
               "active_patch_fraction": u8_active,
               "h2d_gbs_per_gpu_needed": h2d / (u8_ms / args.steps / 1e3) / 1e9,
               "h2d_gbs_per_gpu_alone": h2d_alone_gbs(host_u8[0]),
               "input": "uint8 [B,224,224,3] HWC, the device-resident leg's randn images quantised to 8 bits "
                        "(x = (u8/255 - 0.5) / 0.125: step 0.031, clipped at +-4)",
               "api": "psv_set_u8_input(224, 224, mean 0.5, std 0.125) + psv_forward_host_submit/_wait with "
                      "PSV_PIXELS_U8_HWC: pinned host images -> host logits + n_active, two slots (H2D of step i "
                      "overlaps the forward of step i-1)"}
        # the round-1 form of the same loop (fp32 pixel_values, 154 MB per step) for continuity: this is the leg whose
        # 1->8 GPU curve is bounded by host->device traffic
        f32_steps = min(args.steps, 10)
        host_pin = [p.pin_memory() for p in host_f32]
        f32_ms = time_host_loop(host_pin, f32_steps)
        hb = host_pin[0].numel() * 4
        e2e_fp32 = {"value": world * B * f32_steps / (f32_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": hb,
                    "d2h_bytes_per_step": d2h, "ms_per_step": f32_ms / f32_steps, "steps": f32_steps,
                    "h2d_gbs_per_gpu_needed": hb / (f32_ms / f32_steps / 1e3) / 1e9,
                    "h2d_gbs_per_gpu_alone": h2d_alone_gbs(host_pin[0])}
        del host_pin

    # ---- roofline leg: the in-graph timeline of the same forwards (external event-record nodes between the kernels)
    tl = graph_timeline(eng, pix, outs, mt, reps=min(args.steps, 6), plain_ms=ms_step)
    by_kind = tl["by_kind"]
    step_kernel_ms = sum(v[1] for v in by_kind.values())
    shares = {k: {"launches_per_step": v[0], "ms_per_step": v[1], "share": v[1] / step_kernel_ms}
              for k, v in by_kind.items()}
    D, F, L = geom.hidden, geom.ffn, geom.layers
    T = n_active.mean(axis=0).sum(axis=1).astype(np.float64)                       # rows per layer (mean of the two batches)
    gemm_flops = float(sum(gemm_flops_of_layer(t, D, F) for t in T)) + 2.0 * B * geom.patches * D * 768
    if args.kv_mode == "all":
        gemm_flops += float(sum(4.0 * (B * geom.tokens - t) * D * D for t in T))
    gemm_launches, gemm_ms = by_kind.get("gemm", [0, 0.0])
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    bf = args.precision == "bf16"
    peak = peaks["bf16_tflops_sustained"] if bf else 75.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.isfile(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    hbm_peak = peaks["hbm_gbs"]
    rows_all = float(B * geom.tokens)
    t_sum = float(n_active.mean(axis=0).sum())
    es = 2 if bf else 4
    hbm_bytes = {
        "score_mask": L * (rows_all * D * 4 + rows_all * 5),
        "compact_gather_ln": t_sum * D * (4 + es) + L * rows_all + 12 * t_sum,
        "layernorm": t_sum * D * (4 + es),
    }
    if args.kv_mode == "all":
        hbm_bytes["layernorm"] += L * rows_all * D * (4 + es)
    hbm_kernels = {}
    for k, nbytes in hbm_bytes.items():
        if k in shares and shares[k]["ms_per_step"] > 0:
            gbs = nbytes / (shares[k]["ms_per_step"] / 1e3) / 1e9
            hbm_kernels[k] = {"algorithmic_bytes_per_step": nbytes, "ms_per_step": shares[k]["ms_per_step"],
                              "achieved_gbs": gbs, "peak_gbs": hbm_peak, "frac": gbs / hbm_peak}
    roofline = {
        "bound": "tensor",
        "kernel": "gemm_tc_kernel (tcgen05 bf16 GEMM, all 4 GEMMs of a layer + patch embed)" if bf else "gemm_simt_kernel (fp32 FFMA)",
        "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
        "frac_of_burst_peak": achieved / peaks["bf16_tflops"] if bf else None,
        "peak_source": peaks["source"] + (" bf16_tflops_sustained (the launches are timed INSIDE the graph-replayed step)" if bf
                                          else " (nominal fp32 FFMA)"),
        "timing": "in-graph: CUDA-event deltas between consecutive kernels of the replayed forward, minus the mean "
                  "event-node overhead per launch",
        "traffic": traffic, "traffic_source": "stored ncu figure (profiles/gemm_traffic.json: dram read+write per GEMM launch of one forward)",
        "launches_timed": gemm_launches, "avg_launch_ms": gemm_ms / gemm_launches if gemm_launches else None,
        "algorithmic_flops_per_launch": gemm_flops / gemm_launches if gemm_launches else None,
        "gemm_share_of_step": shares.get("gemm", {}).get("share"),
        "timeline": {k: tl[k] for k in ("launches", "timeline_ms", "plain_replay_ms", "event_overhead_ms_per_launch")},
        "whole_path": {k: whole[k] for k in ("algorithmic_gflop_per_image", "skip_scaled_roofline_images_per_s",
                                             "frac_of_skip_scaled_roofline", "frac_of_skip_scaled_roofline_burst_peak",
                                             "achieved_tflops_per_gpu", "timed_region_ms")},
        "kernel_shares": shares,
        "hbm_kernels": hbm_kernels,
    }

    # ---- sustained leg (1 GPU): the same forwards back to back for ~3 s.  The timed region above is a burst (tens of
    #      ms at the maximum SM clock); after about a second of continuous work the board reaches its power limit and the
    #      power controller lowers the SM clock (sw_power_cap) -- reported beside the headline, not instead of it.
    sustained = None
    if world == 1 and args.profile == "natural" and not args.no_extra_profiles:
        smp = ClockSampler(R.local)
        smp.start()
        t_start, vals = time.time(), []
        while time.time() - t_start < 3.0:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(20):
                eng.forward(pix[i % 2], mt, want_n_active=True, use_graph=True, out=outs[i % 2])
            e1.record()
            torch.cuda.synchronize()
            vals.append((time.time() - t_start, e0.elapsed_time(e1) / 20))
        t_end = time.time()
        tail = [v for t, v in vals if t > 1.5] or [v for _, v in vals]
        ck = smp.stop(t_start + 1.5, t_end)
        ms_sus = sum(tail) / len(tail)
        time.sleep(2.5)          # let the board's power average fall again: the profiles below are bursts like the headline
        sustained = {"value": B / (ms_sus / 1e3), "unit": UNIT, "ms_per_step": ms_sus, "seconds": t_end - t_start,
                     "averaged_over": "steps after the first 1.5 s", "clocks": ck,
                     "frac_of_skip_scaled_roofline": (B / (ms_sus / 1e3)) / whole["skip_scaled_roofline_images_per_s"]}

    # ---- the other two skip profiles of SURVEY.md 8d in the same run (1 GPU): dense (mt = 0) and the reference's
    #      trained per-layer profile (imposed by shifting mlp_layer.2.bias; done last because it edits the weights)
    profiles = {args.profile: dict(whole, clocks=clocks)}
    if world == 1 and args.profile == "natural" and not args.no_extra_profiles:
        psteps = min(args.steps, 10)
        w_d, *_ = run_profile(R, eng, geom, args, peaks, 0.0, pix, psteps, 3, ClockSampler(R.local))
        profiles["dense"] = w_d
        calibrate_trained_profile(eng, sd, geom, pix[0], MT)
        time.sleep(2.0)          # as after the sustained leg: each profile is a burst from a rested board
        w_t, *_ = run_profile(R, eng, geom, args, peaks, MT, pix, psteps, 3, ClockSampler(R.local))
        profiles["trained"] = w_t
    roofline["profiles"] = profiles

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.precision, "data": "synthetic",
        "config": {"workload": workload_name(args), "global_batch": world * B, "batch_per_gpu": B,
                   "active_patch_fraction": active_frac, "skip_fraction": 1.0 - active_frac,
                   "weights": "random-init seed 42 (reference init scheme)", "inputs": "randn seed 1234+",
                   "l2": f"two resident {B * 3 * geom.image * geom.image * 4 / 1e6:.0f} MB fp32 pixel batches (> 126 MB L2) alternated between steps",
                   "cuda_graph": True, "parallelism": f"batch-sharded x{world}, no collective"},
        "e2e": e2e,
        "e2e_fp32_pixels": e2e_fp32,
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step,
        "clocks": clocks,
        "sustained": sustained,
        "roofline": roofline,
    }
    if rank == 0 and world == 1 and not args.no_parity_check and args.precision == "bf16" and args.profile == "natural":
        line["free_running_parity"] = free_running_parity(geom, B)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, secs = cpu_reference_forward_rate(args.cpu_sample, threads, repeats=2, warmup=1, kv_all=(args.kv_mode == "all"))
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{args.cpu_sample} images of the step's batch, fp32, per-image loop "
                                          f"(reference order), best of 2 after 1 warm-up, {secs:.1f} s per pass"}
    else:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line))
    eng.close()
    R.close()


# --------------------------------------------------------------------------------------------- configs 4 and 5
def eager_kernel_shares(eng, fn):
    """per-kind kernel time of one eager call of fn() (events around every launch; includes launch gaps)"""
    import torch
    eng.profile_begin()
    fn()
    torch.cuda.synchronize()
    by = {}
    for k, t in eng.profile_end(capacity=4096):
        a = by.setdefault(k, [0, 0.0])
        a[0] += 1
        a[1] += t
    total = sum(v[1] for v in by.values())
    return {k: {"launches_per_step": v[0], "ms_per_step": v[1], "share": v[1] / total} for k, v in by.items()}, total


def run_config4(args):
    """BASELINE config 4: DeiT-S/16 geometry, similarity ("type=cosine") skip criterion, batch 512 per GPU.
    Per layer: psv_similarity_mask (dense pass of the layer + blended similarity -> mask = [True, sim < st], reference
    pradeep/model_utils.py:73-84,91) then psv_layer_forward(forced mask) on the active set."""
    import numpy as np
    import torch
    import psv_native
    import synth
    R = Runner()
    peaks = load_peaks()
    geom = synth.DEIT_S16
    B = 512 if args.batch == BATCH_PER_GPU else args.batch
    eng = psv_native.Engine(geom, "bf16", B)
    sd = synth.make_state_dict(geom, 42)
    eng.load_state_dict(sd)
    pix = [synth.make_pixels(B, geom, seed=1234 + 17 * R.rank + 1000 * i).cuda() for i in range(2)]
    active = []
    last = {}

    def step(i):
        h = eng.embed(pix[i & 1])
        active.clear()
        for l in range(geom.layers):
            mask, _ = eng.similarity_mask(l, h, ST)
            _, _, n = eng.layer_forward(l, h, MT, forced_mask=mask, want_mask=False, want_scores=False)
            active.append(n)
        last["logits"] = eng.head(h)

    sampler = ClockSampler(R.local)
    ms, clocks = R.timed(step, args.steps, max(args.warmup, 3), sampler)
    value = R.world * B * args.steps / (ms / 1e3)
    n_act = torch.stack(active).cpu().numpy().astype(np.float64)                 # [L, B]
    if args.dump_outputs and R.rank == 0:
        dump_outputs(args.dump_outputs, {"logits": last["logits"], "n_active": n_act})
    D, F, N = geom.hidden, geom.ffn, geom.tokens
    dense_layer = N * (24.0 * D * D) + N * N * 4.0 * D
    skip_flops = synth.algorithmic_flops_per_image(n_act, geom)                   # active-set layers + embed + head (+ unused compressor term)
    flops_img = skip_flops + geom.layers * dense_layer
    shares, eager_ms = eager_kernel_shares(eng, lambda: step(0))
    sus = peaks["bf16_tflops_sustained"]
    gemm = shares.get("gemm", {})
    gemm_flops = float(sum(gemm_flops_of_layer(t, D, F) for t in n_act.sum(axis=1))) + geom.layers * gemm_flops_of_layer(B * N, D, F) \
        + 2.0 * B * geom.patches * D * 768
    ach = gemm_flops / (gemm.get("ms_per_step", 0.0) / 1e3) / 1e12 if gemm else 0.0
    line = {
        "metric": "images/sec DeiT-S/16 patch-skip, similarity (cosine) skip criterion", "value": value, "unit": UNIT,
        "n_gpus": R.world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"BASELINE config 4: DeiT-S/16 (D=384, H=6, F=1536), similarity skip criterion st={ST}, batch {B} per B200, "
                               "per layer: dense pass + similarity -> mask, then the skip layer on the active set",
                   "batch_per_gpu": B, "global_batch": R.world * B,
                   "active_token_fraction": float(n_act.mean() / N), "cuda_graph": False,
                   "l2": "two resident pixel batches alternated (308 MB each > 126 MB L2)"},
        "gpu_launches": eng.last_launch_count, "clocks": clocks, "e2e": None, "cpu_baseline": None,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel (K = 384 / 1536 shapes)", "achieved": ach, "peak": peaks["bf16_tflops"],
                     "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"] if ach else None,
                     "peak_source": peaks["source"] + " bf16_tflops (burst: eager launches timed one by one)", "traffic": None,
                     "whole_path": {"algorithmic_gflop_per_image": flops_img / 1e9,
                                    "frac_of_skip_scaled_roofline": value * flops_img / (R.world * sus * 1e12),
                                    "note": "dense criterion pass of every layer + active-set layers + embedding"},
                     "kernel_shares": shares, "eager_kernel_ms_per_step": eager_ms},
    }
    if R.rank == 0:
        print(json.dumps(line))
    eng.close()
    R.close()


def run_config5(args):
    """BASELINE config 5: one compressor-MLP training step on the frozen ViT-B/16 backbone, batch 64 per GPU
    (reference main_model_utils.py:100-191 with loss_type='cosine' and mlp_train(), himanshu's loss model_utils.py:103-108:
    labels = the layer's own mask, so no dense label pass is needed for the gradient): psv_compressor_grads (skip forward
    + loss + gradients of all 12 compressors) -> exchange of the flat 4.7 MB gradient bucket (fused peer-memory
    all-reduce + Adam, or NCCL all-reduce then Adam) -> the same Adam update on every rank."""
    import numpy as np
    import torch
    import psv_native
    import synth
    import main_model_utils
    R = Runner()
    peaks = load_peaks()
    geom = synth.VIT_B16
    B = 64 if args.batch == BATCH_PER_GPU else args.batch
    eng = psv_native.Engine(geom, "bf16", B)
    eng.load_state_dict(synth.make_state_dict(geom, 42))
    pix = [synth.make_pixels(B, geom, seed=99 + 17 * R.rank + 1000 * i).cuda() for i in range(2)]
    trainer = main_model_utils.CompressorTrainer(eng, mlp_threshold=MT, lr=1e-3)
    losses = []

    def step(i):
        losses.append(trainer.step(pix[i & 1]))

    sampler = ClockSampler(R.local)
    ms, clocks = R.timed(step, args.steps, max(args.warmup, 3), sampler)
    value = R.world * B * args.steps / (ms / 1e3)
    if args.dump_outputs and R.rank == 0:
        dump_outputs(args.dump_outputs, {"loss": losses[-1], "compressor_params": eng.get_compressor_params()})
    r = eng.forward(pix[0], MT, want_n_active=True)
    torch.cuda.synchronize()
    n_act = r["n_active"].cpu().numpy().astype(np.float64)
    D, CH = geom.hidden, geom.comp_hidden
    fwd = synth.algorithmic_flops_per_image(n_act, geom)
    bwd = geom.layers * (2.0 * geom.patches * CH * 2 * D + 2.0 * geom.patches * CH)      # dW1 (+ the small terms) per image
    flops_img = fwd + bwd
    shares, eager_ms = eager_kernel_shares(eng, lambda: trainer.engine.compressor_grads(pix[0], MT))
    sus = peaks["bf16_tflops_sustained"]
    line = {
        "metric": "images/sec compressor-MLP training (frozen ViT-B/16 backbone)", "value": value, "unit": UNIT,
        "n_gpus": R.world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16 backbone / fp32 compressor", "data": "synthetic",
        "config": {"workload": f"BASELINE config 5: compressor training step, batch {B} per B200, Adam lr 1e-3, st={ST} mt={MT}",
                   "batch_per_gpu": B, "global_batch": R.world * B, "collective": trainer.collective,
                   "collective_note": trainer.collective_note,
                   "allreduce_bytes_per_step": int(eng.compressor_param_count) * 4 if R.world > 1 else 0,
                   "loss_first": float(losses[0].sum()), "loss_last": float(losses[-1].sum()),
                   "note": "the reference's pos_weight = mean/(1-mean+1e-16) (model_utils.py:104-105) blows the loss up once a "
                           "layer keeps every token; reproduced as is"},
        "gpu_launches": None, "clocks": clocks, "e2e": None, "cpu_baseline": None,
        "roofline": {"bound": "tensor", "kernel": "whole step", "achieved": value * flops_img / R.world / 1e12, "peak": sus,
                     "unit": "TFLOP/s", "frac": value * flops_img / (R.world * sus * 1e12),
                     "peak_source": peaks["source"] + " bf16_tflops_sustained", "traffic": None,
                     "whole_path": {"algorithmic_gflop_per_image": flops_img / 1e9},
                     "kernel_shares": shares, "eager_kernel_ms_per_step": eager_ms},
    }
    if R.rank == 0:
        print(json.dumps(line))
    eng.close()
    R.close()


def main():
    args = parse_args()
    # keep stdout clean for the single JSON line: libraries (e.g. "NCCL version ...") print to fd 1
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.config == 4:
        run_config4(args)
    elif args.config == 5:
        run_config5(args)
    else:
        run_psv_arm(args)


if __name__ == "__main__":
    main()
