"""Fast same-box A/B number: us per graph-replayed forward (natural profile, batch 256, two resident batches alternated),
in the two regimes the board has (tools/power_probe.py): BURST = a short run after an idle second, SM clock at its
maximum (what a 20-step bench measures), and SUSTAINED = back to back for seconds, board power at its 1000 W cap and the
SM clock lowered by the power controller (sw_power_cap).
usage: [PSV_LIB=path/to/libpsv.so] python tools/quick_bench.py [--geom vitb16|deits16|vitl16] [--profile natural|dense|trained]
                                                             [--steps 12] [--sustain 3] [--tag name]
Also prints the mean active fraction of the patch tokens, the skip-scaled algorithmic GFLOP per image
(synth.algorithmic_flops_per_image), the achieved TFLOP/s and their fraction of the bf16 peak bench.py uses, and the
GPU's name and power limit."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vit-pruning_b200"), ROOT]
import torch  # noqa: E402
import psv_native  # noqa: E402
import synth  # noqa: E402
import bench  # noqa: E402

GEOMS = {"vitb16": synth.VIT_B16, "deits16": synth.DEIT_S16, "vitl16": synth.VIT_L16}
ap = argparse.ArgumentParser()
ap.add_argument("--geom", choices=sorted(GEOMS), default="vitb16")
ap.add_argument("--profile", default="natural")
ap.add_argument("--steps", type=int, default=12)
ap.add_argument("--sustain", type=float, default=3.0, help="seconds of back-to-back forwards for the sustained figure (0: skip)")
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--tag", default=os.environ.get("PSV_LIB", "default"))
args = ap.parse_args()
geom = GEOMS[args.geom]
B = args.batch
mt = 0.0 if args.profile == "dense" else 0.5
sd = synth.make_state_dict(geom, seed=42)
eng = psv_native.Engine(geom, "bf16", max_batch=B)
eng.load_state_dict(sd)
if args.profile == "trained":
    bench.calibrate_trained_profile(eng, sd, geom, synth.make_pixels(B, geom, seed=1234).cuda(), mt)
pix = [synth.make_pixels(B, geom, seed=1234 + 1000 * i).cuda() for i in range(2)]
outs = [dict(logits=torch.empty(B, geom.classes, device="cuda"),
             n_active=torch.empty(geom.layers, B, dtype=torch.int32, device="cuda")) for _ in range(2)]
for i in range(6):
    eng.forward(pix[i % 2], mt, want_n_active=True, use_graph=True, out=outs[i % 2])
torch.cuda.synchronize()
import statistics  # noqa: E402
import time  # noqa: E402


def timed(n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        eng.forward(pix[i % 2], mt, want_n_active=True, use_graph=True, out=outs[i % 2])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


burst = []
for rep in range(5):
    time.sleep(1.0)                      # let the board's power average fall: the next run starts at the maximum clock
    timed(2)
    burst.append(timed(args.steps))
sus = float("nan")
if args.sustain > 0:
    t0, vals = time.perf_counter(), []
    while time.perf_counter() - t0 < args.sustain:
        v = timed(20)
        if time.perf_counter() - t0 > args.sustain / 3:
            vals.append(v)
    sus = statistics.mean(vals)
b = statistics.median(burst)
n_active = [o["n_active"].cpu().numpy() for o in outs]
active = float((sum(a.mean() for a in n_active) / len(n_active) - 1) / (geom.tokens - 1))
flops_img = sum(synth.algorithmic_flops_per_image(a, geom) for a in n_active) / len(n_active)
peaks = bench.load_peaks()
tflops_b, tflops_s = B / b * 1e6 * flops_img / 1e12, B / sus * 1e6 * flops_img / 1e12
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"
print(f"{args.geom} batch {B}, {active:.1%} of patch tokens active, {flops_img / 1e9:.1f} algorithmic GFLOP/image; "
      f"burst {tflops_b:.0f} TFLOP/s = {tflops_b / peaks['bf16_tflops']:.1%} of {peaks['bf16_tflops']:.0f}, sustained "
      f"{tflops_s:.0f} TFLOP/s = {tflops_s / peaks['bf16_tflops_sustained']:.1%} of {peaks['bf16_tflops_sustained']:.0f} "
      f"(bf16 peaks: {peaks['source']})  [{torch.cuda.get_device_name()}, power limit {power}]")
print(f"{args.tag:32s} {args.profile:8s} burst {b:8.1f} us/forward ({B / b * 1e6:7.0f} img/s; min {min(burst):.1f} max {max(burst):.1f})   "
      f"sustained {sus:8.1f} us ({B / sus * 1e6:7.0f} img/s)   checksum {float(outs[0]['logits'].double().sum()):.6f}")
eng.close()
