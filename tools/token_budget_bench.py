"""Throughput of per-layer token budgets (psv_set_token_budget) on ViT-B/16, bf16, batch 256, CUDA-graph replay.

Two resident batches of fp32 pixels (2 x 154 MB, more than the 126 MB L2) are alternated.  Every leg is timed in the
two regimes tools/quick_bench.py describes: BURST (a short run after an idle pause, SM clock at its maximum; median of
5) and SUSTAINED (back to back for --sustain seconds, board at its power cap).  Legs:
  * plain threshold (mt = 0.5, natural profile of the seed-42 weights);
  * EXACT with uniform k in {24, 49, 98, 147, 196};
  * CAP at k = 64 on the natural profile, alternated with the plain threshold;
  * the reference's logged trained skip profile as per-layer EXACT budgets, k_l = round(196 (1 - skip_l)), alternated
    with bench.py's way of reaching it (each mlp_layer.2.bias shifted to a score quantile) at the same mean token count;
  * a separate profiling pass (psv_profile_begin / end, inside the replayed graph): the budget kernel's time per layer.
Usage: python tools/token_budget_bench.py [--out profiles/token_budget.txt] [--steps 12] [--sustain 2]"""
import argparse
import copy
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "vit-pruning_b200"), ROOT):
    sys.path.insert(0, p)

import torch  # noqa: E402

import bench  # noqa: E402
import psv_native  # noqa: E402
import synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "token_budget.txt"))
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--steps", type=int, default=12)
ap.add_argument("--sustain", type=float, default=2.0)
args = ap.parse_args()

geom, B, MT = synth.VIT_B16, args.batch, 0.5
P = geom.tokens - 1
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
except Exception:
    power = "unknown"
say(f"token budget throughput, ViT-B/16 bf16 batch {B}, CUDA-graph replay, two resident fp32 batches alternated")
say(f"device: {torch.cuda.get_device_name()}, power limit {power}")

sd = synth.make_state_dict(geom, seed=42)
eng = psv_native.Engine(geom, "bf16", max_batch=B)
eng.load_state_dict(sd)
pix = [synth.make_pixels(B, geom, seed=1234 + 1000 * i).cuda() for i in range(2)]
outs = [dict(logits=torch.empty(B, geom.classes, device="cuda"),
             n_active=torch.empty(geom.layers, B, dtype=torch.int32, device="cuda")) for _ in range(2)]


def timed(e, mt, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        e.forward(pix[i % 2], mt, want_n_active=True, use_graph=True, out=outs[i % 2])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


def warm(e, mt):
    for _ in range(6):
        timed(e, mt, 2)
    return float(outs[0]["n_active"].float().mean()) - 1.0          # mean kept patches per layer and image


def burst(e, mt):
    time.sleep(0.7)                     # let the board's power average fall: the run starts at the maximum clock
    timed(e, mt, 2)
    return timed(e, mt, args.steps)


def sustained(e, mt):
    t0, vals = time.perf_counter(), []
    while time.perf_counter() - t0 < args.sustain:
        v = timed(e, mt, 20)
        if time.perf_counter() - t0 > args.sustain / 3:
            vals.append(v)
    return statistics.mean(vals)


def row(name, kept, b, s):
    say(f"{name:44s} kept {kept:6.1f}/{P} patches/layer  burst {b:8.1f} us ({B / b * 1e6:6.0f} img/s)  "
        f"sustained {s:8.1f} us ({B / s * 1e6:6.0f} img/s)")


def leg(name, e, mt, setup=None):
    if setup:
        setup()
    kept = warm(e, mt)
    bs = [burst(e, mt) for _ in range(5)]
    row(name, kept, statistics.median(bs), sustained(e, mt))


def pair(names, engines, setups, rounds=3):
    """two configurations alternated in the same call: burst samples interleaved, then sustained each"""
    bs = [[], []]
    kept = [0.0, 0.0]
    for _ in range(rounds):
        for i in range(2):
            setups[i]()
            kept[i] = warm(engines[i], MT)
            bs[i] += [burst(engines[i], MT) for _ in range(2)]
    for i in range(2):
        setups[i]()
        warm(engines[i], MT)
        row(names[i], kept[i], statistics.median(bs[i]), sustained(engines[i], MT))


say()
say("-- EXACT, uniform k (mt ignored) against the plain threshold")
leg("threshold mt=0.5 (natural)", eng, MT, lambda: eng.set_token_budget(None))
for k in (24, 49, 98, 147, 196):
    leg(f"EXACT k={k}", eng, MT, lambda k=k: eng.set_token_budget(k, "exact"))

say()
say("-- CAP k=64 on the natural profile, alternated with the plain threshold")
pair(["threshold mt=0.5 (natural)", "CAP k=64, mt=0.5"], [eng, eng],
     [lambda: eng.set_token_budget(None), lambda: eng.set_token_budget(64, "cap")])

say()
say("-- the logged trained profile: per-layer EXACT budgets vs bench.py's bias-shifted compressors")
keep = [int(round(P * (1 - s))) for s in bench.TRAINED_SKIP]
say(f"budgets k_l = round(196 (1 - skip_l)) = {keep}")
eng_t = psv_native.Engine(geom, "bf16", max_batch=B)
eng_t.load_state_dict(sd)
sd_t = bench.calibrate_trained_profile(eng_t, copy.deepcopy(sd), geom, pix[0], MT)
pair(["trained profile as EXACT budgets", "trained profile by bias shift (bench.py)"], [eng, eng_t],
     [lambda: eng.set_token_budget(keep, "exact"), lambda: None])
eng_t.close()

say()
say("-- in-graph kernel times (profiling pass, separate from the timings above)")
for name, budget, mode in (("EXACT k=49", 49, "exact"), ("trained EXACT budgets", keep, "exact"),
                           ("CAP k=64", 64, "cap")):
    eng.set_token_budget(budget, mode)
    warm(eng, MT)
    eng.profile_begin()
    for i in range(4):
        eng.forward(pix[i % 2], MT, want_n_active=True, use_graph=True, out=outs[i % 2])
    recs = eng.profile_end()
    bud = [ms for k, ms in recs if k == "budget_mask"]
    total = sum(ms for _, ms in recs) / 4
    per = 1e3 * sum(bud) / len(bud)
    say(f"{name:30s} budget_mask {per:6.2f} us per layer (min {1e3 * min(bud):.2f}, max {1e3 * max(bud):.2f}), "
        f"{1e3 * sum(bud) / 4:7.1f} us per forward = {sum(bud) / 4 / total:.2%} of the {1e3 * total:.0f} us of kernels")
eng.close()

os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out, "w") as f:
    f.write("\n".join(lines) + "\n")
print(f"wrote {args.out}")
