"""Time of one backbone fine-tuning step through the C ABI (psv_backbone_forward_train + psv_backbone_backward), ViT-B/16
by default, fp32 parity path: forward and backward separately.
usage: python tools/finetune_bench.py [--geom vitb16|deits16|vitl16] [--batch 64] [--joint] [--kv-mode {active,all}] [--mt 0.5]
                                     [--criterion {mlp,similarity}] [--st 0.9] [--u8]
Prints the GPU's name and power limit with the result, since the time depends on both."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vit-pruning_b200"), ROOT]
import torch  # noqa: E402
import psv_native  # noqa: E402
import synth  # noqa: E402

GEOMS = {"vitb16": ("ViT-B/16", synth.VIT_B16), "deits16": ("DeiT-S/16", synth.DEIT_S16),
         "vitl16": ("ViT-L/16", synth.VIT_L16)}
ap = argparse.ArgumentParser()
ap.add_argument("--geom", choices=sorted(GEOMS), default="vitb16")
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--joint", action="store_true", help="cross-entropy + the layers' compressor losses (loss_type 'both')")
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--kv-mode", choices=("active", "all"), default="active",
                help="'all': query-only pruning, skipped tokens stay keys / values (psv_set_kv_mode)")
ap.add_argument("--mt", type=float, default=0.5, help="mlp_threshold (0.0: every token active)")
ap.add_argument("--criterion", choices=("mlp", "similarity"), default="mlp",
                help="'similarity': each layer's dense pass decides, mask = [1, sim < st] (psv_set_skip_criterion)")
ap.add_argument("--st", type=float, default=0.9, help="sim_threshold of the similarity criterion")
ap.add_argument("--u8", action="store_true", help="raw uint8 [B, 224, 224, 3] images instead of fp32 pixel_values")
args = ap.parse_args()
geom_name, geom = GEOMS[args.geom]
B = args.batch
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"
eng = psv_native.Engine(geom, "fp32", max_batch=B)
eng.load_state_dict(synth.make_state_dict(geom, seed=42))
eng.set_kv_mode(args.kv_mode)
eng.set_skip_criterion(args.criterion, args.st)
if args.u8:
    eng.set_u8_input(geom.image, geom.image)
    x = torch.randint(0, 256, (B, geom.image, geom.image, 3), dtype=torch.uint8,
                      generator=torch.Generator().manual_seed(1234)).cuda()
else:
    x = synth.make_pixels(B, geom, seed=1234).cuda()
dlog = torch.randn(B, geom.classes, device="cuda") / B
dls = torch.ones(geom.layers, device="cuda")
ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
best_f = best_b = 1e9
active = None
for it in range(args.steps + 1):
    ev[0].record()
    eng.backbone_forward_train(x, args.mt, with_layer_losses=args.joint)
    ev[1].record()
    eng.backbone_backward(dlog, dls if args.joint else None)
    ev[2].record()
    torch.cuda.synchronize()
    if it:
        if active is None:
            active = float(eng.backbone_train_masks()[:, :, 1:].float().mean())
        best_f = min(best_f, ev[0].elapsed_time(ev[1]))
        best_b = min(best_b, ev[1].elapsed_time(ev[2]))
crit = f" similarity st {args.st}" if args.criterion == "similarity" else ""
print(f"fine-tune step {geom_name} batch {B}{' joint' if args.joint else ''}{' u8' if args.u8 else ''} kv_mode {args.kv_mode} "
      f"mt {args.mt}{crit} ({active:.0%} of patch tokens active): "
      f"forward {best_f:.1f} ms, backward {best_b:.1f} ms, total {best_f + best_b:.1f} ms -> "
      f"{B / (best_f + best_b) * 1e3:.0f} img/s  [{torch.cuda.get_device_name()}, power limit {power}]")
eng.close()
