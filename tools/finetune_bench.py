"""Time of one backbone fine-tuning step through the C ABI (psv_backbone_forward_train + psv_backbone_backward), ViT-B/16
by default: forward and backward separately, in the split (fp32-exact) or the mixed-precision bf16 arithmetic.
usage: python tools/finetune_bench.py [--geom vitb16|deits16|vitl16] [--batch 64] [--joint] [--kv-mode {active,all}] [--mt 0.5]
                                     [--criterion {mlp,similarity}] [--st 0.9] [--u8] [--train-precision {split,bf16}]
                                     [--launches] [--optimizer {none,torch,native} ...] [--max-grad-norm 1.0]
                                     [--layer-decay 0.75]
Prints the GPU's name and power limit with the result, since the time depends on both, and the size of the activations
the forward keeps for the backward.  --launches: also one profiled step (torch.profiler, after the timed ones), its
kernels aggregated by name: launches, total us, share of the kernel time.
--optimizer torch native: whole training steps instead (cross-entropy on random labels, Adam lr 1e-4), the listed ways
alternating step by step in one process: `torch` is the drop-in model as a user runs it today (model(x) -- which reloads
the weights the previous step changed --, CrossEntropyLoss, backward, torch.optim.Adam.step()); `native` is
BackboneTrainer.step's sequence (training forward + cross-entropy, psv_backbone_backward, psv_backbone_adam_step).
Prints forward, backward, optimizer and total ms (best of --steps) for each.  With `native`, --max-grad-norm and / or
--layer-decay add a third way, `native-groups`: the same step through psv_backbone_adam_step_groups with
backbone_param_groups (weight decay 0.05, the given layer decay) and global-norm clipping, so the optimizer time is
printed with and without them from one run."""
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
ap.add_argument("--train-precision", choices=("split", "bf16"), default="split",
                help="'bf16': mixed precision, one bf16 tensor-core pass per GEMM (psv_set_train_precision)")
ap.add_argument("--launches", action="store_true", help="print the per-kernel list of one profiled step")
ap.add_argument("--optimizer", nargs="+", choices=("none", "torch", "native"), default=["none"],
                help="time whole steps with the optimizer: torch (drop-in + torch.optim.Adam) and / or native")
ap.add_argument("--max-grad-norm", type=float, default=None, help="--optimizer native: also time clipped steps")
ap.add_argument("--layer-decay", type=float, default=None, help="--optimizer native: also time layer-decay groups")
args = ap.parse_args()
geom_name, geom = GEOMS[args.geom]
B = args.batch
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"
if args.optimizer != ["none"]:
    if "none" in args.optimizer or args.joint or args.u8 or args.launches:
        sys.exit("--optimizer torch/native times plain cross-entropy steps on fp32 pixel_values")
    import model_utils  # noqa: E402
    from main_model_utils import BackboneTrainer  # noqa: E402
    from transformers.models.vit.modeling_vit import ViTConfig  # noqa: E402
    sd = synth.make_state_dict(geom, seed=42)
    x = synth.make_pixels(B, geom, seed=1234).cuda()
    y = torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(0)).cuda()
    runners = {}
    if "torch" in args.optimizer:
        cfg = ViTConfig(hidden_size=geom.hidden, num_attention_heads=geom.heads, intermediate_size=geom.ffn,
                        num_hidden_layers=geom.layers)
        cfg.num_labels = geom.classes
        model = model_utils.ModifiedViTModel(cfg, args.st, args.mt, 0)
        model.load_state_dict(sd, strict=False)
        model = model.cuda()
        model.psv_precision, model.psv_train_precision, model.kv_mode = "fp32", args.train_precision, args.kv_mode
        model.skip_criterion = args.criterion
        model.train(); model.vit_train()
        opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4)

        def torch_step(ev):
            ev[0].record()
            logits = model(x).logits
            ev[1].record()
            loss = torch.nn.functional.cross_entropy(logits, y)
            opt.zero_grad()
            loss.backward()
            ev[2].record()
            opt.step()
            ev[3].record()
        runners["torch"] = torch_step
    if "native" in args.optimizer:
        eng = psv_native.Engine(geom, "fp32", max_batch=B)
        eng.load_state_dict(sd)
        eng.set_kv_mode(args.kv_mode)
        eng.set_skip_criterion(args.criterion, args.st)
        eng.set_train_precision(args.train_precision)
        tr = BackboneTrainer(eng, mlp_threshold=args.mt, lr=1e-4)

        def native_step(ev):                      # BackboneTrainer.step at world 1, with events between its stages
            live = tr._advance()
            ev[0].record()
            lg = eng.backbone_forward_train(x, args.mt).requires_grad_(True)
            dl, = torch.autograd.grad(torch.nn.functional.cross_entropy(lg, y), lg)
            ev[1].record()
            g = eng.backbone_backward(dl)
            ev[2].record()
            eng.backbone_adam_step(g, live, lr=1e-4)
            ev[3].record()
        runners["native"] = native_step
        if args.max_grad_norm is not None or args.layer_decay is not None:
            from main_model_utils import backbone_param_groups  # noqa: E402
            eng2 = psv_native.Engine(geom, "fp32", max_batch=B)
            eng2.load_state_dict(sd)
            eng2.set_kv_mode(args.kv_mode)
            eng2.set_skip_criterion(args.criterion, args.st)
            eng2.set_train_precision(args.train_precision)
            keys = list(eng2.backbone_grad_slices())
            groups = backbone_param_groups(keys, geom.layers, 0.05, layer_decay=args.layer_decay)
            tr2 = BackboneTrainer(eng2, mlp_threshold=args.mt, lr=1e-4)
            lrs = {k: 1e-4 * groups[k][0] for k in keys}
            wds = {k: groups[k][1] for k in keys}
            norm = torch.zeros(1, device="cuda", dtype=torch.float64)

            def grouped_step(ev):                 # BackboneTrainer(param_groups=, max_grad_norm=).step's sequence
                live = tr2._advance()
                ev[0].record()
                lg = eng2.backbone_forward_train(x, args.mt).requires_grad_(True)
                dl, = torch.autograd.grad(torch.nn.functional.cross_entropy(lg, y), lg)
                ev[1].record()
                g = eng2.backbone_backward(dl)
                ev[2].record()
                eng2.backbone_adam_step_groups(g, live, lr=lrs, weight_decay=wds, max_grad_norm=args.max_grad_norm,
                                               grad_norm_out=norm if args.max_grad_norm is not None else None)
                ev[3].record()
            runners["native-groups"] = grouped_step
    best = {k: [1e9] * 4 for k in runners}
    for it in range(args.steps + 1):
        for k, fn in runners.items():
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            fn(ev)
            torch.cuda.synchronize()
            if it:
                t = [ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]), ev[0].elapsed_time(ev[3])]
                best[k] = [min(a, b) for a, b in zip(best[k], t)]
    for k, (f, b, o, tot) in best.items():
        print(f"optimizer {k}: {geom_name} batch {B} {args.train_precision} kv_mode {args.kv_mode} mt {args.mt}: forward "
              f"{f:.2f} ms{' (incl. weight reload)' if k == 'torch' else ''}, backward {b:.2f} ms, optimizer {o:.2f} ms, "
              f"total {tot:.2f} ms  [{torch.cuda.get_device_name()}, power limit {power}]"
              + (f"  (layer decay {args.layer_decay}, max_grad_norm {args.max_grad_norm})" if k == "native-groups" else ""))
    sys.exit(0)
eng = psv_native.Engine(geom, "fp32", max_batch=B)
eng.load_state_dict(synth.make_state_dict(geom, seed=42))
eng.set_kv_mode(args.kv_mode)
eng.set_skip_criterion(args.criterion, args.st)
eng.set_train_precision(args.train_precision)
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
            masks = eng.backbone_train_masks()
            active = float(masks[:, :, 1:].float().mean())
            T = masks.reshape(geom.layers, -1).sum(1).double()
            # kept per layer: x0, x1 fp32 [T, D], u fp32 [T, F]; a1, ctx, a2 [T, D] and q|k|v [T, 3D] fp32 (split) or
            # bf16 plus the attention log-sum-exp fp32 [T, heads] (bf16)
            D, Fw, H = geom.hidden, geom.ffn, geom.heads
            fp32_part = float((T * (2 * D + Fw)).sum()) * 4
            split_mb = (fp32_part + float((T * 6 * D).sum()) * 4) / 2 ** 20
            bf16_mb = (fp32_part + float((T * 6 * D).sum()) * 2 + float((T * H).sum()) * 4) / 2 ** 20
        best_f = min(best_f, ev[0].elapsed_time(ev[1]))
        best_b = min(best_b, ev[1].elapsed_time(ev[2]))
crit = f" similarity st {args.st}" if args.criterion == "similarity" else ""
print(f"fine-tune step {geom_name} batch {B} {args.train_precision}{' joint' if args.joint else ''}{' u8' if args.u8 else ''} "
      f"kv_mode {args.kv_mode} "
      f"mt {args.mt}{crit} ({active:.0%} of patch tokens active): "
      f"forward {best_f:.1f} ms, backward {best_b:.1f} ms, total {best_f + best_b:.1f} ms -> "
      f"{B / (best_f + best_b) * 1e3:.0f} img/s  [{torch.cuda.get_device_name()}, power limit {power}]; saved activations "
      f"{bf16_mb if args.train_precision == 'bf16' else split_mb:.0f} MiB (split {split_mb:.0f}, bf16 {bf16_mb:.0f})")
if args.launches:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.backbone_forward_train(x, args.mt, with_layer_losses=args.joint)
        eng.backbone_backward(dlog, dls if args.joint else None)
        torch.cuda.synchronize()
    agg = {}
    for ev_ in prof.events():
        if ev_.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in ev_.name.lower() \
                and "memset" not in ev_.name.lower():
            name = ev_.name.replace("(anonymous namespace)::", "").replace("psv::", "").replace("void ", "")
            name = name.split("(")[0]
            n, t = agg.get(name, (0, 0.0))
            agg[name] = (n + 1, t + ev_.device_time_total)
    total = sum(t for _, t in agg.values())
    print(f"{sum(n for n, _ in agg.values())} launches, {total:.1f} us of kernel time")
    for name, (n, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print(f"{name[:66]:66s} {n:5d} {t:10.1f}  {t / total:.3f}")
eng.close()
