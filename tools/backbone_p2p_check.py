"""Data-parallel backbone fine-tuning: BackboneTrainer's sharded peer-memory step ("p2p-fused") and its NCCL form
against today's torch DDP + torch.optim.Adam on the drop-in model.  Run under torchrun on >= 2 GPUs of one node:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29547 \\
        tools/backbone_p2p_check.py [--geom vitb16] [--batch 64] [--steps 10] [--train-precision split] \\
        [--layer-decay 0.75] [--max-grad-norm 1.0]

Checks (exit code 1 on failure): replicas bit-identical after 3 steps with each exchange; the p2p-fused weights
bit-equal to a single-process emulation (the same gradient buckets all-gathered, summed in rank order in fp32, then
backbone_adam_step); p2p-fused against nccl within 1e-5 of max|p| (their summation orders differ); a checkpoint saved at
world 2 loaded into a world-1 trainer gives equal moments.  Prints one JSON line with the ms per step of each.
With --layer-decay / --max-grad-norm the trainers run with backbone_param_groups (weight decay 0.05) and global-norm
clipping: the p2p-fused step is then the three-barrier form (reduce + partial sum of squares, clipped update, gather).
Its fp64 partial sums are grouped per rank, so it is checked against the emulation (backbone_adam_step_groups on the
rank-order sum) within 8 ulps of max|p| and on the norm to 1e-12 relative instead of bit for bit."""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vit-pruning_b200"), ROOT]
import torch
import torch.distributed as dist
import psv_native, synth, main_model_utils

GEOMS = {"vitb16": synth.VIT_B16, "deits16": synth.DEIT_S16, "vitl16": synth.VIT_L16}


def timed(fn, steps):
    torch.cuda.synchronize(); dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    t = torch.tensor([ev0.elapsed_time(ev1) / steps], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--geom", choices=sorted(GEOMS), default="vitb16")
    ap.add_argument("--batch", type=int, default=64, help="images per GPU")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--train-precision", choices=("split", "bf16"), default="split")
    ap.add_argument("--layer-decay", type=float, default=None, help="parameter groups with this layer-wise lr decay")
    ap.add_argument("--max-grad-norm", type=float, default=None, help="global-norm gradient clipping")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    geom = GEOMS[args.geom]
    sd = synth.make_state_dict(geom, 42)
    B = args.batch
    x = synth.make_pixels(B, geom, seed=99 + rank).cuda()
    y = torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(rank)).cuda()
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(local)],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    result = {"n_gpus": world, "geom": args.geom, "batch_per_gpu": B, "train_precision": args.train_precision,
              "gpu": torch.cuda.get_device_name(), "power_limit": power, "layer_decay": args.layer_decay,
              "max_grad_norm": args.max_grad_norm}
    grouped = args.layer_decay is not None or args.max_grad_norm is not None
    ok = True
    params, states = {}, {}
    for kind in ("p2p-fused", "nccl"):
        eng = psv_native.Engine(geom, "fp32", B)
        eng.load_state_dict(sd)
        eng.set_train_precision(args.train_precision)
        groups = (main_model_utils.backbone_param_groups(list(eng.backbone_grad_slices()), geom.layers, 0.05,
                                                         layer_decay=args.layer_decay) if grouped else None)
        tr = main_model_utils.BackboneTrainer(eng, mlp_threshold=0.5, lr=1e-4, weight_decay=0.05, collective=kind,
                                              param_groups=groups, max_grad_norm=args.max_grad_norm)
        assert tr.collective == kind, (tr.collective, tr.collective_note)
        if kind == "p2p-fused":
            # emulation: the same buckets, gathered and summed in rank order in fp32, then the local step
            emu = psv_native.Engine(geom, "fp32", B)
            emu.load_state_dict(sd)
            norm_diff = 0.0
        for _ in range(3):
            tr.step(x, y)
            if kind == "p2p-fused":
                torch.cuda.synchronize(); dist.barrier()
                parts = [torch.empty_like(tr._gbuf) for _ in range(world)]
                dist.all_gather(parts, tr._gbuf.clone())
                s = parts[0].clone()
                for p in parts[1:]:
                    s += p
                if grouped:
                    keys = list(groups)
                    out = torch.zeros(1, device="cuda", dtype=torch.float64)
                    emu.backbone_adam_step_groups(s, tr.steps, lr={k: 1e-4 * groups[k][0] for k in keys},
                                                  weight_decay={k: groups[k][1] for k in keys}, grad_scale=1.0 / world,
                                                  max_grad_norm=args.max_grad_norm, grad_norm_out=out)
                    if args.max_grad_norm is not None:
                        norm_diff = max(norm_diff, abs(float(out) - float(tr.last_grad_norm)) / float(out))
                else:
                    emu.backbone_adam_step(s, tr.steps, lr=1e-4, weight_decay=0.05,
                                           grad_scale=1.0 / world)
        p3 = eng.get_backbone_params().clone()
        pall = [torch.empty_like(p3) for _ in range(world)]
        dist.all_gather(pall, p3)
        result[f"replicas_identical_{kind}"] = all(torch.equal(pall[0], q) for q in pall[1:])
        ok &= result[f"replicas_identical_{kind}"]
        if kind == "p2p-fused":
            want = emu.get_backbone_params()
            if args.max_grad_norm is not None:
                ulps = float((p3 - want).abs().max()) / (2.0 ** -23 * float(want.abs().max()))
                result["p2p_vs_emulation_ulps_of_max_abs"] = ulps
                result["p2p_vs_emulation_norm_rel"] = norm_diff
                ok &= ulps <= 8.0 and norm_diff <= 1e-12
            else:
                result["p2p_equals_emulation"] = bool(torch.equal(p3, want))
                ok &= result["p2p_equals_emulation"]
            states[kind] = tr.state_dict()
            emu.close()
        params[kind] = p3
        result[f"ms_per_step_{kind}"] = timed(lambda: tr.step(x, y), args.steps)
        eng.close()
    d = float((params["p2p-fused"] - params["nccl"]).abs().max())
    result["max_abs_diff_p2p_vs_nccl"] = d
    result["max_abs_param"] = float(params["nccl"].abs().max())
    ok &= d <= 1e-5 * result["max_abs_param"]
    # a world-2 checkpoint loads into a world-1 trainer with equal moments
    st = states["p2p-fused"]
    solo = [dist.new_group([r]) for r in range(world)]          # every rank creates every group
    eng1 = psv_native.Engine(geom, "fp32", B)
    eng1.load_state_dict(sd)
    tr1 = main_model_utils.BackboneTrainer(eng1, process_group=solo[rank])
    tr1.load_state_dict(st)
    m1, v1 = eng1.get_backbone_adam_state()
    result["checkpoint_moments_equal"] = bool(torch.equal(m1.cpu(), st["exp_avg"]) and torch.equal(v1.cpu(), st["exp_avg_sq"])
                                              and torch.equal(eng1.get_backbone_params().cpu(), st["params"]))
    ok &= result["checkpoint_moments_equal"]
    eng1.close()
    # today: the drop-in model under torch DDP + torch.optim.Adam
    import model_utils
    from transformers.models.vit.modeling_vit import ViTConfig
    cfg = ViTConfig(hidden_size=geom.hidden, num_attention_heads=geom.heads, intermediate_size=geom.ffn,
                    num_hidden_layers=geom.layers)
    cfg.num_labels = geom.classes
    model = model_utils.ModifiedViTModel(cfg, 0.9, 0.5, 0)
    model.load_state_dict(sd, strict=False)
    model = model.cuda()
    model.psv_precision = "fp32"
    model.psv_train_precision = args.train_precision
    model.train(); model.vit_train()
    ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=True)
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4)

    def ddp_step():
        loss = torch.nn.functional.cross_entropy(ddp(x).logits, y)
        opt.zero_grad()
        loss.backward()
        opt.step()
    for _ in range(2):
        ddp_step()
    result["ms_per_step_torch_ddp_adam"] = timed(ddp_step, args.steps)
    result["ok"] = bool(ok)
    if rank == 0:
        print(json.dumps(result))
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
