"""Parameter groups and global-norm gradient clipping of the native backbone optimizer (psv_backbone_adam_step_groups,
the sharded psv_backbone_peer_reduce_sqnorm + psv_backbone_peer_adam_step_groups, the clipped compressor steps,
main_model_utils.backbone_param_groups and BackboneTrainer(param_groups=, max_grad_norm=)).

CPU: the group helper against the rules restated here; an fp64 model of clipped, grouped AdamW against
torch.optim.AdamW(param_groups) + clip_grad_norm_, and planted defects in it, each at least 2x the GPU bar.
GPU: the default groups are today's step bit for bit; the norm; five steps against torch on DeiT-S and ViT-B; the
sharded clipped step; graph capture; BackboneTrainer against the drop-in; checkpoint resume; refusals; two GPUs."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import synth

# the bar of the plain step: |native - torch| <= ULP_BAR * 2^-23 * max|p| per tensor
ULP_BAR = 8.0
EPS32 = 2.0 ** -23
LR = 1e-3
LAYER_DECAY, WD = 0.75, 0.05


def _keys_and_shapes(geom):
    """The backbone state-dict keys and shapes, restated from the reference model (HF ViTForImageClassification)."""
    D, F, N = geom.hidden, geom.ffn, geom.tokens
    out = {"embeddings.cls_token": (1, 1, D), "embeddings.position_embeddings": (1, N, D),
           "embeddings.patch_embeddings.projection.weight": (D, geom.channels, geom.patch, geom.patch),
           "embeddings.patch_embeddings.projection.bias": (D,)}
    for i in range(geom.layers):
        p = f"encoder.layer.{i}."
        for name, shape in (("layernorm_before.weight", (D,)), ("layernorm_before.bias", (D,)),
                            ("attention.attention.query.weight", (D, D)), ("attention.attention.key.weight", (D, D)),
                            ("attention.attention.value.weight", (D, D)), ("attention.attention.query.bias", (D,)),
                            ("attention.attention.key.bias", (D,)), ("attention.attention.value.bias", (D,)),
                            ("attention.output.dense.weight", (D, D)), ("attention.output.dense.bias", (D,)),
                            ("layernorm_after.weight", (D,)), ("layernorm_after.bias", (D,)),
                            ("intermediate.dense.weight", (F, D)), ("intermediate.dense.bias", (F,)),
                            ("output.dense.weight", (D, F)), ("output.dense.bias", (D,))):
            out[p + name] = shape
    out.update({"layernorm.weight": (D,), "layernorm.bias": (D,), "classifier.weight": (geom.classes, D),
                "classifier.bias": (geom.classes,)})
    return out


# ------------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("geom", [synth.DEIT_S16, synth.VIT_B16, synth.VIT_L16], ids=["deits16", "vitb16", "vitl16"])
def test_group_helper_follows_the_rules(geom):
    from main_model_utils import backbone_param_groups
    shapes = _keys_and_shapes(geom)
    L = geom.layers
    groups = backbone_param_groups(list(shapes), L, WD, layer_decay=LAYER_DECAY)
    assert set(groups) == set(shapes)
    for k, shape in shapes.items():
        decays = len(shape) > 1 and k not in ("embeddings.cls_token", "embeddings.position_embeddings")
        if k.startswith("encoder.layer."):
            lid = int(k.split(".")[2]) + 1
        elif k.startswith("embeddings."):
            lid = 0
        else:
            lid = L + 1
        assert groups[k] == (pytest.approx(LAYER_DECAY ** (L + 1 - lid), rel=1e-15), WD if decays else 0.0), k
    for q in ("query", "key", "value"):
        assert groups[f"encoder.layer.0.attention.attention.{q}.bias"] == (pytest.approx(LAYER_DECAY ** L), 0.0)
    assert groups["embeddings.patch_embeddings.projection.weight"] == (pytest.approx(LAYER_DECAY ** (L + 1)), WD)
    assert groups["embeddings.cls_token"][1] == 0.0 and groups["embeddings.position_embeddings"][1] == 0.0
    for k in ("layernorm.weight", "layernorm.bias", "classifier.bias"):
        assert groups[k] == (1.0, 0.0)
    assert groups["classifier.weight"] == (1.0, WD)
    assert groups[f"encoder.layer.{L - 1}.output.dense.weight"] == (pytest.approx(LAYER_DECAY), WD)
    flat = backbone_param_groups(list(shapes), L, WD)
    assert all(s == 1.0 for s, _ in flat.values())


def _clip_adamw_fp64(params, grads_seq, live_seq, lrs, wds, max_norm, betas=(0.9, 0.999), eps=1e-8, defect=None):
    """fp64 AdamW with per-tensor lr / weight decay, per-tensor steps (live_seq: frozen tensors get no gradient) and
    clip_grad_norm_ over the live tensors; `defect` plants one known mistake."""
    b1, b2 = betas
    p = [x.clone() for x in params]
    m = [torch.zeros_like(x) for x in params]
    v = [torch.zeros_like(x) for x in params]
    steps = [0] * len(params)
    for grads, live in zip(grads_seq, live_seq):
        counted = range(len(p)) if defect == "norm_over_frozen" else [i for i in range(len(p)) if live[i]]
        norm = math.sqrt(sum(float(grads[i].pow(2).sum()) for i in counted))
        coef = max_norm / (norm + 1e-6)
        if defect != "unclamped":
            coef = min(coef, 1.0)
        for i, g in enumerate(grads):
            if not live[i]:
                continue
            steps[i] += 1
            st = steps[i]
            lr, wd = lrs[i], wds[i]
            if defect == "decay_no_decay" and wd == 0.0:
                wd = WD
            if defect == "layer_off_by_one":
                lr = lr * LAYER_DECAY
            gc = g if defect == "clip_after_moments" else g * coef
            p[i] = p[i] * (1 - lr * wd)
            m[i] = b1 * m[i] + (1 - b1) * gc
            v[i] = b2 * v[i] + (1 - b2) * gc * gc
            bc1, bc2 = 1 - b1 ** st, 1 - b2 ** st
            upd = lr / bc1 * m[i] / (v[i].sqrt() / bc2 ** 0.5 + eps)
            p[i] = p[i] - (upd * coef if defect == "clip_after_moments" else upd)
    return p


def _torch_clip_adamw(params, grads_seq, live_seq, lrs, wds, max_norm):
    p = [x.clone().requires_grad_(True) for x in params]
    opt = torch.optim.AdamW([{"params": [x], "lr": lr, "weight_decay": wd} for x, lr, wd in zip(p, lrs, wds)],
                            foreach=False)
    for grads, live in zip(grads_seq, live_seq):
        for x, g, on in zip(p, grads, live):
            x.grad = g.clone() if on else None
        torch.nn.utils.clip_grad_norm_([x for x in p if x.grad is not None], max_norm, foreach=False)
        opt.step()
    return [x.detach() for x in p]


def _cpu_case():
    gen = torch.Generator().manual_seed(11)
    # (shape, |p|, |g|, layer id, decays): two "layers" of a weight and a bias, a frozen-then-trained embedding
    spec = [((64, 48), 0.02, 1e-3, 1, True), ((48,), 1.0, 1e-3, 1, False), ((32, 32), 0.05, 1e-2, 2, True),
            ((96,), 0.1, 1e-4, 2, False), ((40, 8), 0.02, 5e-3, 0, False)]
    params = [torch.randn(s, generator=gen, dtype=torch.float64) * sp for s, sp, *_ in spec]
    step_scale = (0.3, 3.0, 1.0, 0.5, 2.0)          # the clip binds on some steps and not on others
    grads_seq = [[torch.randn(s, generator=gen, dtype=torch.float64) * sg * f for s, _, sg, *_ in spec]
                 for f in step_scale]
    live_seq = [[1, 1, 1, 1, 0]] * 2 + [[1, 1, 1, 1, 1]] * 3
    lrs = [LR * LAYER_DECAY ** (3 - lid) for *_, lid, _ in spec]
    wds = [WD if dec else 0.0 for *_, dec in spec]
    norms = [math.sqrt(sum(float(g.pow(2).sum()) for g, on in zip(gs, live) if on)) for gs, live in zip(grads_seq, live_seq)]
    max_norm = sorted(norms)[2]
    assert any(n > max_norm for n in norms) and any(n < max_norm for n in norms)
    return params, grads_seq, live_seq, lrs, wds, max_norm


def _worst_ulps(got, ref):
    return max(float((a - b).abs().max()) / (EPS32 * float(b.abs().max())) for a, b in zip(got, ref))


def test_fp64_model_matches_torch_and_planted_defects_exceed_the_bar():
    params, grads_seq, live_seq, lrs, wds, max_norm = _cpu_case()
    ref = _torch_clip_adamw(params, grads_seq, live_seq, lrs, wds, max_norm)
    assert _worst_ulps(_clip_adamw_fp64(params, grads_seq, live_seq, lrs, wds, max_norm), ref) < 1e-6 * ULP_BAR
    for d in ("norm_over_frozen", "clip_after_moments", "decay_no_decay", "layer_off_by_one", "unclamped"):
        err = _worst_ulps(_clip_adamw_fp64(params, grads_seq, live_seq, lrs, wds, max_norm, defect=d), ref)
        assert err >= 2 * ULP_BAR, (d, err)


# ------------------------------------------------------------------------------------------------------------------ GPU
def _engine(geom, sd, batch=8, precision="fp32"):
    import psv_native
    e = psv_native.Engine(geom, precision, batch)
    e.load_state_dict(sd)
    return e


def _grad_sequence(geom, sd, batch=8, k=5):
    """k real backward gradients (cross-entropy on random labels, different batches, fixed weights)."""
    e = _engine(geom, sd, batch)
    seq = []
    for i in range(k):
        x = synth.make_pixels(batch, geom, seed=700 + i, kind="randn").cuda()
        y = torch.randint(0, geom.classes, (batch,), generator=torch.Generator().manual_seed(70 + i)).cuda()
        lg = e.backbone_forward_train(x, 0.5).detach().requires_grad_(True)
        dl, = torch.autograd.grad(torch.nn.functional.cross_entropy(lg, y), lg)
        seq.append(e.backbone_backward(dl).clone())
    torch.cuda.synchronize()
    e.close()
    return seq


@pytest.fixture(scope="module")
def deits(state_dicts):
    geom, sd = state_dicts("deits16")
    return geom, sd, _grad_sequence(geom, sd)


@pytest.fixture(scope="module")
def vitb(state_dicts):
    geom, sd = state_dicts("vitb16")
    return geom, sd, _grad_sequence(geom, sd, k=5)


def _groups(e):
    from main_model_utils import backbone_param_groups
    keys = list(e.backbone_grad_slices())
    return keys, backbone_param_groups(keys, e.geom.layers, WD, layer_decay=LAYER_DECAY)


def _fp64_norm(g, slices, live, grad_scale=1.0):
    tot = 0.0
    for (k, (off, shape)), on in zip(slices.items(), live):
        if on:
            tot += float((g[off:off + int(np.prod(shape))] * grad_scale).double().pow(2).sum())
    return math.sqrt(tot)


@pytest.mark.gpu
def test_default_groups_are_todays_step(deits):
    """All lr equal, uniform weight decay, no clipping: the grouped local and sharded steps give the weights and
    moments of psv_backbone_adam_step / psv_backbone_peer_reduce_adam_step bit for bit."""
    geom, sd, seq = deits
    a, b = _engine(geom, sd), _engine(geom, sd)
    nt = len(a.backbone_grad_slices())
    for t, g in enumerate(seq):
        a.backbone_adam_step(g, [t + 1] * nt, lr=LR, weight_decay=WD, grad_scale=0.5)
        b.backbone_adam_step_groups(g, [t + 1] * nt, lr=[LR] * nt, weight_decay=WD, grad_scale=0.5)
    assert torch.equal(a.get_backbone_params(), b.get_backbone_params())
    for x, y in zip(a.get_backbone_adam_state(), b.get_backbone_adam_state()):
        assert torch.equal(x, y)
    world = 2
    old, new = [_engine(geom, sd) for _ in range(world)], [_engine(geom, sd) for _ in range(world)]
    n = a.backbone_param_count
    gbufs = [torch.empty(n + 4, device="cuda") for _ in range(world)]
    pbufs = {k: [torch.zeros(n + 4, device="cuda") for _ in range(world)] for k in ("old", "new")}
    for t in range(3):
        for r in range(world):
            gbufs[r][:n].copy_(seq[(t + r) % len(seq)])
        gp = [x.data_ptr() for x in gbufs]
        for r in range(world):
            old[r].backbone_peer_reduce_adam_step(gp, pbufs["old"][r], r, [t + 1] * nt, lr=LR, weight_decay=WD,
                                                  grad_scale=0.5)
            new[r].backbone_peer_adam_step_groups(gp, pbufs["new"][r], r, [t + 1] * nt, lr=LR, weight_decay=[WD] * nt,
                                                  grad_scale=0.5)
        for r in range(world):
            old[r].backbone_peer_gather_params([x.data_ptr() for x in pbufs["old"]], r)
            new[r].backbone_peer_gather_params([x.data_ptr() for x in pbufs["new"]], r)
    for r in range(world):
        assert torch.equal(old[r].get_backbone_params(), new[r].get_backbone_params())
        for x, y in zip(old[r].get_backbone_adam_state(), new[r].get_backbone_adam_state()):
            assert torch.equal(x, y)
    for e in [a, b] + old + new:
        e.close()


@pytest.mark.gpu
def test_norm_is_exact_deterministic_and_ignores_frozen(deits):
    geom, sd, seq = deits
    e = _engine(geom, sd)
    slices = e.backbone_grad_slices()
    keys = list(slices)
    nt = len(keys)
    live = [0 if k.startswith("embeddings.") else 1 for k in keys]
    g = seq[1]
    outs = []
    for _ in range(2):
        out = torch.zeros(1, device="cuda", dtype=torch.float64)
        e.backbone_adam_step_groups(g, live, lr=0.0, grad_scale=0.37, grad_norm_out=out)
        outs.append(out.clone())
    assert torch.equal(outs[0], outs[1])
    want = _fp64_norm(g, slices, live, 0.37)
    # the scaled gradient is rounded to fp32 before squaring, as in the kernel
    got = float(outs[0])
    assert abs(got - want) <= 1e-9 * want, (got, want)
    g2 = g.clone()
    lo = slices["encoder.layer.0.layernorm_before.weight"][0]
    g2[:lo] = 1e3                                                  # frozen tensors: no effect on the norm
    out = torch.zeros(1, device="cuda", dtype=torch.float64)
    e.backbone_adam_step_groups(g2, live, lr=0.0, grad_scale=0.37, grad_norm_out=out)
    assert torch.equal(out, outs[0])
    e.close()


def _torch_clip_steps(sd, slices, seq, live_seq, lrs, wds, max_norm):
    keys = list(slices)
    p = {k: sd[k].detach().float().cuda().clone().requires_grad_(True) for k in keys}
    opt = torch.optim.AdamW([{"params": [p[k]], "lr": lrs[k], "weight_decay": wds[k]} for k in keys], foreach=False)
    norms = []
    for g, live in zip(seq, live_seq):
        for k, on in zip(keys, live):
            off, shape = slices[k]
            p[k].grad = g[off:off + int(np.prod(shape))].reshape(p[k].shape).clone() if on else None
        norms.append(float(torch.nn.utils.clip_grad_norm_([x for x in p.values() if x.grad is not None], max_norm,
                                                          foreach=False)))
        opt.step()
    return {k: v.detach() for k, v in p.items()}, norms


def _compare(e, ref, label):
    got = e.export_backbone_state_dict()
    worst = 0.0
    for k, r in ref.items():
        if not float(r.abs().max()):                   # an all-zero tensor (a frozen zero-initialised bias) stays so
            assert torch.equal(got[k].reshape(r.shape), r), (label, k)
            continue
        ulps = float((got[k].reshape(r.shape) - r).abs().max()) / (EPS32 * float(r.abs().max()))
        worst = max(worst, ulps)
        assert ulps <= ULP_BAR, (label, k, ulps)
    print(f"{label}: worst {worst:.2f} ulps of max|p| (bar {ULP_BAR})")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["deits", "vitb", "deits-classifier-first"])
def test_five_clipped_grouped_steps_match_torch(request, case):
    geom, sd, seq = request.getfixturevalue(case.split("-")[0])
    e = _engine(geom, sd)
    slices = e.backbone_grad_slices()
    keys, groups = _groups(e)
    lrs = {k: LR * groups[k][0] for k in keys}
    wds = {k: groups[k][1] for k in keys}
    if case.endswith("classifier-first"):
        live_seq = [[int(k.startswith("classifier.")) for k in keys]] * 2 + [[1] * len(keys)] * 3
    else:
        live_seq = [[1] * len(keys)] * 5
    norms = [_fp64_norm(g, slices, live) for g, live in zip(seq, live_seq)]
    max_norm = sorted(norms)[2]
    assert any(n > max_norm * (1 + 1e-6) for n in norms) and any(n < max_norm for n in norms)
    counters = [0] * len(keys)
    before = e.get_backbone_params().clone()
    got_norms = []
    for t, (g, live) in enumerate(zip(seq, live_seq)):
        counters = [c + on for c, on in zip(counters, live)]
        out = torch.zeros(1, device="cuda", dtype=torch.float64)
        e.backbone_adam_step_groups(g, [c if on else 0 for c, on in zip(counters, live)], lr=lrs, weight_decay=wds,
                                    max_grad_norm=max_norm, grad_norm_out=out)
        got_norms.append(float(out))
        if case.endswith("classifier-first") and t == 1:
            lo = slices["classifier.weight"][0]
            m, v = e.get_backbone_adam_state()
            assert torch.equal(e.get_backbone_params()[:lo], before[:lo])
            assert int(torch.count_nonzero(m[:lo])) == 0 and int(torch.count_nonzero(v[:lo])) == 0
    ref, ref_norms = _torch_clip_steps(sd, slices, seq, live_seq, lrs, wds, max_norm)
    for a, b in zip(got_norms, ref_norms):
        assert abs(a - b) <= 1e-5 * b
    _compare(e, ref, case)
    e.close()


def _sharded_clipped(geom, sd, seq, world, steps_fn, lrs, wds, max_norm, grad_scale):
    """`world` engines on one GPU run reduce_sqnorm -> adam_step_groups(peer_sqnorms) -> gather (the peer pointers are
    plain device pointers); returns the engines, their per-step norms and the summed buckets."""
    engines = [_engine(geom, sd) for _ in range(world)]
    n = engines[0].backbone_param_count
    gbufs = [torch.empty(n + 4, device="cuda") for _ in range(world)]
    pbufs = [torch.zeros(n + 4, device="cuda") for _ in range(world)]
    slots = [torch.zeros(1, device="cuda", dtype=torch.float64) for _ in range(world)]
    gp, pp, sp = [x.data_ptr() for x in gbufs], [x.data_ptr() for x in pbufs], [x.data_ptr() for x in slots]
    norms, totals = [], []
    for t in range(3):
        total = None
        for r in range(world):
            gbufs[r][:n].copy_(seq[(t + r) % len(seq)] * (r + 1))
            total = gbufs[r][:n].clone() if total is None else total + gbufs[r][:n]
        totals.append(total)
        steps = steps_fn(t)
        for r, e in enumerate(engines):
            e.backbone_peer_reduce_sqnorm(gp, r, steps, slots[r], grad_scale=grad_scale)
        outs = [torch.zeros(1, device="cuda", dtype=torch.float64) for _ in range(world)]
        for r, e in enumerate(engines):
            e.backbone_peer_adam_step_groups(gp, pbufs[r], r, steps, lr=lrs, weight_decay=wds, grad_scale=grad_scale,
                                             max_grad_norm=max_norm, peer_sqnorms=sp, grad_norm_out=outs[r])
        for r, e in enumerate(engines):
            e.backbone_peer_gather_params(pp, r)
        norms.append(outs)
    return engines, norms, totals


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_clipped_step_on_one_gpu(deits, world):
    geom, sd, seq = deits
    emu = _engine(geom, sd)
    keys, groups = _groups(emu)
    lrs = {k: LR * groups[k][0] for k in keys}
    wds = {k: groups[k][1] for k in keys}

    def steps_fn(t):
        return [0 if k.startswith("embeddings.") else t + 1 for k in keys]
    slices = emu.backbone_grad_slices()
    gs = 1.0 / world
    probe = [_fp64_norm(sum(seq[(t + r) % len(seq)] * (r + 1) for r in range(world)), slices, steps_fn(t), gs)
             for t in range(3)]
    max_norm = sorted(probe)[1]
    engines, norms, totals = _sharded_clipped(geom, sd, seq, world, steps_fn, lrs, wds, max_norm, gs)
    emu_norms = []
    for t, total in enumerate(totals):
        out = torch.zeros(1, device="cuda", dtype=torch.float64)
        emu.backbone_adam_step_groups(total, steps_fn(t), lr=lrs, weight_decay=wds, grad_scale=gs,
                                      max_grad_norm=max_norm, grad_norm_out=out)
        emu_norms.append(float(out))
    want = engines[0].get_backbone_params()
    for e in engines[1:]:
        assert torch.equal(e.get_backbone_params(), want)
    for t, outs in enumerate(norms):
        assert all(torch.equal(o, outs[0]) for o in outs[1:])
        assert abs(float(outs[0]) - emu_norms[t]) <= 1e-12 * emu_norms[t]
    ref = emu.export_backbone_state_dict()
    _compare(engines[0], ref, f"sharded world {world} against the local clipped step")
    lo = slices["encoder.layer.0.layernorm_before.weight"][0]
    assert torch.equal(want[:lo], _engine(geom, sd).get_backbone_params()[:lo])
    for e in engines + [emu]:
        e.close()


@pytest.mark.gpu
def test_clipped_grouped_step_captures_into_a_graph(deits):
    geom, sd, seq = deits
    eager, graphed = _engine(geom, sd), _engine(geom, sd)
    keys, groups = _groups(eager)
    lrs = {k: LR * groups[k][0] for k in keys}
    wds = {k: groups[k][1] for k in keys}
    nt = len(keys)
    max_norm = 0.5 * _fp64_norm(seq[1], eager.backbone_grad_slices(), [1] * nt)
    for e in (eager, graphed):                                  # the first step allocates the moments
        e.backbone_adam_step_groups(seq[0], [1] * nt, lr=lrs, weight_decay=wds, max_grad_norm=max_norm)
    out_e = torch.zeros(1, device="cuda", dtype=torch.float64)
    eager.backbone_adam_step_groups(seq[1], [2] * nt, lr=lrs, weight_decay=wds, max_grad_norm=max_norm,
                                    grad_norm_out=out_e)
    static_g = seq[2].clone()
    out_g = torch.zeros(1, device="cuda", dtype=torch.float64)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.backbone_adam_step_groups(static_g, [2] * nt, lr=lrs, weight_decay=wds, max_grad_norm=max_norm,
                                          grad_norm_out=out_g)
    static_g.copy_(seq[1])
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out_g, out_e)
    assert torch.equal(graphed.get_backbone_params(), eager.get_backbone_params())
    for x, y in zip(graphed.get_backbone_adam_state(), eager.get_backbone_adam_state()):
        assert torch.equal(x, y)
    eager.close()
    graphed.close()


def _drop_in(geom, sd, train_precision, joint):
    import model_utils
    from transformers.models.vit.modeling_vit import ViTConfig
    cfg = ViTConfig(hidden_size=geom.hidden, num_attention_heads=geom.heads, intermediate_size=geom.ffn)
    cfg.num_labels = geom.classes
    model = model_utils.ModifiedViTModel(cfg, 0.9, 0.5, 0)
    model.load_state_dict(sd, strict=False)
    model = model.to("cuda")
    model.psv_precision = "fp32"
    model.psv_train_precision = train_precision
    model.train()
    model.vit_mlp_train() if joint else model.vit_train()
    return model


@pytest.mark.gpu
@pytest.mark.parametrize("train_precision, joint", [("split", False), ("bf16", False), ("split", True)],
                         ids=["split", "bf16", "joint"])
def test_trainer_with_groups_and_clipping_matches_drop_in(state_dicts, train_precision, joint):
    """BackboneTrainer(param_groups, max_grad_norm) against the drop-in trained with torch.optim.AdamW param groups +
    clip_grad_norm_ over every trained parameter (the compressors too in the joint case), within TRAINER_BARS."""
    from main_model_utils import BackboneTrainer, backbone_param_groups
    from test_gpu_backbone_optimizer import TRAINER_BARS
    geom, sd = state_dicts("deits16")
    B, K, lr = 16, 3, 1e-4
    xs = [synth.make_pixels(B, geom, seed=900 + i, kind="randn").cuda() for i in range(K)]
    ys = [torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(90 + i)).cuda() for i in range(K)]
    ref = _drop_in(geom, sd, train_precision, joint)
    named = {k: p for k, p in ref.named_parameters() if p.requires_grad}
    groups = backbone_param_groups([k for k in named if "mlp_layer" not in k], geom.layers, WD,
                                   layer_decay=LAYER_DECAY)
    opt = torch.optim.AdamW([{"params": [p], "lr": lr * groups[k][0] if k in groups else lr,
                              "weight_decay": groups[k][1] if k in groups else 0.0} for k, p in named.items()],
                            foreach=False)
    ref_hist, ref_norms, max_norm = [], [], None
    for x, y in zip(xs, ys):
        loss = torch.nn.CrossEntropyLoss()(ref(x).logits, y)
        if joint:
            loss = loss + sum((layer.loss for layer in ref.encoder.layer), 0.0)
        opt.zero_grad()
        loss.backward()
        if max_norm is None:                                   # binds on the first step
            max_norm = 0.7 * float(torch.nn.utils.get_total_norm([p.grad for p in named.values() if p.grad is not None]))
        ref_norms.append(float(torch.nn.utils.clip_grad_norm_(list(named.values()), max_norm, foreach=False)))
        opt.step()
        ref_hist.append(loss.item())
    model = _drop_in(geom, sd, train_precision, joint)
    eng = model._psv_engine_for(B, xs[0].device)
    tr = BackboneTrainer(eng, mlp_threshold=model.mlp_threshold, lr=lr, joint=joint, param_groups=groups,
                         max_grad_norm=max_norm)
    hist, norms = [], []
    for x, y in zip(xs, ys):
        hist.append(float(tr.step(x, y)))
        norms.append(float(tr.last_grad_norm))
    rel = max(abs(a - b) / abs(b) for a, b in zip(hist, ref_hist))
    norm_rel = max(abs(a - b) / b for a, b in zip(norms, ref_norms))
    init = {k: v.float().cuda() for k, v in sd.items()}
    out = eng.export_backbone_state_dict()
    if joint:
        out.update(eng.export_compressor_state_dict())
    refp = dict(ref.named_parameters())
    num = den = 0.0
    for k, v in out.items():
        num += float((v.reshape(refp[k].shape) - refp[k].detach()).double().pow(2).sum())
        den += float((refp[k].detach() - init[k].reshape(refp[k].shape)).double().pow(2).sum())
    upd = (num / den) ** 0.5
    loss_bar, update_bar = TRAINER_BARS["joint" if joint else train_precision]
    print(f"{train_precision}{' joint' if joint else ''}: loss rel {rel:.2e} (bar {loss_bar}), |dp| / |update| "
          f"{upd:.2e} (bar {update_bar}), norm rel {norm_rel:.2e}, norms {norms} max {max_norm:.4g}")
    assert rel <= loss_bar and upd <= update_bar
    assert norm_rel <= 10 * loss_bar


@pytest.mark.gpu
def test_checkpoint_resume_with_groups_and_clipping(deits):
    """Five clipped grouped steps straight through against three, a checkpoint (the weights, the moments read back in
    two ranges) into a fresh engine, and two more: bit for bit, norms included.  Fixed gradients: the backward
    accumulates with float atomics, so two trainer runs differ in the last bits of every gradient."""
    geom, sd, seq = deits
    straight, first = _engine(geom, sd), _engine(geom, sd)
    keys, groups = _groups(straight)
    lrs = {k: LR * groups[k][0] for k in keys}
    wds = {k: groups[k][1] for k in keys}
    nt = len(keys)
    max_norm = sorted(_fp64_norm(g, straight.backbone_grad_slices(), [1] * nt) for g in seq)[2]

    def step(e, t):
        out = torch.zeros(1, device="cuda", dtype=torch.float64)
        e.backbone_adam_step_groups(seq[t], [t + 1] * nt, lr=lrs, weight_decay=wds, max_grad_norm=max_norm,
                                    grad_norm_out=out)
        return out
    want = [step(straight, t) for t in range(5)]
    for t in range(3):
        step(first, t)
    params, half = first.get_backbone_params(), first.backbone_param_count // 2
    resumed = _engine(geom, {**{k: params[o:o + int(np.prod(sh))].reshape(sh)
                                for k, (o, sh) in first.backbone_grad_slices().items()},
                             **{k: v for k, v in sd.items() if "mlp_layer" in k}})
    for lo, hi in ((0, half), (half, first.backbone_param_count)):
        m, v = first.get_backbone_adam_state(lo, hi)
        resumed.set_backbone_adam_state(m, v, lo=lo)
    got = [step(resumed, t) for t in range(3, 5)]
    assert all(torch.equal(a, b) for a, b in zip(got, want[3:]))
    assert torch.equal(resumed.get_backbone_params(), straight.get_backbone_params())
    for a, b in zip(resumed.get_backbone_adam_state(), straight.get_backbone_adam_state()):
        assert torch.equal(a, b)
    for e in (straight, first, resumed):
        e.close()


@pytest.mark.gpu
def test_refusals(deits):
    import psv_native
    lib = psv_native.lib
    geom, sd, seq = deits
    e = _engine(geom, sd)
    nt = len(e.backbone_grad_slices())
    n = e.backbone_param_count
    g = seq[0]
    s = psv_native._stream()
    steps = (C.c_int32 * nt)(*([1] * nt))
    good = (C.c_float * nt)(*([LR] * nt))
    zero = (C.c_float * nt)(*([0.0] * nt))
    gp = C.c_void_p(g.data_ptr())
    before = e.get_backbone_params().clone()

    def local(grads=gp, st=steps, lr=good, wd=zero, clip=1.0, comp=None):
        return lib.psv_backbone_adam_step_groups(e._h, grads, st, lr, wd, 0.9, 0.999, 1e-8, 1.0, clip, comp, None, s)
    assert local(grads=None) == -1
    mis = torch.zeros(n + 1, device="cuda")[1:]
    assert local(grads=C.c_void_p(mis.data_ptr())) == -1
    assert local(comp=C.c_void_p(mis.data_ptr())) == -1
    assert local(st=None) == -1 and local(lr=None) == -1 and local(wd=None) == -1
    for bad in (-1e-3, float("nan"), float("inf")):
        arr = (C.c_float * nt)(*([LR] * (nt - 1) + [bad]))
        assert local(lr=arr) == -1 and local(wd=arr) == -1, bad
    for bad in (float("nan"), float("inf"), float("-inf")):
        assert local(clip=bad) == -1, bad
    peers = (C.c_void_p * 1)(g.data_ptr())
    bucket = torch.zeros(n + 4, device="cuda")
    slot = torch.zeros(1, device="cuda", dtype=torch.float64)
    slots = (C.c_void_p * 1)(slot.data_ptr())

    def peer(clip=0.0, sq=None, world=1, rank=0):
        return lib.psv_backbone_peer_adam_step_groups(e._h, peers, C.c_void_p(bucket.data_ptr()), world, rank, steps,
                                                      good, zero, 0.9, 0.999, 1e-8, 1.0, clip, sq, None, s)
    assert peer(clip=1.0) == -1                                   # clipping needs the norm pass and its slots
    assert peer(sq=slots) == -3                                   # no reduce_sqnorm before
    assert peer(world=17) == -1 and peer(world=2, rank=2) == -1
    odd = C.c_void_p(slot.data_ptr() + 4)
    assert lib.psv_backbone_peer_reduce_sqnorm(e._h, peers, 1, 0, steps, 1.0, None, odd, s) == -1
    assert lib.psv_backbone_peer_reduce_sqnorm(e._h, peers, 1, 0, steps, 1.0, None, None, s) == -1
    torch.cuda.synchronize()
    assert torch.equal(e.get_backbone_params(), before)
    c = e.get_compressor_params()
    assert lib.psv_compressor_adam_step_clipped(e._h, C.c_void_p(c.data_ptr()), 1e-3, 0.9, 0.999, 1e-8, 1, 1.0, s) == -3
    assert lib.psv_compressor_peer_reduce_adam_step_clipped(e._h, (C.c_void_p * 1)(c.data_ptr()), 1, 1e-3, 0.9, 0.999,
                                                            1e-8, 1, 1.0, s) == -3
    # a reduce + clipped update pair at world 1 works, and the reduce is consumed by one update
    assert lib.psv_backbone_peer_reduce_sqnorm(e._h, peers, 1, 0, steps, 1.0, None, C.c_void_p(slot.data_ptr()), s) == 0
    assert peer(clip=1.0, sq=slots) == 0
    assert peer(clip=1.0, sq=slots) == -3
    e.close()
    e16 = _engine(geom, sd, 8, "bf16")
    assert lib.psv_backbone_adam_step_groups(e16._h, gp, steps, good, zero, 0.9, 0.999, 1e-8, 1.0, 1.0, None, None,
                                             s) == -4
    assert lib.psv_backbone_peer_reduce_sqnorm(e16._h, peers, 1, 0, steps, 1.0, None,
                                               C.c_void_p(slot.data_ptr()), s) == -4
    e16.close()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs with peer access")
def test_clipped_sharded_step_two_gpus():
    """tools/backbone_p2p_check.py --max-grad-norm at world 2: the three-barrier clipped step over NVLink peer memory."""
    from conftest import ROOT
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29549", os.path.join(ROOT, "tools", "backbone_p2p_check.py"), "--steps", "3",
           "--batch", "16", "--geom", "deits16", "--layer-decay", "0.75", "--max-grad-norm", "0.5"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:], r.stderr[-1500:])
    res = json.loads(lines[-1])
    assert res["ok"], res
