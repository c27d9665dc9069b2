"""Backbone fine-tuning (psv_backbone_forward_train / psv_backbone_backward) against a float64 autograd reference at
training batch sizes, element by element on every gradient tensor.

The reference is the patch-skip forward written in the dense masked form, which is exact for the active rows: at every
layer the compressor scores come from the undetached [h[:, 0]; h[:, t]], attention runs on all N rows with the keys of
skipped tokens at -inf (CLS is always active, so no row is fully masked), and h = where(mask, layer(h), h).  With
``joint`` the layers' compressor losses (himanshu/model_utils.py:103-108) are outputs too, as for loss_type "both"
(main_model_utils.py:131-135).  On the GPU the reference is teacher-forced with the masks the training forward decided
(``Engine.backbone_train_masks``); those decisions are checked against the reference's own scores outside the 1e-4
band.  On the CPU the reference itself is checked against the goldens of the unmodified reference.

The backward's GEMMs multiply two bf16 planes per operand (about 16 mantissa bits) with fp32 accumulation; the bars
below sit about 4x above the worst errors measured on a B200 (values in the comment).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
from conftest import load_golden

LN_EPS = 1e-12
BAND = 1e-4

# Bars about 4x above the worst errors measured on a B200 (1000 W): backbone tensors 3.3e-5 rel-Frobenius, 4.3e-5
# max-abs (joint DeiT-S, batch 64); compressor tensors 5.7e-4 / 1.9e-3 (joint ViT-B, batch 64).  With one bf16 plane
# per operand instead of two the backbone errors grow to about 7e-3.
REL_FROB_TOL = 1.5e-4        # ||g - r|| / ||r||
MAX_ABS_TOL = 2e-4           # max |g - r| / max |r|
COMP_REL_FROB_TOL = 2.5e-3   # compressor tensors (a few hidden units may sit next to the ReLU kink)
COMP_MAX_ABS_TOL = 1e-2


# ------------------------------------------------------------------------------------------------ the fp64 reference
def _ln(x, p, prefix):
    return F.layer_norm(x, (x.shape[-1],), p[prefix + ".weight"], p[prefix + ".bias"], LN_EPS)


def reference_forward(p, pixels, mt, heads, forced_masks=None, joint=False):
    """p: reference-keyed parameters, pixels [B, 3, H, W] (both in the compute dtype).  Returns (logits [B, C],
    masks bool [L, B, N], scores [L, B, N-1], layer losses [L] or None)."""
    w = p["embeddings.patch_embeddings.projection.weight"]
    x = F.conv2d(pixels, w, p["embeddings.patch_embeddings.projection.bias"], stride=w.shape[-1]).flatten(2).transpose(1, 2)
    h = torch.cat((p["embeddings.cls_token"].expand(x.shape[0], -1, -1), x), 1) + p["embeddings.position_embeddings"]
    B, N, D = h.shape
    dh = D // heads
    L = 0
    while f"encoder.layer.{L}.layernorm_before.weight" in p:
        L += 1
    masks, scores, losses = [], [], []
    for l in range(L):
        q_ = f"encoder.layer.{l}."
        z = torch.cat((h[:, :1].expand(-1, N - 1, -1), h[:, 1:]), -1)
        z = F.relu(F.linear(z, p[q_ + "mlp_layer.0.weight"], p[q_ + "mlp_layer.0.bias"]))
        s = torch.sigmoid(F.linear(z, p[q_ + "mlp_layer.2.weight"], p[q_ + "mlp_layer.2.bias"])).squeeze(-1)
        if forced_masks is None:
            m = torch.cat((torch.ones(B, 1, dtype=torch.bool, device=h.device), s.detach() >= mt), 1)
        else:
            m = forced_masks[l].bool()
        if joint:
            labels = m[:, 1:].to(s.dtype)
            mean = labels.mean()
            losses.append(F.binary_cross_entropy_with_logits(s, labels, pos_weight=(mean / (1 - mean + 1e-16)).reshape(1)))
        a = _ln(h, p, q_ + "layernorm_before")
        q, k, v = (F.linear(a, p[q_ + f"attention.attention.{n}.weight"], p[q_ + f"attention.attention.{n}.bias"])
                   .view(B, N, heads, dh).transpose(1, 2) for n in ("query", "key", "value"))
        att = torch.matmul(q, k.transpose(2, 3)) * (dh ** -0.5)
        att = att.masked_fill(~m[:, None, None, :], float("-inf"))
        ctx = torch.matmul(torch.softmax(att, -1), v).transpose(1, 2).reshape(B, N, D)
        x1 = F.linear(ctx, p[q_ + "attention.output.dense.weight"], p[q_ + "attention.output.dense.bias"]) + h
        u = F.gelu(F.linear(_ln(x1, p, q_ + "layernorm_after"), p[q_ + "intermediate.dense.weight"],
                            p[q_ + "intermediate.dense.bias"]))
        y = F.linear(u, p[q_ + "output.dense.weight"], p[q_ + "output.dense.bias"]) + x1
        h = torch.where(m[..., None], y, h)
        masks.append(m)
        scores.append(s.detach())
    logits = F.linear(_ln(h[:, 0], p, "layernorm"), p["classifier.weight"], p["classifier.bias"])
    return logits, torch.stack(masks), torch.stack(scores), (torch.stack(losses) if joint else None)


def reference_params(sd, device, dtype=torch.float64):
    return {k: v.to(device=device, dtype=dtype).requires_grad_(True) for k, v in sd.items() if not k.startswith("pooler.")}


def reference_grads(p, outputs, upstream, joint):
    """Gradients of sum(<output, upstream>) with respect to every parameter the objective reaches."""
    keys = [k for k in p if joint or "mlp_layer" not in k]
    gs = torch.autograd.grad(outputs, [p[k] for k in keys], upstream, allow_unused=True)
    return {k: (torch.zeros_like(p[k]) if g is None else g).detach() for k, g in zip(keys, gs)}


# ------------------------------------------------------------------------------------------------ CPU: reference vs goldens
@pytest.mark.parametrize("golden, geom_name", [("finetune_deits16_randn_b4", "deits16"),
                                               ("finetune_both_deits16_randn_b4", "deits16"),
                                               ("finetune_both_vitb16_randn_b2", "vitb16")])
def test_reference_matches_goldens(state_dicts, golden, geom_name):
    """The fp64 dense-masked reference reproduces the unmodified reference's logits, loss, gradient norms and complete
    small tensors (its own decisions, no teacher forcing)."""
    g = load_golden(golden)
    geom, sd = state_dicts(geom_name)
    joint = str(g["loss_type"]) == "both"
    p = reference_params(sd, "cpu")
    x = synth.make_pixels(int(g["batch"]), geom, seed=int(g["seed_pixels"]), kind=str(g["kind"])).double()
    logits, _, _, losses = reference_forward(p, x, float(g["mt"]), geom.heads, joint=joint)
    assert float((logits.detach() - torch.from_numpy(g["logits"]).double()).abs().max()) < 1e-5
    loss = F.cross_entropy(logits, torch.from_numpy(g["labels"]))
    if joint:
        assert np.abs(losses.detach().numpy() - g["layer_losses"]).max() < 1e-5 * np.abs(g["layer_losses"]).max()
        loss = loss + losses.sum()
    assert abs(float(loss.detach()) - float(g["loss"])) < 2e-5
    grads = reference_grads(p, [loss], None, joint)
    norms = dict(zip(map(str, g["grad_keys"]), g["grad_norms"].astype(np.float64)))
    assert set(grads) == set(norms), set(grads) ^ set(norms)
    for k, ref in norms.items():
        got = float(grads[k].norm())
        if k.endswith("attention.key.bias"):           # zero in exact arithmetic: both sides hold rounding noise
            qb = norms[k.replace("key.bias", "query.bias")]
            assert got <= 1e-3 * qb and ref <= 1e-3 * qb, (k, got, ref)
            continue
        # the goldens come from an fp32 autograd: the norms of the largest weight gradients (FC1) are 1e-4 off
        assert abs(got - ref) <= 5e-4 * ref, (k, got, ref)
    for k in map(str, g["full_keys"]):
        ref = g["full:" + k].astype(np.float64)
        if k.endswith("attention.key.bias"):
            continue
        err = np.abs(grads[k].numpy().reshape(ref.shape) - ref).max()
        assert err <= 2e-5 * np.abs(ref).max(), (k, err, np.abs(ref).max())


# ------------------------------------------------------------------------------------------------ GPU helpers
def _flat_to_dict(flat, slices):
    return {k: flat[o:o + int(np.prod(shape))].reshape(shape) for k, (o, shape) in slices.items()}


def _comp_to_dict(cflat, geom):
    per = cflat.numel() // geom.layers
    ch, D = geom.comp_hidden, geom.hidden
    out = {}
    for l in range(geom.layers):
        o = l * per
        for name, shape in (("0.weight", (ch, 2 * D)), ("0.bias", (ch,)), ("2.weight", (1, ch)), ("2.bias", (1,))):
            n = int(np.prod(shape))
            out[f"encoder.layer.{l}.mlp_layer.{name}"] = cflat[o:o + n].reshape(shape)
            o += n
    return out


def _compare(got, ref, label):
    """Per-tensor relative Frobenius and max-abs errors; prints the worst of each and asserts the bars."""
    assert set(got) == set(ref), set(got) ^ set(ref)
    worst = {"rel_frob": (0.0, ""), "max_abs": (0.0, ""), "comp_rel_frob": (0.0, ""), "comp_max_abs": (0.0, "")}
    fails = []
    for k, r in ref.items():
        g = got[k].detach().double().reshape(r.shape)
        r = r.double()
        if k.endswith("attention.attention.key.bias"):
            # softmax ignores the per-row constant q . b_k: the exact gradient is zero, both sides hold rounding noise
            qb = float(ref[k.replace("key.bias", "query.bias")].norm())
            if float(g.norm()) > 1e-3 * qb + 1e-12:
                fails.append((k, "abs", float(g.norm()), qb))
            continue
        rn, rmax = float(r.norm()), float(r.abs().max())
        if rn == 0.0:                                 # exactly zero (e.g. q / k with one token per image)
            if float(g.abs().max()) > 1e-12:
                fails.append((k, "zero", float(g.abs().max()), 0.0))
            continue
        d = g - r
        if "mlp_layer" in k:
            rf, ma = float(d.norm()) / rn, float(d.abs().max()) / rmax
            if k.endswith("0.weight") or k.endswith("0.bias"):
                # a pre-activation next to the ReLU kink moves one hidden unit's row: up to 2 units may deviate
                per_unit = d.reshape(r.shape[0], -1).abs().amax(1) > COMP_MAX_ABS_TOL * rmax
                ok = int(per_unit.sum()) <= 2
                keep = ~per_unit
                ma = float(d.reshape(r.shape[0], -1)[keep].abs().max()) / rmax if bool(keep.any()) else 0.0
                rf = float(d.reshape(r.shape[0], -1)[keep].norm()) / rn
            else:
                ok = True
            for name, v in (("comp_rel_frob", rf), ("comp_max_abs", ma)):
                if v > worst[name][0]:
                    worst[name] = (v, k)
            if not ok or rf > COMP_REL_FROB_TOL or ma > COMP_MAX_ABS_TOL:
                fails.append((k, "comp", rf, ma))
            continue
        rf, ma = float(d.norm()) / rn, float(d.abs().max()) / rmax
        for name, v in (("rel_frob", rf), ("max_abs", ma)):
            if v > worst[name][0]:
                worst[name] = (v, k)
        if rf > REL_FROB_TOL or ma > MAX_ABS_TOL:
            fails.append((k, "backbone", rf, ma))
    print(f"\n[{label}] {len(ref)} tensors; worst rel-Frobenius {worst['rel_frob'][0]:.2e} ({worst['rel_frob'][1]}), "
          f"worst max-abs/max|r| {worst['max_abs'][0]:.2e} ({worst['max_abs'][1]})"
          + (f"; compressors: rel-Frobenius {worst['comp_rel_frob'][0]:.2e} ({worst['comp_rel_frob'][1]}), "
             f"max-abs {worst['comp_max_abs'][0]:.2e} ({worst['comp_max_abs'][1]})" if worst["comp_max_abs"][1] else ""))
    assert not fails, fails[:10]


def _check_decisions(gpu_masks, ref_scores, mt, label):
    """Outside the band the GPU decision equals the fp64 score >= mt on the teacher-forced layer input."""
    want = ref_scores >= mt
    got = gpu_masks[:, :, 1:].bool()
    band = (ref_scores - mt).abs() < BAND
    assert bool(gpu_masks[:, :, 0].bool().all())
    bad = int(((got != want) & ~band).sum())
    flips = int(((got != want) & band).sum())
    print(f"[{label}] decisions: {int(got.sum())} of {got.numel()} patch tokens active, {flips} in-band flips, "
          f"{int(band.sum())} in band")
    assert bad == 0, f"{bad} decisions differ outside the {BAND} band"


def _case(e, geom, sd, B, mt, upstream="ce", joint=False, seed=1234, label=""):
    """One GPU training step against the teacher-forced fp64 reference on the same upstream gradients."""
    x = synth.make_pixels(B, geom, seed=seed, kind="randn").cuda()
    gen = torch.Generator().manual_seed(seed)
    if joint:
        logits, _ = e.backbone_forward_train(x, mt, with_layer_losses=True)
    else:
        logits = e.backbone_forward_train(x, mt)
    masks = e.backbone_train_masks()
    if upstream == "ce":
        labels = torch.randint(0, geom.classes, (B,), generator=gen).cuda()
        lg = logits.detach().clone().requires_grad_(True)
        F.cross_entropy(lg, labels).backward()
        dlogits = lg.grad
    else:                                  # no structure: CE rows sum to zero, which hides per-row constant errors
        dlogits = torch.randn(B, geom.classes, generator=gen).cuda()
    dlosses = torch.rand(geom.layers, generator=gen).cuda() * 2 + 0.25 if joint else None
    out = e.backbone_backward(dlogits, dlosses)
    torch.cuda.synchronize()
    flat, cflat = out if joint else (out, None)
    got = _flat_to_dict(flat, e.backbone_grad_slices())
    if joint:
        got.update(_comp_to_dict(cflat, geom))
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    p = reference_params(sd, "cuda")
    rl, _, rs, rlosses = reference_forward(p, x.double(), mt, geom.heads, forced_masks=masks, joint=joint)
    outputs, ups = [rl], [dlogits.double()]
    if joint:
        outputs.append(rlosses)
        ups.append(dlosses.double())
    ref = reference_grads(p, outputs, ups, joint)
    peak = (torch.cuda.max_memory_allocated() - base) / 2 ** 30
    print(f"\n[{label}] fp64 reference peak memory {peak:.2f} GiB; logits max-abs err "
          f"{float((logits.double() - rl.detach()).abs().max()):.2e}")
    assert float((logits.double() - rl.detach()).abs().max()) < 1e-4
    _check_decisions(masks, rs, mt, label)
    _compare(got, ref, label)
    del p, rl, rs, rlosses, ref


# ------------------------------------------------------------------------------------------------ GPU: the matrix
@pytest.mark.gpu
@pytest.mark.parametrize("geom_name, B, mt, upstream", [
    ("deits16", 64, 0.0, "ce"),          # every token active: 197-row sequences, wgrad K = 12 608
    ("deits16", 64, 0.5, "ce"),          # the natural ragged profile
    ("deits16", 64, 0.5, "randn"),       # upstream gradient without the zero row sums of cross-entropy
    ("deits16", 64, 1.5, "ce"),          # CLS only: T = batch, wgrad K padded from 64, dgrad M < 128
    ("vitb16", 48, 0.5, "ce"),           # D = 768 LayerNorm backward, more GEMM tiles than SMs
    ("vitb16", 64, 0.5, "ce"),
])
def test_backbone_gradients_match_fp64(state_dicts, geom_name, B, mt, upstream):
    import psv_native
    geom, sd = state_dicts(geom_name)
    e = psv_native.Engine(geom, "fp32", B)
    e.load_state_dict(sd)
    try:
        _case(e, geom, sd, B, mt, upstream, label=f"{geom_name} B={B} mt={mt} {upstream}")
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("geom_name, B", [("vitb16", 32), ("deits16", 64)])
def test_joint_objective_gradients_match_fp64(state_dicts, geom_name, B):
    """Cross-entropy plus the layers' compressor losses with distinct upstream gradients: backbone and compressors."""
    import psv_native
    geom, sd = state_dicts(geom_name)
    e = psv_native.Engine(geom, "fp32", B)
    e.load_state_dict(sd)
    try:
        _case(e, geom, sd, B, 0.5, "ce", joint=True, seed=99, label=f"joint {geom_name} B={B}")
    finally:
        e.close()


@pytest.mark.gpu
def test_smaller_batches_on_a_larger_handle(state_dicts):
    """Batches 64, 37, 1 on one max_batch-64 handle: state left by a larger batch, MB-strided compaction records."""
    import psv_native
    geom, sd = state_dicts("deits16")
    e = psv_native.Engine(geom, "fp32", 64)
    e.load_state_dict(sd)
    try:
        for i, B in enumerate((64, 37, 1)):
            _case(e, geom, sd, B, 0.5, "ce", seed=500 + i, label=f"max_batch 64, B={B}")
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: pending backward
def _engine_grads(e, x, mt, dlogits, between=None):
    e.backbone_forward_train(x, mt)
    if between is not None:
        between()
    flat = e.backbone_backward(dlogits)
    torch.cuda.synchronize()
    return flat


@pytest.mark.gpu
def test_backward_survives_inference_calls_in_between(state_dicts):
    """backbone_forward_train(x1), then forward(x2) eagerly and as a CUDA graph and compressor_grads(x2), then the
    backward: the gradients are those of x1."""
    import psv_native
    geom, sd = state_dicts("deits16")
    B, mt = 8, 0.5
    e = psv_native.Engine(geom, "fp32", B)
    e.load_state_dict(sd)
    x1 = synth.make_pixels(B, geom, seed=11).cuda()
    x2 = synth.make_pixels(B, geom, seed=12).cuda()
    dlogits = torch.randn(B, geom.classes, generator=torch.Generator().manual_seed(3)).cuda()
    clean = _engine_grads(e, x1, mt, dlogits)

    def other_work():
        e.forward(x2, mt)
        e.forward(x2, mt, use_graph=True)
        e.forward(x2, mt, use_graph=True)
        e.compressor_grads(x2, mt)
    disturbed = _engine_grads(e, x1, mt, dlogits, other_work)
    err = float((disturbed - clean).abs().max()) / float(clean.abs().max())
    assert err <= 1e-5, f"gradients changed by inference calls between forward and backward: {err:.3e}"
    # and they are x1's gradients
    masks = e.backbone_train_masks()
    p = reference_params(sd, "cuda")
    rl, _, _, _ = reference_forward(p, x1.double(), mt, geom.heads, forced_masks=masks)
    ref = reference_grads(p, [rl], [dlogits.double()], False)
    _compare(_flat_to_dict(disturbed, e.backbone_grad_slices()), ref, "forward / compressor_grads in between")
    e.close()


def _drop_in_model(geom, sd, mt):
    import model_utils
    from transformers.models.vit.modeling_vit import ViTConfig
    cfg = ViTConfig(hidden_size=geom.hidden, num_attention_heads=geom.heads, intermediate_size=geom.ffn)
    cfg.num_labels = geom.classes
    model = model_utils.ModifiedViTModel(cfg, 0.9, mt, 0)
    model.load_state_dict(sd, strict=False)
    model = model.to("cuda")
    model.psv_precision = "fp32"
    model.train()
    model.vit_train()
    return model


@pytest.mark.gpu
def test_drop_in_evaluation_between_forward_and_backward(state_dicts):
    """loss = ce(model(x).logits, y); model.eval(); model(val); model.train(); loss.backward() gives x's gradients."""
    geom, sd = state_dicts("deits16")
    B, mt = 8, 0.5
    model = _drop_in_model(geom, sd, mt)
    x = synth.make_pixels(B, geom, seed=21).cuda()
    val = synth.make_pixels(B, geom, seed=22).cuda()
    y = torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(4)).cuda()

    def step(evaluate):
        model.zero_grad(set_to_none=True)
        loss = F.cross_entropy(model(x).logits, y)
        if evaluate:
            model.eval()
            with torch.no_grad():
                model(val)
            model.train()
        loss.backward()
        return {k: q.grad.detach().clone() for k, q in model.named_parameters() if q.grad is not None}
    clean = step(False)
    disturbed = step(True)
    scale = max(float(v.abs().max()) for v in clean.values())
    for k in clean:
        err = float((disturbed[k] - clean[k]).abs().max())
        assert err <= 1e-5 * scale, f"{k}: the evaluation forward changed the gradient by {err:.3e} (scale {scale:.3e})"
    # and they are x's gradients
    e = model._psv_engine
    logits = e.backbone_forward_train(x, mt)
    masks = e.backbone_train_masks()
    p = reference_params(sd, "cuda")
    rl, _, _, _ = reference_forward(p, x.double(), mt, geom.heads, forced_masks=masks)
    lg = logits.detach().clone().requires_grad_(True)
    F.cross_entropy(lg, y).backward()
    ref = reference_grads(p, [rl], [lg.grad.double()], False)
    _compare({k: disturbed[k] for k in ref}, ref, "evaluation in between")


@pytest.mark.gpu
def test_drop_in_two_forwards_one_backward_raises(state_dicts):
    """Gradient accumulation over two training forwards and one backward cannot be served by one saved forward: it
    raises instead of returning the second forward's state for the first."""
    import psv_native
    geom, sd = state_dicts("deits16")
    B, mt = 4, 0.5
    model = _drop_in_model(geom, sd, mt)
    x1 = synth.make_pixels(B, geom, seed=31).cuda()
    x2 = synth.make_pixels(B, geom, seed=32).cuda()
    y = torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(5)).cuda()
    loss = F.cross_entropy(model(x1).logits, y) + F.cross_entropy(model(x2).logits, y)
    with pytest.raises(psv_native.PsvError, match="another training forward"):
        loss.backward()
    # one forward + backward per micro-batch accumulates correctly
    model.zero_grad(set_to_none=True)
    F.cross_entropy(model(x1).logits, y).backward()
    F.cross_entropy(model(x2).logits, y).backward()
    assert all(torch.isfinite(q.grad).all() for q in model.parameters() if q.grad is not None)


@pytest.mark.gpu
def test_backward_rejects_mismatched_dlogits(state_dicts):
    import psv_native
    geom, sd = state_dicts("deits16")
    e = psv_native.Engine(geom, "fp32", 8)
    e.load_state_dict(sd)
    with pytest.raises(psv_native.PsvError):
        e.backbone_train_masks()                      # no training forward yet
    e.backbone_forward_train(synth.make_pixels(4, geom, seed=41).cuda(), 0.5)
    with pytest.raises(psv_native.PsvError, match="dlogits"):
        e.backbone_backward(torch.zeros(8, geom.classes, device="cuda"))
    assert e.backbone_train_masks().shape == (geom.layers, 4, geom.tokens)
    e.close()
