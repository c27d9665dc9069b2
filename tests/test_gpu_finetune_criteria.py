"""Backbone fine-tuning under the similarity skip criterion and from raw uint8 images, and the one-call forward under the
similarity criterion.

Similarity criterion (psv_set_skip_criterion(PSV_SKIP_SIMILARITY), reference pradeep/model_utils.py:73-84): each layer
runs the dense layer on its input (all tokens are queries and keys), sim = 0.3 (cos + 1) / 2 + 0.7 / (1 + ed) of that
output with the input (oracle.vit_skip_oracle.similarity) and mask = [1, sim < st].  The fp64 reference below makes that
decision on its own layer input; on the CPU it runs free on its own decisions and reproduces the oracle's
forward(criterion="similarity").  On the GPU the gradient reference is the teacher-forced one of
test_gpu_finetune_fp64.py (or its keep-all-keys form), fed the masks the training forward decided, and every decision
outside the 1e-4 band must equal the fp64 sim < st on the teacher-forced layer input.  Bars: those of
test_gpu_finetune_fp64.py.

ST = 0.923.  On the synthetic weights (seed 42) and randn inputs the similarity of a token grows with depth (median 0.91
in layer 0, 0.94 in layer 9), so no single threshold makes every layer skip between 10 % and 90 % of the patch tokens;
0.923 comes closest.  Skipped fraction per layer, fp64 reference free-running on seed-1234 inputs: DeiT-S (batch 4)
9.7 % in layer 0 to 92.1 % in layer 9, 66 % overall; ViT-B (batch 2) 3.3 % in layer 0 to 97.4 % in layer 11, 71 %
overall.  Every layer thus both skips and keeps tokens; the CPU test pins this (2 % to 98 %).

uint8: the training input is raw [B, H, W, 3] images (psv_set_u8_input), compared with the same step on the
preprocessing oracle's fp32 pixels: the patches are identical, so logits and masks are bit-equal and the gradients agree
to 1e-6 (relative Frobenius; the bias column sums use atomics).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import preprocess_oracle as P
from oracle import vit_skip_oracle as O
from test_gpu_finetune_fp64 import (_comp_to_dict, _compare, _drop_in_model, _flat_to_dict, _ln, reference_forward,
                                    reference_grads, reference_params)
from test_gpu_finetune_kv_all import reference_forward_kv_all

ST = 0.923
MT = 0.5            # the compressor threshold: its scores are computed (the joint objective reads them) but do not decide
BAND = 1e-4
U8_REL_TOL = 1e-6


# ------------------------------------------------------------------------------------------------ the fp64 reference
def _dense_layer(p, l, h, heads, key_mask=None):
    """The ViT layer on all rows of h [B, N, D]; key_mask (bool [B, N], optional) sets the keys of skipped tokens to
    -inf, which is exact for the active rows of the patch-skip layer."""
    q_ = f"encoder.layer.{l}."
    B, N, D = h.shape
    dh = D // heads
    a = _ln(h, p, q_ + "layernorm_before")
    q, k, v = (F.linear(a, p[q_ + f"attention.attention.{n}.weight"], p[q_ + f"attention.attention.{n}.bias"])
               .view(B, N, heads, dh).transpose(1, 2) for n in ("query", "key", "value"))
    att = torch.matmul(q, k.transpose(2, 3)) * (dh ** -0.5)
    if key_mask is not None:
        att = att.masked_fill(~key_mask[:, None, None, :], float("-inf"))
    ctx = torch.matmul(torch.softmax(att, -1), v).transpose(1, 2).reshape(B, N, D)
    x1 = F.linear(ctx, p[q_ + "attention.output.dense.weight"], p[q_ + "attention.output.dense.bias"]) + h
    u = F.gelu(F.linear(_ln(x1, p, q_ + "layernorm_after"), p[q_ + "intermediate.dense.weight"],
                        p[q_ + "intermediate.dense.bias"]))
    return F.linear(u, p[q_ + "output.dense.weight"], p[q_ + "output.dense.bias"]) + x1


@torch.no_grad()
def reference_similarity(p, pixels, st, heads, forced_masks=None, kv_all=False):
    """The patch-skip forward under the similarity criterion.  Each layer: sim of the dense layer on the layer input,
    mask = [1, sim < st] (or forced_masks[l] when given: teacher forcing), then the skip layer with that mask.
    Returns (logits [B, C], masks bool [L, B, N], sims [L, B, N-1])."""
    w = p["embeddings.patch_embeddings.projection.weight"]
    x = F.conv2d(pixels, w, p["embeddings.patch_embeddings.projection.bias"], stride=w.shape[-1]).flatten(2).transpose(1, 2)
    h = torch.cat((p["embeddings.cls_token"].expand(x.shape[0], -1, -1), x), 1) + p["embeddings.position_embeddings"]
    B = h.shape[0]
    L = 0
    while f"encoder.layer.{L}.layernorm_before.weight" in p:
        L += 1
    masks, sims = [], []
    for l in range(L):
        sim = O.similarity(_dense_layer(p, l, h, heads), h)
        if forced_masks is None:
            m = torch.cat((torch.ones(B, 1, dtype=torch.bool, device=h.device), sim < st), 1)
        else:
            m = forced_masks[l].bool()
        h = torch.where(m[..., None], _dense_layer(p, l, h, heads, None if kv_all else m), h)
        masks.append(m)
        sims.append(sim)
    logits = F.linear(_ln(h[:, 0], p, "layernorm"), p["classifier.weight"], p["classifier.bias"])
    return logits, torch.stack(masks), torch.stack(sims)


# ------------------------------------------------------------------------------------------------ CPU: reference vs oracle
@pytest.mark.parametrize("geom_name, B", [("deits16", 3), ("vitb16", 2)])
def test_similarity_reference_matches_oracle(state_dicts, geom_name, B):
    """Free-running on its own decisions, the fp64 reference reproduces oracle.forward(..., criterion="similarity")."""
    geom, sd = state_dicts(geom_name)
    x = synth.make_pixels(B, geom, seed=1234, kind="randn")
    with torch.no_grad():
        ref = O.forward(sd, x, MT, ST, criterion="similarity")
    p = {k: v.double() for k, v in sd.items() if not k.startswith("pooler.")}
    logits, masks, sims = reference_similarity(p, x.double(), ST, geom.heads)
    band = (sims - ST).abs() < BAND
    assert int(((masks[:, :, 1:] != ref.masks[:, :, 1:]) & ~band).sum()) == 0
    assert bool(masks[:, :, 0].all()) and bool(ref.masks[:, :, 0].all())
    err = float((logits - ref.logits.double()).abs().max())
    assert err < 1e-5, err
    skipped = 1.0 - masks[:, :, 1:].double().mean((1, 2))
    print(f"\n[{geom_name} B={B} st={ST}] skipped fraction per layer {[round(float(f), 2) for f in skipped]}, "
          f"overall {float(skipped.mean()):.2f}; logits max-abs err {err:.2e}")
    assert bool(((skipped >= 0.02) & (skipped <= 0.98)).all()), skipped


# ------------------------------------------------------------------------------------------------ GPU helpers
def _engine(geom, sd, B, precision="fp32", kv_mode="active", criterion="similarity"):
    import psv_native
    e = psv_native.Engine(geom, precision, B)
    e.load_state_dict(sd)
    e.set_kv_mode(kv_mode)
    e.set_skip_criterion(criterion, ST)
    return e


def _upstream(geom, B, logits, upstream, gen):
    if upstream == "ce":
        labels = torch.randint(0, geom.classes, (B,), generator=gen).cuda()
        lg = logits.detach().clone().requires_grad_(True)
        F.cross_entropy(lg, labels).backward()
        return lg.grad
    return torch.randn(B, geom.classes, generator=gen).cuda()


def _check_sim_decisions(gpu_masks, ref_sims, label):
    """Outside the band the GPU decision equals the fp64 sim < st on the teacher-forced layer input."""
    want = ref_sims < ST
    got = gpu_masks[:, :, 1:].bool()
    band = (ref_sims - ST).abs() < BAND
    assert bool(gpu_masks[:, :, 0].bool().all())
    bad = int(((got != want) & ~band).sum())
    skipped = 1.0 - got.double().mean((1, 2))
    print(f"[{label}] decisions: {int(got.sum())} of {got.numel()} patch tokens active, skipped per layer "
          f"{[round(float(f), 2) for f in skipped]}, {int(((got != want) & band).sum())} in-band flips")
    assert bad == 0, f"{bad} decisions differ from sim < st outside the {BAND} band"


def _sim_case(e, geom, sd, B, upstream="ce", joint=False, kv_all=False, seed=1234, label=""):
    """One training step under the similarity criterion against the teacher-forced fp64 reference."""
    x = synth.make_pixels(B, geom, seed=seed, kind="randn").cuda()
    gen = torch.Generator().manual_seed(seed)
    if joint:
        logits, _ = e.backbone_forward_train(x, MT, with_layer_losses=True)
    else:
        logits = e.backbone_forward_train(x, MT)
    masks = e.backbone_train_masks()
    dlogits = _upstream(geom, B, logits, upstream, gen)
    dlosses = torch.rand(geom.layers, generator=gen).cuda() * 2 + 0.25 if joint else None
    out = e.backbone_backward(dlogits, dlosses)
    torch.cuda.synchronize()
    flat, cflat = out if joint else (out, None)
    got = _flat_to_dict(flat, e.backbone_grad_slices())
    if joint:
        got.update(_comp_to_dict(cflat, geom))
    p = reference_params(sd, "cuda")
    _, _, sims = reference_similarity(p, x.double(), ST, geom.heads, forced_masks=masks, kv_all=kv_all)
    _check_sim_decisions(masks, sims, label)
    fwd = reference_forward_kv_all if kv_all else reference_forward
    rl, _, _, rlosses = fwd(p, x.double(), MT, geom.heads, forced_masks=masks, joint=joint)
    outputs, ups = [rl], [dlogits.double()]
    if joint:
        outputs.append(rlosses)
        ups.append(dlosses.double())
    ref = reference_grads(p, outputs, ups, joint)
    err = float((logits.double() - rl.detach()).abs().max())
    print(f"[{label}] logits max-abs err {err:.2e}")
    assert err < 1e-4
    _compare(got, ref, label)
    del p, rl, rlosses, ref, sims


# ------------------------------------------------------------------------------------------------ GPU: gradients
@pytest.mark.gpu
@pytest.mark.parametrize("geom_name, B, upstream, kv_mode", [
    ("deits16", 64, "ce", "active"),
    ("deits16", 64, "randn", "active"),   # upstream gradient without the zero row sums of cross-entropy
    ("vitb16", 48, "ce", "active"),
    ("deits16", 64, "ce", "all"),         # similarity criterion in the keep-all-keys mode
])
def test_similarity_backbone_gradients_match_fp64(state_dicts, geom_name, B, upstream, kv_mode):
    geom, sd = state_dicts(geom_name)
    e = _engine(geom, sd, B, kv_mode=kv_mode)
    try:
        _sim_case(e, geom, sd, B, upstream, kv_all=kv_mode == "all",
                  label=f"similarity {geom_name} B={B} {upstream} kv {kv_mode}")
    finally:
        e.close()


@pytest.mark.gpu
def test_similarity_joint_objective_gradients_match_fp64(state_dicts):
    """Cross-entropy plus the layers' compressor losses, whose labels are the layer's own (similarity) mask."""
    geom, sd = state_dicts("deits16")
    e = _engine(geom, sd, 64)
    try:
        _sim_case(e, geom, sd, 64, "ce", joint=True, seed=99, label="similarity joint deits16 B=64")
    finally:
        e.close()


@pytest.mark.gpu
def test_similarity_smaller_batches_on_a_larger_handle(state_dicts):
    geom, sd = state_dicts("deits16")
    e = _engine(geom, sd, 64)
    try:
        for i, B in enumerate((64, 37, 1)):
            _sim_case(e, geom, sd, B, "ce", seed=500 + i, label=f"similarity max_batch 64, B={B}")
    finally:
        e.close()


def _step(e, x, dlogits, between=None):
    e.backbone_forward_train(x, MT)
    if between is not None:
        between()
    flat = e.backbone_backward(dlogits)
    torch.cuda.synchronize()
    return flat


@pytest.mark.gpu
def test_similarity_backward_survives_a_criterion_switch(state_dicts):
    """A similarity-criterion training forward, then set_skip_criterion("mlp") with an inference forward in that mode,
    then the backward: the gradients are those of the similarity forward."""
    geom, sd = state_dicts("deits16")
    B = 8
    e = _engine(geom, sd, B)
    x1 = synth.make_pixels(B, geom, seed=71).cuda()
    x2 = synth.make_pixels(B, geom, seed=72).cuda()
    dlogits = torch.randn(B, geom.classes, generator=torch.Generator().manual_seed(7)).cuda()
    try:
        clean = _step(e, x1, dlogits)

        def other_work():
            e.set_skip_criterion("mlp")
            e.forward(x2, MT)
            e.forward(x2, MT, use_graph=True)
        disturbed = _step(e, x1, dlogits, other_work)
        e.set_skip_criterion("similarity", ST)
        err = float((disturbed - clean).abs().max()) / float(clean.abs().max())
        assert err <= 1e-5, f"gradients changed by a criterion switch between forward and backward: {err:.3e}"
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: uint8 images
def _u8_and_reference(B, hw, seed):
    rng = np.random.default_rng(seed)
    imgs = rng.integers(0, 256, size=(B, hw[0], hw[1], 3), dtype=np.uint8)
    return torch.from_numpy(imgs).cuda(), torch.from_numpy(P.preprocess_u8(imgs)).cuda()


def _rel_frob(a, b, slices):
    """Worst per-tensor relative Frobenius difference (the key bias, zero in exact arithmetic, against the query bias)."""
    da, db = _flat_to_dict(a, slices), _flat_to_dict(b, slices)
    worst = 0.0
    for k in da:
        scale = db[k.replace("key.bias", "query.bias")] if k.endswith("attention.key.bias") else db[k]
        n = float(scale.double().norm())
        if n > 0:
            worst = max(worst, float((da[k] - db[k]).double().norm()) / n)
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("criterion", ["mlp", "similarity"])
@pytest.mark.parametrize("hw", [(32, 32), (224, 224)])
def test_u8_training_step_equals_preprocessed_step(state_dicts, hw, criterion):
    """uint8 [B, H, W, 3] training input (32 x 32 up-scaled, 224 x 224) against the same step on the preprocessing
    oracle's fp32 pixels: logits and masks bit-equal, gradients within 1e-6; set_u8_input(64, 64) between the forward
    and the backward leaves the gradients unchanged."""
    geom, sd = state_dicts("deits16")
    B = 16
    e = _engine(geom, sd, B, criterion=criterion)
    u8, ref_pixels = _u8_and_reference(B, hw, hw[0] * 31 + hw[1])
    dlogits = torch.randn(B, geom.classes, generator=torch.Generator().manual_seed(3)).cuda()
    slices = e.backbone_grad_slices()
    try:
        e.set_u8_input(*hw)
        lu = e.backbone_forward_train(u8, MT).clone()
        mu = e.backbone_train_masks().clone()
        gu = e.backbone_backward(dlogits).clone()
        lf = e.backbone_forward_train(ref_pixels, MT).clone()
        mf = e.backbone_train_masks().clone()
        gf = e.backbone_backward(dlogits).clone()
        torch.cuda.synchronize()
        assert torch.equal(lu, lf) and torch.equal(mu, mf)
        err = _rel_frob(gu, gf, slices)
        # the setup of the forward, not the handle's current one, drives the backward's im2col
        e.backbone_forward_train(u8, MT)
        e.set_u8_input(64, 64)
        gs = e.backbone_backward(dlogits)
        torch.cuda.synchronize()
        err_switch = _rel_frob(gs, gu, slices)
        print(f"\n[u8 {hw} {criterion}] gradients vs fp32 pixels {err:.2e}, after set_u8_input(64, 64) {err_switch:.2e}")
        assert err <= U8_REL_TOL and err_switch <= U8_REL_TOL
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: one-call forward
def _per_layer(e, x, st):
    """embed -> per layer similarity_mask + layer_forward(forced) -> head: the drop-in's per-layer path."""
    hidden = e.embed(x)
    masks = []
    for l in range(e.geom.layers):
        m, _ = e.similarity_mask(l, hidden, st)
        mask, _, _ = e.layer_forward(l, hidden, MT, forced_mask=m)
        masks.append(mask)
    return e.head(hidden), torch.stack(masks)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_similarity_forward_equals_per_layer_sequence(state_dicts, precision):
    """psv_forward under PSV_SKIP_SIMILARITY, eager and as a CUDA graph, is bit-equal (logits and masks) to the per-layer
    similarity_mask + layer_forward sequence (bf16: the packed-row attention kernel, chosen explicitly)."""
    geom, sd = state_dicts("deits16")
    B = 16
    e = _engine(geom, sd, B, precision=precision)
    if precision == "bf16":
        e.set_attention_kernel("pk")
    x = synth.make_pixels(B, geom, seed=1234, kind="randn").cuda()
    try:
        for use_graph in (False, True, True):
            r = e.forward(x, MT, want_masks=True, use_graph=use_graph)
            logits, masks = r["logits"].clone(), r["masks"].clone()
            ref_logits, ref_masks = _per_layer(e, x, ST)
            torch.cuda.synchronize()
            skipped = 1.0 - masks[:, :, 1:].double().mean()
            print(f"\n[{precision} graph={use_graph}] skipped {float(skipped):.2f}")
            assert torch.equal(masks, ref_masks), int((masks != ref_masks).sum())
            assert torch.equal(logits, ref_logits), float((logits - ref_logits).abs().max())
            assert 0.05 < float(skipped) < 0.95
    finally:
        e.close()


@pytest.mark.gpu
def test_similarity_criterion_refusals(state_dicts):
    import psv_native
    geom, sd = state_dicts("deits16")
    e = _engine(geom, sd, 4)
    x = synth.make_pixels(4, geom, seed=5).cuda()
    try:
        with pytest.raises(psv_native.PsvError):
            e.compressor_grads(x, MT)                  # native compressor training follows the mlp criterion only
        with pytest.raises(psv_native.PsvError):
            e.set_skip_criterion("similarity", float("nan"))
        with pytest.raises(psv_native.PsvError):
            e.backbone_forward_train(x.bfloat16(), MT)
        e.set_skip_criterion("mlp")
        e.compressor_grads(x, MT)
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: the drop-in
def _similarity_model(geom, sd):
    model = _drop_in_model(geom, sd, MT)
    model.skip_criterion = "similarity"
    for layer in model.encoder.layer:
        layer.sim_threshold = ST
    return model


@pytest.mark.gpu
def test_similarity_drop_in_cross_entropy_step_matches_fp64(state_dicts):
    """model.skip_criterion = "similarity", vit_train(): the .grad of one cross-entropy step equal the fp64 reference's."""
    geom, sd = state_dicts("deits16")
    B = 8
    model = _similarity_model(geom, sd)
    x = synth.make_pixels(B, geom, seed=81).cuda()
    y = torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(8)).cuda()
    model.zero_grad(set_to_none=True)
    logits = model(x).logits
    lg = logits.detach().clone().requires_grad_(True)
    F.cross_entropy(lg, y).backward()
    F.cross_entropy(logits, y).backward()
    got = {k: q.grad for k, q in model.named_parameters() if q.grad is not None}
    masks = model._psv_engine.backbone_train_masks()
    p = reference_params(sd, "cuda")
    _, _, sims = reference_similarity(p, x.double(), ST, geom.heads, forced_masks=masks)
    _check_sim_decisions(masks, sims, "similarity drop-in")
    rl, _, _, _ = reference_forward(p, x.double(), MT, geom.heads, forced_masks=masks)
    ref = reference_grads(p, [rl], [lg.grad.double()], False)
    _compare({k: got[k] for k in ref}, ref, "similarity drop-in cross-entropy step")
    # an evaluation forward takes the one-call path under the criterion and agrees with the per-layer one
    model.eval()
    with torch.no_grad():
        one_call = model(x, output_mask=True)
        per_layer = model(x, output_mask=True, output_hidden_states=True)
    assert all(torch.equal(a, b) for a, b in zip(one_call.boolean_masks, per_layer.boolean_masks))
    assert float((one_call.logits - per_layer.logits).abs().max()) < 1e-4


@pytest.mark.gpu
def test_similarity_drop_in_train_both(state_dicts):
    """train(loss_type="both") for one epoch of two batches under the similarity criterion: finite losses."""
    import main_model_utils
    geom, sd = state_dicts("deits16")
    B = 8
    model = _similarity_model(geom, sd)
    before = {k: q.detach().clone() for k, q in model.named_parameters()}
    loader = main_model_utils.synthetic_loader(2 * B, B, geom=geom, seed=91)
    history = main_model_utils.train(model, loader, None, "cuda", num_epochs=1, loss_type="both")
    assert len(history) == 1 and np.isfinite(history[0]), history
    moved = [k for k, q in model.named_parameters() if not torch.equal(q.detach(), before[k])]
    assert any("mlp_layer" in k for k in moved) and any("attention.attention.key" in k for k in moved)


@pytest.mark.gpu
def test_drop_in_u8_step_equals_preprocessed_step(state_dicts):
    """One cross-entropy step of the drop-in on uint8 [B, 32, 32, 3] images gives the .grad of the same step on the
    preprocessed fp32 pixels."""
    geom, sd = state_dicts("deits16")
    B = 8
    model = _drop_in_model(geom, sd, MT)
    u8, ref_pixels = _u8_and_reference(B, (32, 32), 17)
    y = torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(9)).cuda()

    def step(x):
        model.zero_grad(set_to_none=True)
        F.cross_entropy(model(x).logits, y).backward()
        return {k: q.grad.detach().clone() for k, q in model.named_parameters() if q.grad is not None}
    gu, gf = step(u8), step(ref_pixels)
    assert set(gu) == set(gf)
    worst = 0.0
    for k in gf:
        scale = gf[k.replace("key.bias", "query.bias")] if k.endswith("attention.key.bias") else gf[k]
        n = float(scale.double().norm())
        if n > 0:
            worst = max(worst, float((gu[k] - gf[k]).double().norm()) / n)
    print(f"\n[drop-in u8] worst relative Frobenius {worst:.2e}")
    assert worst <= U8_REL_TOL
