"""Training in the keep-all-keys mode (query-only pruning, psv_set_kv_mode(PSV_KV_ALL), reference recap/convprad4.py:99-125):
backbone fine-tuning (psv_backbone_forward_train / psv_backbone_backward) and native compressor training
(psv_compressor_grads) against a float64 autograd reference, element by element on every gradient tensor.

In this mode skipped tokens are not queries but still serve as keys and values.  Everything after attention works row by
row, so the layer equals the dense layer followed by h = where(mask, layer(h), h): the exact float64 reference is the
dense-masked reference of test_gpu_finetune_fp64.py without the masking of the keys.  On the CPU it is checked against the
goldens of the unmodified recap layer (tests/golden/kvall_*.npz); on the GPU it is teacher-forced with the masks the
training forward decided, and those decisions are checked against the reference's own scores outside the 1e-4 band.

Bars: those of test_gpu_finetune_fp64.py.  Worst errors measured on a B200 (1000 W) over the cases below: backbone
tensors 3.0e-5 rel-Frobenius, 4.9e-5 max-abs (joint ViT-B, batch 32; bars 1.5e-4 / 2e-4); compressor tensors 2.0e-4
rel-Frobenius (joint ViT-B, batch 32), 7.0e-4 max-abs (psv_compressor_grads, DeiT-S, batch 64; bars 2.5e-3 / 1e-2).  At
mt 0.0 the keep-all-keys gradients differ from the active-mode ones by 4.2e-7 (relative max-abs).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
from conftest import load_golden
from test_gpu_finetune_fp64 import (_check_decisions, _comp_to_dict, _compare, _drop_in_model, _flat_to_dict, _ln,
                                    reference_forward, reference_grads, reference_params)


# ------------------------------------------------------------------------------------------------ the fp64 reference
def reference_forward_kv_all(p, pixels, mt, heads, forced_masks=None, joint=False, hidden_out=None):
    """reference_forward of test_gpu_finetune_fp64.py with every token a key / value.  Same arguments and returns;
    ``hidden_out`` (a list) receives the output of every layer."""
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
        ctx = torch.matmul(torch.softmax(att, -1), v).transpose(1, 2).reshape(B, N, D)
        x1 = F.linear(ctx, p[q_ + "attention.output.dense.weight"], p[q_ + "attention.output.dense.bias"]) + h
        u = F.gelu(F.linear(_ln(x1, p, q_ + "layernorm_after"), p[q_ + "intermediate.dense.weight"],
                            p[q_ + "intermediate.dense.bias"]))
        y = F.linear(u, p[q_ + "output.dense.weight"], p[q_ + "output.dense.bias"]) + x1
        h = torch.where(m[..., None], y, h)
        if hidden_out is not None:
            hidden_out.append(h.detach())
        masks.append(m)
        scores.append(s.detach())
    logits = F.linear(_ln(h[:, 0], p, "layernorm"), p["classifier.weight"], p["classifier.bias"])
    return logits, torch.stack(masks), torch.stack(scores), (torch.stack(losses) if joint else None)


# ------------------------------------------------------------------------------------------------ CPU: reference vs goldens
@pytest.mark.parametrize("golden, geom_name", [("kvall_vitb16_randn_b3", "vitb16"), ("kvall_deits16_randn_b2", "deits16")])
def test_kv_all_reference_matches_recap_goldens(state_dicts, golden, geom_name):
    """Free-running on its own decisions, the fp64 keep-all-keys reference reproduces the unmodified recap layer:
    masks, logits and the sampled layer-output rows."""
    g = load_golden(golden)
    geom, sd = state_dicts(geom_name)
    p = reference_params(sd, "cpu")
    x = synth.make_pixels(int(g["batch"]), geom, seed=int(g["seed_pixels"]), kind=str(g["kind"])).double()
    hidden = []
    with torch.no_grad():
        logits, masks, _, _ = reference_forward_kv_all(p, x, float(g["mt"]), geom.heads, hidden_out=hidden)
    assert np.array_equal(masks.numpy().astype(np.uint8), g["masks"])
    assert float((logits - torch.from_numpy(g["logits_oracle"]).double()).abs().max()) < 1e-5
    rows = g["sample_rows"].tolist()
    for l in g["layers"].tolist():
        err = float((hidden[l][:, rows] - torch.from_numpy(g[f"out_rows_{l}"]).double()).abs().max())
        assert err < 1e-5, (l, err)


@pytest.mark.parametrize("mt, equal", [(0.0, True), (0.5, False)])
def test_kv_all_reference_against_active_reference(state_dicts, mt, equal):
    """With every token active (mt 0.0) the two modes are one computation; at mt 0.5 they are told apart."""
    geom, sd = state_dicts("deits16")
    p = reference_params(sd, "cpu")
    x = synth.make_pixels(2, geom, seed=7).double()
    with torch.no_grad():
        a, ma, _, _ = reference_forward_kv_all(p, x, mt, geom.heads)
        b, mb, _, _ = reference_forward(p, x, mt, geom.heads)
    diff = float((a - b).abs().max())
    if equal:
        assert bool(ma.all()) and diff < 1e-10, diff
    else:
        assert not bool(ma.all()) and diff > 1e-2, diff


# ------------------------------------------------------------------------------------------------ GPU helpers
def _engine(geom, sd, B, precision="fp32"):
    import psv_native
    e = psv_native.Engine(geom, precision, B)
    e.load_state_dict(sd)
    e.set_kv_mode("all")
    return e


def _upstream(geom, B, logits, upstream, gen):
    if upstream == "ce":
        labels = torch.randint(0, geom.classes, (B,), generator=gen).cuda()
        lg = logits.detach().clone().requires_grad_(True)
        F.cross_entropy(lg, labels).backward()
        return lg.grad
    return torch.randn(B, geom.classes, generator=gen).cuda()


def _case(e, geom, sd, B, mt, upstream="ce", joint=False, seed=1234, label=""):
    """One keep-all-keys training step against the teacher-forced fp64 reference on the same upstream gradients."""
    x = synth.make_pixels(B, geom, seed=seed, kind="randn").cuda()
    gen = torch.Generator().manual_seed(seed)
    if joint:
        logits, _ = e.backbone_forward_train(x, mt, with_layer_losses=True)
    else:
        logits = e.backbone_forward_train(x, mt)
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
    rl, _, rs, rlosses = reference_forward_kv_all(p, x.double(), mt, geom.heads, forced_masks=masks, joint=joint)
    outputs, ups = [rl], [dlogits.double()]
    if joint:
        outputs.append(rlosses)
        ups.append(dlosses.double())
    ref = reference_grads(p, outputs, ups, joint)
    err = float((logits.double() - rl.detach()).abs().max())
    print(f"\n[{label}] logits max-abs err {err:.2e}")
    assert err < 1e-4
    _check_decisions(masks, rs, mt, label)
    _compare(got, ref, label)
    del p, rl, rs, rlosses, ref


# ------------------------------------------------------------------------------------------------ GPU: the matrix
@pytest.mark.gpu
@pytest.mark.parametrize("geom_name, B, mt, upstream", [
    ("deits16", 64, 0.5, "ce"),          # the natural ragged profile
    ("deits16", 64, 0.5, "randn"),       # upstream gradient without the zero row sums of cross-entropy
    ("deits16", 64, 1.5, "ce"),          # CLS only: one query against 197 keys per image
    ("vitb16", 48, 0.5, "ce"),           # D = 768
])
def test_kv_all_backbone_gradients_match_fp64(state_dicts, geom_name, B, mt, upstream):
    geom, sd = state_dicts(geom_name)
    e = _engine(geom, sd, B)
    try:
        _case(e, geom, sd, B, mt, upstream, label=f"kv_all {geom_name} B={B} mt={mt} {upstream}")
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("geom_name, B", [("vitb16", 32), ("deits16", 64)])
def test_kv_all_joint_objective_gradients_match_fp64(state_dicts, geom_name, B):
    """Cross-entropy plus the layers' compressor losses with distinct upstream gradients: backbone and compressors."""
    geom, sd = state_dicts(geom_name)
    e = _engine(geom, sd, B)
    try:
        _case(e, geom, sd, B, 0.5, "ce", joint=True, seed=99, label=f"kv_all joint {geom_name} B={B}")
    finally:
        e.close()


@pytest.mark.gpu
def test_kv_all_smaller_batches_on_a_larger_handle(state_dicts):
    geom, sd = state_dicts("deits16")
    e = _engine(geom, sd, 64)
    try:
        for i, B in enumerate((64, 37, 1)):
            _case(e, geom, sd, B, 0.5, "ce", seed=500 + i, label=f"kv_all max_batch 64, B={B}")
    finally:
        e.close()


def _step(e, x, mt, dlogits, between=None):
    e.backbone_forward_train(x, mt)
    if between is not None:
        between()
    flat = e.backbone_backward(dlogits)
    torch.cuda.synchronize()
    return flat


@pytest.mark.gpu
def test_kv_all_equals_active_when_every_token_is_active(state_dicts):
    """At mt 0.0 both modes do the same work: the keep-all-keys gradients equal the active-mode ones of the handle."""
    geom, sd = state_dicts("deits16")
    B = 16
    e = _engine(geom, sd, B)
    x = synth.make_pixels(B, geom, seed=61).cuda()
    dlogits = torch.randn(B, geom.classes, generator=torch.Generator().manual_seed(6)).cuda()
    try:
        kv_all = _step(e, x, 0.0, dlogits)
        e.set_kv_mode("active")
        active = _step(e, x, 0.0, dlogits)
        err = float((kv_all - active).abs().max()) / float(active.abs().max())
        print(f"\n[kv_all vs active at mt 0.0] relative max-abs {err:.2e}")
        assert err <= 1e-6
    finally:
        e.close()


@pytest.mark.gpu
def test_kv_all_backward_follows_the_forward_mode(state_dicts):
    """A keep-all-keys training forward, then set_kv_mode("active") with an inference forward and a compressor step in
    that mode, then the backward: the gradients are those of the keep-all-keys forward."""
    geom, sd = state_dicts("deits16")
    B, mt = 8, 0.5
    e = _engine(geom, sd, B)
    x1 = synth.make_pixels(B, geom, seed=71).cuda()
    x2 = synth.make_pixels(B, geom, seed=72).cuda()
    dlogits = torch.randn(B, geom.classes, generator=torch.Generator().manual_seed(7)).cuda()
    try:
        clean = _step(e, x1, mt, dlogits)

        def other_work():
            e.set_kv_mode("active")
            e.forward(x2, mt)
            e.compressor_grads(x2, mt)
        disturbed = _step(e, x1, mt, dlogits, other_work)
        err = float((disturbed - clean).abs().max()) / float(clean.abs().max())
        assert err <= 1e-5, f"gradients changed by a kv-mode switch between forward and backward: {err:.3e}"
        masks = e.backbone_train_masks()               # of the keep-all-keys forward of x1
        p = reference_params(sd, "cuda")
        rl, _, _, _ = reference_forward_kv_all(p, x1.double(), mt, geom.heads, forced_masks=masks)
        ref = reference_grads(p, [rl], [dlogits.double()], False)
        _compare(_flat_to_dict(disturbed, e.backbone_grad_slices()), ref, "kv_all: mode switch in between")
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: the drop-in
@pytest.mark.gpu
def test_kv_all_drop_in_cross_entropy_step_matches_fp64(state_dicts):
    """model.kv_mode = "all", vit_train(): the .grad of one cross-entropy step equal the fp64 reference's."""
    geom, sd = state_dicts("deits16")
    B, mt = 8, 0.5
    model = _drop_in_model(geom, sd, mt)
    model.kv_mode = "all"
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
    rl, _, rs, _ = reference_forward_kv_all(p, x.double(), mt, geom.heads, forced_masks=masks)
    ref = reference_grads(p, [rl], [lg.grad.double()], False)
    _check_decisions(masks, rs, mt, "kv_all drop-in")
    _compare({k: got[k] for k in ref}, ref, "kv_all drop-in cross-entropy step")


@pytest.mark.gpu
def test_kv_all_drop_in_train_both(state_dicts):
    """train(loss_type="both") for one epoch of two batches in keep-all-keys mode: finite losses, parameters move."""
    import main_model_utils
    geom, sd = state_dicts("deits16")
    B = 8
    model = _drop_in_model(geom, sd, 0.5)
    model.kv_mode = "all"
    before = {k: q.detach().clone() for k, q in model.named_parameters()}
    loader = main_model_utils.synthetic_loader(2 * B, B, geom=geom, seed=91)
    history = main_model_utils.train(model, loader, None, "cuda", num_epochs=1, loss_type="both")
    assert len(history) == 1 and np.isfinite(history[0]), history
    moved = [k for k, q in model.named_parameters() if not torch.equal(q.detach(), before[k])]
    assert any("mlp_layer" in k for k in moved) and any("attention.attention.key" in k for k in moved)


# ------------------------------------------------------------------------------------------------ GPU: compressor training
@pytest.mark.gpu
def test_kv_all_compressor_grads_match_fp64(state_dicts):
    """psv_compressor_grads on an fp32 handle in keep-all-keys mode = the gradients of sum(layer losses) of the fp64
    reference, teacher-forced with the masks of forward(want_masks=True) in the same mode."""
    geom, sd = state_dicts("deits16")
    B, mt = 64, 0.5
    e = _engine(geom, sd, B)
    x = synth.make_pixels(B, geom, seed=1234, kind="randn").cuda()
    try:
        masks = e.forward(x, mt, want_masks=True)["masks"].clone()
        cflat, loss = e.compressor_grads(x, mt)
        torch.cuda.synchronize()
        p = reference_params(sd, "cuda")
        _, _, rs, rlosses = reference_forward_kv_all(p, x.double(), mt, geom.heads, forced_masks=masks, joint=True)
        ref = reference_grads(p, [rlosses], [torch.ones_like(rlosses)], True)
        ref = {k: v for k, v in ref.items() if "mlp_layer" in k}
        _check_decisions(masks, rs, mt, "kv_all compressor_grads")
        lerr = float(((loss.double() - rlosses.detach()).abs() / rlosses.detach().abs()).max())
        print(f"\n[kv_all compressor_grads] layer-loss relative error {lerr:.2e}")
        assert lerr < 1e-4
        _compare(_comp_to_dict(cflat, geom), ref, "kv_all compressor_grads fp32")
    finally:
        e.close()


@pytest.mark.gpu
def test_kv_all_compressor_trainer_step_bf16(state_dicts):
    import main_model_utils
    geom, sd = state_dicts("deits16")
    B = 64
    e = _engine(geom, sd, B, "bf16")
    try:
        before = e.get_compressor_params().clone()
        trainer = main_model_utils.CompressorTrainer(e, mlp_threshold=0.5)
        loss = trainer.step(synth.make_pixels(B, geom, seed=1234, kind="randn").cuda())
        torch.cuda.synchronize()
        assert loss.shape == (geom.layers,) and bool(torch.isfinite(loss).all()), loss
        assert not torch.equal(e.get_compressor_params(), before)
    finally:
        e.close()
