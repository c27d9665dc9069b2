"""ViT-L/16 (hidden 1024, 16 heads of width 64, FFN 4096, 24 layers, 197 tokens) on every path: inference in both
precisions and kv modes and under both skip criteria, raw uint8 input, the tcgen05 GEMM at the ViT-L shapes,
compressor training and backbone fine-tuning.

The weights are synth.make_state_dict(synth.VIT_L16, seed=42), built here (the shared fixture knows DeiT-S and ViT-B).
On the CPU the oracle's layer, compressor and similarity are pinned at D = 1024 against transformers' own ViTLayer;
the goldens pin them at the other two widths.  On the GPU every comparison uses the bar of the matching DeiT-S / ViT-B
test; the measured ViT-L errors are printed beside it.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import preprocess_oracle as P
from oracle import vit_skip_oracle as O
from test_gpu_finetune_criteria import ST, U8_REL_TOL, _per_layer, _rel_frob, _sim_case
from test_gpu_finetune_fp64 import (_case, _check_decisions, _comp_to_dict, _compare, reference_forward, reference_grads,
                                    reference_params)
from test_gpu_finetune_kv_all import _case as _kv_all_case

GEOM = synth.VIT_L16
MT = 0.5
BAND = 1e-4


@pytest.fixture(scope="module")
def sd():
    return synth.make_state_dict(GEOM, seed=42)


def _engine(sd, precision, max_batch):
    import psv_native
    e = psv_native.Engine(GEOM, precision, max_batch)
    e.load_state_dict(sd)
    return e


# ------------------------------------------------------------------------------------------------ CPU: the oracle at D = 1024
def _hf_layer(sd, l):
    from transformers.models.vit.modeling_vit import ViTConfig, ViTLayer
    cfg = ViTConfig(hidden_size=GEOM.hidden, num_attention_heads=GEOM.heads, intermediate_size=GEOM.ffn,
                    num_hidden_layers=GEOM.layers, layer_norm_eps=GEOM.ln_eps)
    cfg._attn_implementation = "eager"
    layer = ViTLayer(cfg).eval()
    p = f"encoder.layer.{l}."
    own = {k[len(p):]: v for k, v in sd.items() if k.startswith(p) and not k.startswith(p + "mlp_layer.")}
    missing, unexpected = layer.load_state_dict(own, strict=True)
    assert not missing and not unexpected
    return layer


def test_oracle_matches_transformers_vit_layer_at_vitl16(sd):
    """oracle.vit_layer, compressor_scores and similarity at D = 1024 against transformers' ViTLayer (eager attention) and
    the reference's compressor module, both loaded with the same weights, on two layers: equal to fp32 rounding."""
    x = synth.make_pixels(2, GEOM, seed=5)
    with torch.no_grad():
        h = O.embed(sd, x)
        assert h.shape == (2, GEOM.tokens, GEOM.hidden)
        for l in (0, 1):
            dense = _hf_layer(sd, l)(h)
            dense = dense[0] if isinstance(dense, tuple) else dense
            ours = O.vit_layer(sd, l, h)
            err = float((ours - dense).abs().max())
            print(f"\n[layer {l}] vit_layer vs transformers ViTLayer: max-abs {err:.2e} (max |out| {float(dense.abs().max()):.2f})")
            assert err < 2e-5 * max(1.0, float(dense.abs().max()))
            # the reference's compressor (model_utils.py: Linear(2D, 64) -> ReLU -> Linear(64, 1) -> Sigmoid on [cls; token])
            comp = torch.nn.Sequential(torch.nn.Linear(2 * GEOM.hidden, GEOM.comp_hidden), torch.nn.ReLU(),
                                       torch.nn.Linear(GEOM.comp_hidden, 1), torch.nn.Sigmoid())
            comp.load_state_dict({k: sd[f"encoder.layer.{l}.mlp_layer.{k}"] for k in ("0.weight", "0.bias", "2.weight", "2.bias")})
            want = comp(torch.cat((h[:, :1].expand(-1, GEOM.patches, -1), h[:, 1:]), -1)).squeeze(-1)
            assert float((O.compressor_scores(sd, l, h) - want).abs().max()) < 1e-6
            # similarity of the dense output with the layer input (0.3 (cos + 1) / 2 + 0.7 / (1 + |y - h|^2 / |y|^2))
            real, cur = dense[:, 1:], h[:, 1:]
            want_sim = 0.3 * (F.cosine_similarity(real, cur, dim=-1) + 1) / 2 + \
                0.7 / (1 + ((real - cur) ** 2).sum(-1) / (real ** 2).sum(-1))
            assert float((O.similarity(ours, h) - want_sim).abs().max()) < 1e-5
            h = ours


def _psv_create_rc(hidden, heads):
    import psv_native
    cfg = psv_native.PsvConfig(hidden=hidden, heads=heads, ffn=4 * hidden, layers=2, tokens=197, classes=10, image=224,
                               patch=16, channels=3, comp_hidden=64, precision=psv_native.PSV_FP32, max_batch=2,
                               ln_eps=1e-12)
    h = ctypes.c_void_p()
    rc = psv_native.lib.psv_create(ctypes.byref(cfg), ctypes.byref(h))
    msg = psv_native.lib.psv_last_error(None).decode()
    if rc == 0:
        psv_native.lib.psv_destroy(h)
    return rc, msg


@pytest.mark.parametrize("hidden, heads", [(512, 8), (192, 3)])
def test_create_refuses_other_widths(hidden, heads):
    """psv_create checks the geometry before it looks for a device: any width but 384 / 768 / 1024 is unsupported, and
    the message names the three it covers."""
    rc, msg = _psv_create_rc(hidden, heads)
    assert rc == -4, (rc, msg)                                   # PSV_ERR_UNSUPPORTED
    assert "1024" in msg and "768" in msg and "384" in msg, msg


def test_create_accepts_vitl16_geometry():
    """hidden 1024 passes the geometry checks: a handle on a GPU, the no-device error without one."""
    rc, msg = _psv_create_rc(1024, 16)
    assert rc == (0 if torch.cuda.is_available() else -2), (rc, msg)


# ------------------------------------------------------------------------------------------------ GPU: inference
@pytest.fixture(scope="module")
def oracle64(sd):
    """The CPU oracle's free-running forward of 64 randn images (the first 16 serve the batch-16 cases)."""
    x = synth.make_pixels(64, GEOM, seed=1234)
    with torch.no_grad():
        return x, O.forward(sd, x, MT, 0.9)


def _band(scores):
    return torch.cat((torch.zeros(*scores.shape[:-1], 1, dtype=torch.bool), (scores - MT).abs() < BAND), -1)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [16, 64])
def test_fp32_free_running_against_oracle(sd, oracle64, B):
    """fp32, own decisions: masks bit-exact outside the 1e-4 band, logits within 1e-4 and the same top-1 on every image
    whose decisions all agree."""
    x, ref = oracle64
    x = x[:B]
    e = _engine(sd, "fp32", B)
    try:
        for use_graph in (False, True):
            r = e.forward(x.cuda(), MT, want_masks=True, want_scores=True, use_graph=use_graph)
            torch.cuda.synchronize()
            diff = r["masks"].cpu().bool() != ref.masks[:, :B]
            assert not (diff & ~_band(ref.scores[:, :B])).any(), "fp32 mask flip outside the 1e-4 band"
            clean = ~diff.any(0).any(1)
            err = float((r["logits"].cpu() - ref.logits[:B])[clean].abs().max())
            print(f"\n[fp32 B={B} graph={use_graph}] {int(diff.sum())} in-band flips, {int(clean.sum())} clean images, "
                  f"logits max-abs err {err:.2e}; {float(ref.masks[:, :B, 1:].float().mean()):.1%} of patch tokens active")
            assert int(clean.sum()) >= B - 2 and err < 1e-4
            assert torch.equal(r["logits"].cpu()[clean].argmax(-1), ref.logits[:B][clean].argmax(-1))
    finally:
        e.close()


@pytest.mark.gpu
def test_bf16_logits_teacher_forced(sd, oracle64):
    """bf16 with the oracle's masks: logits within 2e-2; top-1 agreement on every image whose oracle top-2 margin exceeds
    twice that (random-init classifier margins are often below the tolerance)."""
    x, ref = oracle64
    e = _engine(sd, "bf16", 64)
    try:
        for attention in ("auto", "tc", "pk"):
            e.set_attention_kernel(attention)
            r = e.forward(x.cuda(), MT, forced_masks=ref.masks.to(torch.uint8).cuda(), want_masks=True, use_graph=True)
            torch.cuda.synchronize()
            assert torch.equal(r["masks"].cpu().bool(), ref.masks)
            lg = r["logits"].cpu()
            err = float((lg - ref.logits).abs().max())
            top2 = ref.logits.topk(2, dim=1).values
            decided = (top2[:, 0] - top2[:, 1]) > 4e-2
            agree = lg.argmax(1) == ref.logits.argmax(1)
            print(f"\n[bf16 attention={attention}] teacher-forced logits max-abs err {err:.4f}; top-1 agreement "
                  f"{float(agree.float().mean()):.2%} raw, {int(agree[decided].sum())} of {int(decided.sum())} decided")
            assert err < 2e-2
            assert bool(agree[decided].all())
    finally:
        e.close()


@pytest.mark.gpu
def test_bf16_layers_on_oracle_inputs(sd):
    """Every layer fed the oracle's fp32 layer input: split-bf16 compressor scores within 2e-5, masks exact outside the
    band, the compaction of the mask it used, and the teacher-forced layer output within the bf16 layer bar."""
    B = 3
    e = _engine(sd, "bf16", B)
    x = synth.make_pixels(B, GEOM, seed=21)
    worst_s = worst_out = 0.0
    try:
        with torch.no_grad():
            h = O.embed(sd, x)
            for l in range(GEOM.layers):
                out, mask, scores = O.layer_forward(sd, l, h, MT)
                m_free, s_free, n_free = e.layer_forward(l, h.cuda().contiguous(), MT)
                torch.cuda.synchronize()
                s_err = float((s_free.cpu() - scores).abs().max())
                worst_s = max(worst_s, s_err)
                assert s_err < 2e-5, f"layer {l}: score err {s_err}"
                assert not ((m_free.cpu().bool() != mask) & ~_band(scores)).any(), f"layer {l}: flip outside the band"
                assert torch.equal(n_free.cpu().long(), m_free.cpu().long().sum(1))
                idx_gpu, cu_gpu = e.get_compaction(B)
                idx, cu, _ = O.compact(m_free.cpu().bool())
                assert torch.equal(cu_gpu.cpu(), cu) and torch.equal(idx_gpu.cpu()[:int(cu[-1])], idx)
                hg = h.cuda().contiguous()
                e.layer_forward(l, hg, MT, forced_mask=mask.to(torch.uint8).cuda())
                torch.cuda.synchronize()
                err = float((hg.cpu() - out).abs().max())
                worst_out = max(worst_out, err)
                assert err < 3e-2, f"layer {l}: {err}"
                assert torch.equal(hg.cpu()[~mask], h[~mask])
                h = out
    finally:
        e.close()
    print(f"\n[bf16 per layer] worst score err {worst_s:.2e}, worst teacher-forced layer output err {worst_out:.4f}")


@pytest.mark.gpu
def test_bf16_one_call_equals_per_layer_path(sd):
    """psv_forward, eager and as a CUDA graph, is bit-equal to embed -> layer_forward per layer -> head (one attention
    kernel for both: "auto" may choose per call)."""
    B = 16
    e = _engine(sd, "bf16", B)
    e.set_attention_kernel("pk")
    x = synth.make_pixels(B, GEOM, seed=4321).cuda()
    try:
        for use_graph in (False, True, True):
            r = e.forward(x, MT, want_masks=True, use_graph=use_graph)
            logits, masks = r["logits"].clone(), r["masks"].clone()
            h = e.embed(x)
            per = [e.layer_forward(l, h, MT)[0] for l in range(GEOM.layers)]
            ref_logits = e.head(h)
            torch.cuda.synchronize()
            assert torch.equal(masks, torch.stack(per))
            assert torch.equal(logits, ref_logits), float((logits - ref_logits).abs().max())
    finally:
        e.close()


@pytest.mark.gpu
def test_bf16_shard_equals_half_batch(sd):
    """A batch of 256 and its two halves of 128: logits, masks and active counts bit-equal; two runs identical."""
    B = 256
    e = _engine(sd, "bf16", B)
    x = synth.make_pixels(B, GEOM, seed=99).cuda()
    keys = ("logits", "masks", "n_active")
    try:
        full = e.forward(x, MT, want_masks=True, want_n_active=True, use_graph=True)
        torch.cuda.synchronize()
        full = {k: full[k].clone() for k in keys}
        again = e.forward(x, MT, want_masks=True, want_n_active=True, use_graph=True)
        torch.cuda.synchronize()
        assert all(torch.equal(full[k], again[k]) for k in keys)
        for lo in (0, 128):
            part = e.forward(x[lo:lo + 128].contiguous(), MT, want_masks=True, want_n_active=True)
            torch.cuda.synchronize()
            assert torch.equal(part["masks"], full["masks"][:, lo:lo + 128])
            assert torch.equal(part["n_active"], full["n_active"][:, lo:lo + 128])
            assert torch.equal(part["logits"], full["logits"][lo:lo + 128])
        print(f"\n[bf16 B=256] {float((full['n_active'].float().mean() - 1) / GEOM.patches):.1%} of patch tokens active")
    finally:
        e.close()


GEMM_SHAPES = [
    # m, n, k, gelu, residual, out_fp32
    (77, 3072, 1024, False, False, False),            # QKV, bf16 out
    (16 * 197, 3072, 1024, False, False, False),
    (128 * 150 - 5, 3072, 1024, False, False, False),  # 12 full waves of 148 tiles and a tail
    (77, 1024, 1024, False, True, True),              # proj, residual epilogue
    (128 * 170 + 5, 1024, 1024, False, True, True),
    (333, 4096, 1024, True, False, False),            # FC1 + GELU
    (128 * 150 - 3, 4096, 1024, True, False, False),
    (200, 1024, 4096, False, True, True),             # FC2, K = 4096 (64 k-blocks)
    (16 * 197, 1024, 4096, False, True, True),
]


@pytest.fixture(scope="module")
def bf16_engine(sd):
    e = _engine(sd, "bf16", 4)
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,k,gelu,use_res,out_fp32", GEMM_SHAPES)
def test_gemm_at_vitl16_shapes(bf16_engine, m, n, k, gelu, use_res, out_fp32):
    torch.manual_seed(m * 7 + n + k)
    a = torch.randn(m, k, device="cuda").to(torch.bfloat16)
    w = (torch.randn(n, k, device="cuda") * (k ** -0.5)).to(torch.bfloat16)
    bias = torch.randn(n, device="cuda")
    res = torch.randn(m, n, device="cuda") if use_res else None
    out = bf16_engine.gemm(a, w, bias, res, out_fp32=out_fp32, gelu=gelu)
    torch.cuda.synchronize()
    ref = a.double() @ w.double().t() + bias.double()
    if gelu:
        ref = F.gelu(ref)
    if use_res:
        ref = ref + res.double()
    err = float((out.double() - ref).abs().max())
    tol = 2e-4 if out_fp32 else 2e-2 * max(1.0, float(ref.abs().max()))
    assert err < tol, f"max err {err} (tol {tol})"


@pytest.mark.gpu
def test_kv_all_against_query_pruned_oracle(sd):
    """Keep-all-keys mode, fp32: layers on the oracle's inputs against oracle.vit_layer_query_pruned (via
    layer_forward(kv_all=True)), then the whole forward on its own decisions."""
    B = 3
    e = _engine(sd, "fp32", B)
    e.set_kv_mode("all")
    x = synth.make_pixels(B, GEOM, seed=55)
    try:
        with torch.no_grad():
            o = O.forward(sd, x, MT, keep_hidden=True, kv_all=True)
        hidden_in = [O.embed(sd, x)] + o.hidden[:-1]
        worst = 0.0
        for l in (0, 1, 12, 23):
            h = hidden_in[l].clone().cuda()
            e.layer_forward(l, h, MT, forced_mask=o.masks[l].to(torch.uint8).cuda())
            torch.cuda.synchronize()
            out = h.cpu()
            worst = max(worst, float((out - o.hidden[l]).abs().max()))
            assert torch.equal(out[~o.masks[l]], hidden_in[l][~o.masks[l]])
        print(f"\n[kv all] layer outputs max-abs err {worst:.2e}")
        assert worst < 1e-4
        for use_graph in (False, True):
            r = e.forward(x.cuda(), MT, want_masks=True, use_graph=use_graph)
            torch.cuda.synchronize()
            diff = r["masks"].cpu().bool() != o.masks
            assert not (diff & ~_band(o.scores)).any()
            clean = ~diff.any(0).any(1)
            assert int(clean.sum()) >= 2
            assert float((r["logits"].cpu() - o.logits)[clean].abs().max()) < 1e-4
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_similarity_one_call_equals_per_layer(sd, precision):
    """Under the similarity criterion psv_forward (eager and graph) is bit-equal to similarity_mask + layer_forward per
    layer."""
    B = 8
    e = _engine(sd, precision, B)
    e.set_skip_criterion("similarity", ST)
    if precision == "bf16":
        e.set_attention_kernel("pk")
    x = synth.make_pixels(B, GEOM, seed=1234).cuda()
    try:
        for use_graph in (False, True):
            r = e.forward(x, MT, want_masks=True, use_graph=use_graph)
            logits, masks = r["logits"].clone(), r["masks"].clone()
            ref_logits, ref_masks = _per_layer(e, x, ST)
            torch.cuda.synchronize()
            print(f"\n[similarity {precision} graph={use_graph}] skipped {1.0 - float(masks[:, :, 1:].double().mean()):.2f}")
            assert torch.equal(masks, ref_masks), int((masks != ref_masks).sum())
            assert torch.equal(logits, ref_logits), float((logits - ref_logits).abs().max())
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_u8_input_equals_preprocessed_pixels(sd, precision):
    B = 4
    e = _engine(sd, precision, B)
    rng = np.random.default_rng(7)
    try:
        for hw in ((32, 32), (224, 224)):
            imgs = rng.integers(0, 256, size=(B, hw[0], hw[1], 3), dtype=np.uint8)
            ref_pixels = torch.from_numpy(P.preprocess_u8(imgs)).cuda()
            e.set_u8_input(*hw)
            u8 = torch.from_numpy(imgs).cuda()
            assert torch.equal(e.embed(u8), e.embed(ref_pixels))
            for use_graph in (False, True):
                a = e.forward(u8, MT, want_masks=True, use_graph=use_graph)
                b = e.forward(ref_pixels, MT, want_masks=True, use_graph=use_graph)
                torch.cuda.synchronize()
                assert torch.equal(a["masks"], b["masks"]) and torch.equal(a["logits"], b["logits"])
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: compressor training
@pytest.mark.gpu
def test_compressor_grads_fp32_match_fp64(sd):
    """psv_compressor_grads on an fp32 handle = the gradients of the sum of the layer losses of the fp64 reference,
    teacher-forced with the forward's masks."""
    B = 16
    e = _engine(sd, "fp32", B)
    x = synth.make_pixels(B, GEOM, seed=1234).cuda()
    try:
        masks = e.forward(x, MT, want_masks=True)["masks"].clone()
        cflat, loss = e.compressor_grads(x, MT)
        torch.cuda.synchronize()
        p = reference_params(sd, "cuda")
        _, _, rs, rlosses = reference_forward(p, x.double(), MT, GEOM.heads, forced_masks=masks, joint=True)
        ref = {k: v for k, v in reference_grads(p, [rlosses], [torch.ones_like(rlosses)], True).items() if "mlp_layer" in k}
        _check_decisions(masks, rs, MT, "vitl16 compressor_grads fp32")
        lerr = float(((loss.double() - rlosses.detach()).abs() / rlosses.detach().abs()).max())
        print(f"\n[vitl16 compressor_grads fp32] layer-loss relative error {lerr:.2e}")
        assert lerr < 1e-4
        _compare(_comp_to_dict(cflat, GEOM), ref, "vitl16 compressor_grads fp32")
    finally:
        e.close()


@pytest.mark.gpu
def test_compressor_grads_bf16_layer0_match_fp64(sd):
    """bf16 handle: the layer-0 block of psv_compressor_grads (pre-activations from the split-bf16 score kernel, light
    backward) against the fp64 autograd of that layer's loss on the handle's own layer-0 input and mask."""
    B = 16
    e = _engine(sd, "bf16", B)
    x = synth.make_pixels(B, GEOM, seed=17).cuda()
    try:
        cflat, loss = e.compressor_grads(x, MT)
        h0 = e.embed(x)
        mask, _, _ = e.layer_forward(0, h0.clone(), MT)
        torch.cuda.synchronize()
        assert bool(torch.isfinite(loss).all())
        pre = "encoder.layer.0.mlp_layer."
        p = {k: sd[pre + k].to("cuda", torch.float64).requires_grad_(True) for k in ("0.weight", "0.bias", "2.weight", "2.bias")}
        h = h0.double()
        z = torch.cat((h[:, :1].expand(-1, GEOM.patches, -1), h[:, 1:]), -1)
        s = torch.sigmoid(F.linear(F.relu(F.linear(z, p["0.weight"], p["0.bias"])), p["2.weight"], p["2.bias"])).squeeze(-1)
        labels = mask[:, 1:].double()
        mean = labels.mean()
        l0 = F.binary_cross_entropy_with_logits(s, labels, pos_weight=(mean / (1 - mean + 1e-16)).reshape(1))
        gs = torch.autograd.grad(l0, list(p.values()))
        ref = {pre + k: g.detach() for k, g in zip(p, gs)}
        got = {k: v for k, v in _comp_to_dict(cflat, GEOM).items() if k.startswith(pre)}
        print(f"\n[vitl16 compressor_grads bf16] layer-0 loss {float(loss[0]):.6f} vs fp64 {float(l0):.6f}")
        assert abs(float(loss[0]) - float(l0)) <= 1e-4 * abs(float(l0))
        _compare(got, ref, "vitl16 compressor_grads bf16 layer 0")
    finally:
        e.close()


@pytest.mark.gpu
def test_compressor_trainer_step_bf16(sd):
    import main_model_utils
    B = 16
    e = _engine(sd, "bf16", B)
    try:
        before = e.get_compressor_params().clone()
        trainer = main_model_utils.CompressorTrainer(e, mlp_threshold=MT)
        loss = trainer.step(synth.make_pixels(B, GEOM, seed=1234).cuda())
        torch.cuda.synchronize()
        assert loss.shape == (GEOM.layers,) and bool(torch.isfinite(loss).all()), loss
        assert not torch.equal(e.get_compressor_params(), before)
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: backbone fine-tuning
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["ce", "joint", "kv_all", "similarity"])
def test_backbone_gradients_match_fp64(sd, mode):
    """Every gradient tensor of one training step at batch 16 against the fp64 autograd reference, teacher-forced with
    the training forward's masks; decisions outside the band equal the fp64 ones."""
    B = 16
    e = _engine(sd, "fp32", B)
    try:
        if mode == "ce":
            _case(e, GEOM, sd, B, MT, "ce", label="vitl16 B=16 ce")
        elif mode == "joint":
            _case(e, GEOM, sd, B, MT, "ce", joint=True, seed=99, label="vitl16 joint B=16")
        elif mode == "kv_all":
            e.set_kv_mode("all")
            _kv_all_case(e, GEOM, sd, B, MT, "ce", label="vitl16 kv_all B=16")
        else:
            e.set_skip_criterion("similarity", ST)
            _sim_case(e, GEOM, sd, B, "ce", label="vitl16 similarity B=16")
    finally:
        e.close()


@pytest.mark.gpu
def test_u8_training_step_equals_preprocessed_step(sd):
    """One training step on raw uint8 32 x 32 images against the same step on the preprocessed fp32 pixels: logits and
    masks bit-equal, gradients within 1e-6."""
    B = 8
    e = _engine(sd, "fp32", B)
    rng = np.random.default_rng(31)
    imgs = rng.integers(0, 256, size=(B, 32, 32, 3), dtype=np.uint8)
    u8, ref_pixels = torch.from_numpy(imgs).cuda(), torch.from_numpy(P.preprocess_u8(imgs)).cuda()
    dlogits = torch.randn(B, GEOM.classes, generator=torch.Generator().manual_seed(3)).cuda()
    try:
        e.set_u8_input(32, 32)
        lu = e.backbone_forward_train(u8, MT).clone()
        mu = e.backbone_train_masks().clone()
        gu = e.backbone_backward(dlogits).clone()
        lf = e.backbone_forward_train(ref_pixels, MT).clone()
        mf = e.backbone_train_masks().clone()
        gf = e.backbone_backward(dlogits).clone()
        torch.cuda.synchronize()
        assert torch.equal(lu, lf) and torch.equal(mu, mf)
        err = _rel_frob(gu, gf, e.backbone_grad_slices())
        print(f"\n[vitl16 u8 step] gradients vs fp32 pixels {err:.2e}")
        assert err <= U8_REL_TOL
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: the drop-in
def _model(sd):
    import model_utils
    from transformers.models.vit.modeling_vit import ViTConfig
    cfg = ViTConfig(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
                    num_labels=100)
    model = model_utils.ModifiedViTModel(cfg, 0.9, 0.5, 0)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not missing and not unexpected
    return model.to("cuda")


@pytest.mark.gpu
def test_drop_in_inference_paths(sd, oracle64):
    """ModifiedViTModel with the ViT-L config: the one-call path against the oracle, and the per-layer path
    (compute_cosine, output_hidden_states) against the one-call path."""
    x, ref = oracle64
    x, B = x[:4].cuda(), 4
    model = _model(sd).eval()
    with torch.no_grad():
        one = model(x, output_mask=True)
        masks = torch.stack(one.boolean_masks).cpu()
        diff = masks != ref.masks[:, :B]
        assert not (diff & ~_band(ref.scores[:, :B])).any()
        clean = ~diff.any(0).any(1)
        assert float((one.logits.cpu() - ref.logits[:B])[clean].abs().max()) < 1e-4
        per = model(x, output_mask=True, compute_cosine=True, output_hidden_states=True)
        assert all(torch.equal(a, b) for a, b in zip(one.boolean_masks, per.boolean_masks))
        assert float((one.logits - per.logits).abs().max()) < 1e-4
        assert len(per.hidden_states) == GEOM.layers + 1
        for layer in model.encoder.layer:
            assert np.isfinite(float(layer.loss)) and layer.mlp_confusion_matrix.shape == (2, 2)


@pytest.mark.gpu
def test_drop_in_compressor_trainer(sd):
    import main_model_utils
    model = _model(sd).eval()
    x = synth.make_pixels(4, GEOM, seed=3).cuda()
    with torch.no_grad():
        model(x)
    tr = main_model_utils.CompressorTrainer(model._psv_engine, mlp_threshold=0.5, lr=1e-3)
    losses = [tr.step(x) for _ in range(2)]
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(l).all()) for l in losses)


@pytest.mark.gpu
@pytest.mark.parametrize("loss_type", ["cosine", "classification", "both", "alternate"])
def test_drop_in_train(sd, loss_type):
    """train() for one epoch of two batches of four in each loss type: finite losses, the trained parameters move."""
    import main_model_utils
    model = _model(sd)
    model.psv_precision = "fp32"
    before = {k: q.detach().clone() for k, q in model.named_parameters()}
    loader = main_model_utils.synthetic_loader(8, 4, geom=GEOM, seed=91, kind="randn", pin_memory=False)
    history = main_model_utils.train(model, loader, None, "cuda", num_epochs=1, loss_type=loss_type)
    assert len(history) == 1 and np.isfinite(history[0]), history
    moved = [k for k, q in model.named_parameters() if not torch.equal(q.detach(), before[k])]
    if loss_type in ("cosine", "alternate", "both"):            # "alternate" trains the compressors in epoch 0
        assert any("mlp_layer" in k for k in moved)
    if loss_type in ("classification", "both"):
        assert any("attention.attention.key" in k for k in moved)
