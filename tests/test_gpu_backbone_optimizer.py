"""The backbone optimizer step inside the library (psv_backbone_adam_step and its sharded peer-memory form) and
BackboneTrainer.

CPU: the shard rule, and planted defects in an fp64 Adam model against torch.optim.Adam / AdamW -- each defect must
exceed the GPU bar below by at least 2x.
GPU: five steps on real DeiT-S backward gradients against torch.optim.Adam / AdamW (foreach=False) tensor by tensor;
frozen tensors and per-tensor step counters; every forward path reads the new weights; checkpoint / resume is
bit-exact; refusals; BackboneTrainer against the drop-in's torch path; on two GPUs, tools/backbone_p2p_check.py."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import synth

# |native - torch| <= ULP_BAR * 2^-23 * max|p| per tensor after five steps.  Worst value measured on a B200 (1000 W):
# 2.44 over two runs (Adam 2.36, AdamW 2.40, grad_scale 0.37 2.44, classifier first then all 1.95).
ULP_BAR = 8.0
EPS32 = 2.0 ** -23
LR = 1e-3


def _param_count(geom):
    D, F, N, KP = geom.hidden, geom.ffn, geom.tokens, geom.channels * geom.patch * geom.patch
    per = 2 * D + 3 * D * D + 3 * D + D * D + D + 2 * D + F * D + F + D * F + D
    return D + N * D + D * KP + D + geom.layers * per + 2 * D + geom.classes * D + geom.classes


# ------------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("geom", [synth.VIT_B16, synth.DEIT_S16, synth.VIT_L16], ids=["vitb16", "deits16", "vitl16"])
def test_shard_rule_covers_the_vector(geom):
    import psv_native
    base = _param_count(geom)
    for n in (base, base + 1, base + 2, base + 3, 5):
        for world in range(1, 17):
            prev = 0
            for rank in range(world):
                lo, hi = psv_native.backbone_shard(n, world, rank)
                assert lo == prev and lo <= hi and lo % 4 == 0
                assert hi % 4 == 0 or (rank == world - 1 and hi == n)
                prev = hi
            assert prev == n
    for bad in ((base, 0, 0), (base, 17, 0), (base, 2, 2), (base, 2, -1), (-1, 1, 0)):
        with pytest.raises(psv_native.PsvError):
            psv_native.backbone_shard(*bad)


def _adam_fp64(params, grads_seq, steps_seq, lr, betas, eps, wd, defect=None):
    """fp64 Adam / AdamW with per-tensor steps (0 = frozen); `defect` plants one known mistake."""
    b1, b2 = betas
    p = [x.clone() for x in params]
    m = [torch.zeros_like(x) for x in params]
    v = [torch.zeros_like(x) for x in params]
    for grads, steps in zip(grads_seq, steps_seq):
        for i, (g, st) in enumerate(zip(grads, steps)):
            if st == 0:
                if defect == "frozen_moments":
                    m[i] = b1 * m[i] + (1 - b1) * g
                    v[i] = b2 * v[i] + (1 - b2) * g * g
                continue
            if wd:
                if defect == "l2_decay":
                    g = g + wd * p[i]
                else:
                    p[i] = p[i] * (1 - lr * wd)
            m[i] = b1 * m[i] + (1 - b1) * g
            v[i] = b2 * v[i] + (1 - b2) * g * g
            s = st + 1 if defect == "bias_step" else st
            bc1, bc2 = 1 - b1 ** s, 1 - b2 ** s
            denom = (v[i] / bc2 + eps).sqrt() if defect == "eps_in_sqrt" else v[i].sqrt() / bc2 ** 0.5 + eps
            p[i] = p[i] - lr / bc1 * m[i] / denom
    return p


def _torch_adam(params, grads_seq, steps_seq, lr, betas, eps, wd):
    p = [x.clone().requires_grad_(True) for x in params]
    opt = (torch.optim.AdamW if wd else torch.optim.Adam)(p, lr=lr, betas=betas, eps=eps, weight_decay=wd,
                                                         foreach=False)
    for grads, steps in zip(grads_seq, steps_seq):
        for x, g, st in zip(p, grads, steps):
            x.grad = g.clone() if st else None
        opt.step()
    return [x.detach() for x in p]


def _cpu_case():
    gen = torch.Generator().manual_seed(7)
    shapes = [(64, 48), (48,), (32, 32), (96,)]
    params = [torch.randn(s, generator=gen, dtype=torch.float64) * sc for s, sc in zip(shapes, (0.02, 1.0, 0.05, 0.1))]
    # gradient scales from 1e-6 to 1e-2, as across the tensors of a real backward
    grads_seq = [[torch.randn(s, generator=gen, dtype=torch.float64) * sc for s, sc in zip(shapes, (1e-3, 1e-5, 1e-2, 1e-6))]
                 for _ in range(5)]
    steps_seq = [[1, 0, 1, 1], [2, 0, 2, 2], [3, 0, 3, 3], [4, 1, 4, 4], [5, 2, 5, 5]]   # tensor 1 frozen for 3 steps
    return params, grads_seq, steps_seq


def _worst_ulps(got, ref):
    return max(float((a - b).abs().max()) / (EPS32 * float(b.abs().max())) for a, b in zip(got, ref))


@pytest.mark.parametrize("wd", [0.0, 0.05])
def test_planted_defects_exceed_the_bar(wd):
    params, grads_seq, steps_seq = _cpu_case()
    betas, eps = (0.9, 0.999), 1e-8
    ref = _torch_adam(params, grads_seq, steps_seq, LR, betas, eps, wd)
    assert _worst_ulps(_adam_fp64(params, grads_seq, steps_seq, LR, betas, eps, wd), ref) < 1e-6
    defects = ["bias_step", "eps_in_sqrt", "frozen_moments"] + (["l2_decay"] if wd else [])
    for d in defects:
        err = _worst_ulps(_adam_fp64(params, grads_seq, steps_seq, LR, betas, eps, wd, defect=d), ref)
        assert err >= 2 * ULP_BAR, (d, err)


# ------------------------------------------------------------------------------------------------------------------ GPU
def _engine(geom, sd, batch, precision="fp32"):
    import psv_native
    e = psv_native.Engine(geom, precision, batch)
    e.load_state_dict(sd)
    return e


def _grad_sequence(geom, sd, batch=8, k=5):
    """k real backward gradients of DeiT-S (cross-entropy on random labels, different batches, fixed weights)."""
    e = _engine(geom, sd, batch)
    seq = []
    for i in range(k):
        x = synth.make_pixels(batch, geom, seed=300 + i, kind="randn").cuda()
        y = torch.randint(0, geom.classes, (batch,), generator=torch.Generator().manual_seed(i)).cuda()
        lg = e.backbone_forward_train(x, 0.5).detach().requires_grad_(True)
        dl, = torch.autograd.grad(torch.nn.functional.cross_entropy(lg, y), lg)
        seq.append(e.backbone_backward(dl).clone())
    torch.cuda.synchronize()
    e.close()
    return seq


def _torch_steps(sd, slices, seq, steps_seq, wd, grad_scale):
    keys = list(slices)
    p = {k: sd[k].detach().float().cuda().clone().requires_grad_(True) for k in keys}
    opt = (torch.optim.AdamW if wd else torch.optim.Adam)(list(p.values()), lr=LR, weight_decay=wd, foreach=False)
    for g, steps in zip(seq, steps_seq):
        for k, st in zip(keys, steps):
            off, shape = slices[k]
            n = int(np.prod(shape))
            p[k].grad = (g[off:off + n].reshape(p[k].shape) * grad_scale) if st else None
        opt.step()
    return {k: v.detach() for k, v in p.items()}


@pytest.fixture(scope="module")
def deits(state_dicts):
    geom, sd = state_dicts("deits16")
    return geom, sd, _grad_sequence(geom, sd)


def _compare(e, ref, label):
    got = e.export_backbone_state_dict()
    worst = 0.0
    for k, r in ref.items():
        err = float((got[k].reshape(r.shape) - r).abs().max())
        ulps = err / (EPS32 * float(r.abs().max()))
        worst = max(worst, ulps)
        assert ulps <= ULP_BAR, (label, k, ulps)
    print(f"{label}: worst {worst:.2f} ulps of max|p| (bar {ULP_BAR})")
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("wd, grad_scale", [(0.0, 1.0), (0.05, 1.0), (0.0, 0.37)], ids=["adam", "adamw", "scaled"])
def test_adam_matches_torch(deits, wd, grad_scale):
    geom, sd, seq = deits
    e = _engine(geom, sd, 8)
    slices = e.backbone_grad_slices()
    nt = len(slices)
    steps_seq = [[t + 1] * nt for t in range(len(seq))]
    for g, steps in zip(seq, steps_seq):
        e.backbone_adam_step(g, steps, lr=LR, weight_decay=wd, grad_scale=grad_scale)
    ref = _torch_steps(sd, slices, seq, steps_seq, wd, grad_scale)
    _compare(e, ref, f"wd {wd} grad_scale {grad_scale}")
    e.close()


@pytest.mark.gpu
def test_frozen_tensors_and_per_tensor_steps(deits):
    """classifier alone for 3 steps, then everything for 2: frozen tensors and their moments stay bit-identical, and the
    result matches torch, whose classifier counter runs ahead."""
    geom, sd, seq = deits
    e = _engine(geom, sd, 8)
    slices = e.backbone_grad_slices()
    keys = list(slices)
    before = e.get_backbone_params().clone()
    cls = [k.startswith("classifier.") for k in keys]
    steps_seq = [[t + 1 if c else 0 for c in cls] for t in range(3)] + [[t + 4 if c else t + 1 for c in cls]
                                                                          for t in range(2)]
    for t in range(3):
        e.backbone_adam_step(seq[t], steps_seq[t], lr=LR)
    after = e.get_backbone_params()
    m, v = e.get_backbone_adam_state()
    lo = slices["classifier.weight"][0]
    assert torch.equal(after[:lo], before[:lo])
    assert not torch.equal(after[lo:], before[lo:])
    assert int(torch.count_nonzero(m[:lo])) == 0 and int(torch.count_nonzero(v[:lo])) == 0
    for t in range(3, 5):
        e.backbone_adam_step(seq[t], steps_seq[t], lr=LR)
    ref = _torch_steps(sd, slices, seq, steps_seq, 0.0, 1.0)
    _compare(e, ref, "frozen then all")
    e.close()


def _comp_sd(sd):
    return {k: v for k, v in sd.items() if "mlp_layer" in k}


@pytest.mark.gpu
def test_new_weights_reach_every_forward_path(deits):
    """After native steps every forward path gives exactly what a fresh handle loaded with the exported weights gives:
    no stale copy of a weight is left anywhere (eager forward, a graph captured BEFORE the steps, per-layer path,
    training forward in split and bf16 mode)."""
    geom, sd, seq = deits
    B = 8
    x = synth.make_pixels(B, geom, seed=77, kind="randn").cuda()
    e = _engine(geom, sd, B)
    e.forward(x, 0.5, use_graph=True)                       # captured before the steps
    nt = len(e.backbone_grad_slices())
    for t, g in enumerate(seq):
        e.backbone_adam_step(g, [t + 1] * nt, lr=LR, weight_decay=0.05)
    fresh = _engine(geom, {**e.export_backbone_state_dict(), **_comp_sd(sd)}, B)
    assert torch.equal(fresh.get_backbone_params(), e.get_backbone_params())

    def per_layer(eng):
        h = eng.embed(x)
        for layer in range(geom.layers):
            eng.layer_forward(layer, h, 0.5)
        return eng.head(h)

    got_graph = e.forward(x, 0.5, use_graph=True)["logits"].clone()
    assert torch.equal(got_graph, fresh.forward(x, 0.5, use_graph=True)["logits"])
    assert torch.equal(e.forward(x, 0.5)["logits"], fresh.forward(x, 0.5)["logits"])
    assert not torch.equal(got_graph, _engine(geom, sd, B).forward(x, 0.5)["logits"])    # the steps did move the model
    assert torch.equal(per_layer(e), per_layer(fresh))
    for mode in ("split", "bf16"):
        e.set_train_precision(mode)
        fresh.set_train_precision(mode)
        assert torch.equal(e.backbone_forward_train(x, 0.5), fresh.backbone_forward_train(x, 0.5)), mode
    e.close()
    fresh.close()


@pytest.mark.gpu
def test_checkpoint_resume_is_bit_exact(deits):
    geom, sd, seq = deits
    straight = _engine(geom, sd, 8)
    nt = len(straight.backbone_grad_slices())
    for t, g in enumerate(seq):
        straight.backbone_adam_step(g, [t + 1] * nt, lr=LR, weight_decay=0.05)
    first = _engine(geom, sd, 8)
    for t in range(3):
        first.backbone_adam_step(seq[t], [t + 1] * nt, lr=LR, weight_decay=0.05)
    params, (m, v) = first.get_backbone_params(), first.get_backbone_adam_state()
    half = first.backbone_param_count // 2
    m_hi, v_hi = first.get_backbone_adam_state(half, first.backbone_param_count)
    assert torch.equal(m_hi, m[half:]) and torch.equal(v_hi, v[half:])
    resumed = _engine(geom, {**{k: params[o:o + int(np.prod(s))].reshape(s)
                                for k, (o, s) in first.backbone_grad_slices().items()}, **_comp_sd(sd)}, 8)
    resumed.set_backbone_adam_state(m[:half], v[:half])
    resumed.set_backbone_adam_state(m[half:], v[half:], lo=half)
    for t in range(3, 5):
        resumed.backbone_adam_step(seq[t], [t + 1] * nt, lr=LR, weight_decay=0.05)
    assert torch.equal(resumed.get_backbone_params(), straight.get_backbone_params())
    for a, b in zip(resumed.get_backbone_adam_state(), straight.get_backbone_adam_state()):
        assert torch.equal(a, b)
    for x in (straight, first, resumed):
        x.close()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_step_on_one_gpu_equals_the_local_step(deits, world):
    """The sharded reduce + update + gather with `world` engines on one GPU (the peer pointers are plain device
    pointers): every replica is bit-equal to one engine stepping on the rank-order fp32 sum of the buckets, and the
    frozen tensors (here the embeddings) stay unchanged through the parameter buckets."""
    import psv_native
    geom, sd, seq = deits
    engines = [_engine(geom, sd, 8) for _ in range(world)]
    emu = _engine(geom, sd, 8)
    keys = list(emu.backbone_grad_slices())
    n = emu.backbone_param_count
    pbufs = [torch.zeros(n + 4, device="cuda") for _ in range(world)]
    gbufs = [torch.empty(n + 4, device="cuda") for _ in range(world)]
    gptrs, pptrs = [g.data_ptr() for g in gbufs], [p.data_ptr() for p in pbufs]
    for t in range(3):
        steps = [0 if k.startswith("embeddings.") else t + 1 for k in keys]
        total = None
        for r in range(world):
            gbufs[r][:n].copy_(seq[(t + r) % len(seq)] * (r + 1))
            total = gbufs[r][:n].clone() if total is None else total + gbufs[r][:n]
        for r, e in enumerate(engines):
            e.backbone_peer_reduce_adam_step(gptrs, pbufs[r], r, steps, lr=LR, weight_decay=0.05,
                                             grad_scale=1.0 / world)
        for r, e in enumerate(engines):
            e.backbone_peer_gather_params(pptrs, r)
        emu.backbone_adam_step(total, steps, lr=LR, weight_decay=0.05, grad_scale=1.0 / world)
    want = emu.get_backbone_params()
    for e in engines:
        assert torch.equal(e.get_backbone_params(), want)
    lo = emu.backbone_grad_slices()["encoder.layer.0.layernorm_before.weight"][0]
    init = _engine(geom, sd, 8).get_backbone_params()
    assert torch.equal(want[:lo], init[:lo]) and not torch.equal(want[lo:], init[lo:])
    for r, e in enumerate(engines):                      # each rank's own shard of the moments is current
        a, b = psv_native.backbone_shard(n, world, r)
        for x, y in zip(e.get_backbone_adam_state(a, b), emu.get_backbone_adam_state(a, b)):
            assert torch.equal(x, y)
    for e in engines + [emu]:
        e.close()


@pytest.mark.gpu
def test_refusals(deits):
    import psv_native
    lib = psv_native.lib
    geom, sd, seq = deits
    e = _engine(geom, sd, 8)
    nt = len(e.backbone_grad_slices())
    n = e.backbone_param_count
    g = seq[0]
    steps = (C.c_int32 * nt)(*([1] * nt))
    s = psv_native._stream()
    args = (C.c_float(LR), C.c_float(0.9), C.c_float(0.999), C.c_float(1e-8), C.c_float(0.0), C.c_float(1.0), s)
    before = e.get_backbone_params().clone()
    assert lib.psv_backbone_adam_step(e._h, None, steps, *args) == -1
    mis = torch.zeros(n + 1, device="cuda")[1:]
    assert lib.psv_backbone_adam_step(e._h, C.c_void_p(mis.data_ptr()), steps, *args) == -1
    assert lib.psv_backbone_adam_step(e._h, C.c_void_p(g.data_ptr()), None, *args) == -1
    neg = (C.c_int32 * nt)(*([1] * (nt - 1) + [-1]))
    assert lib.psv_backbone_adam_step(e._h, C.c_void_p(g.data_ptr()), neg, *args) == -1
    bucket = torch.zeros(n + 4, device="cuda")
    peers = (C.c_void_p * 17)(*([g.data_ptr()] * 17))
    for world, rank in ((17, 0), (0, 0), (2, 2), (2, -1)):
        rc = lib.psv_backbone_peer_reduce_adam_step(e._h, peers, C.c_void_p(bucket.data_ptr()), world, rank, steps,
                                                    *args)
        assert rc == -1, (world, rank)
    assert lib.psv_backbone_peer_reduce_adam_step(e._h, peers, C.c_void_p(mis.data_ptr()), 1, 0, steps, *args) == -1
    misp = (C.c_void_p * 2)(g.data_ptr(), mis.data_ptr())
    assert lib.psv_backbone_peer_reduce_adam_step(e._h, misp, C.c_void_p(bucket.data_ptr()), 2, 0, steps, *args) == -1
    assert lib.psv_backbone_peer_gather_params(e._h, peers, 1, 0, s) == -3          # no peer step yet
    torch.cuda.synchronize()
    assert torch.equal(e.get_backbone_params(), before)                              # nothing was touched
    # world 1 is the local step; the gather must name the bucket that step published into
    assert lib.psv_backbone_peer_reduce_adam_step(e._h, peers, C.c_void_p(bucket.data_ptr()), 1, 0, steps, *args) == 0
    other = (C.c_void_p * 1)(g.data_ptr())
    assert lib.psv_backbone_peer_gather_params(e._h, other, 1, 0, s) == -1
    own = (C.c_void_p * 1)(bucket.data_ptr())
    assert lib.psv_backbone_peer_gather_params(e._h, own, 1, 0, s) == 0
    torch.cuda.synchronize()
    assert torch.equal(bucket[:n], e.get_backbone_params())
    m = torch.zeros(4, device="cuda")
    assert lib.psv_get_backbone_adam_state(e._h, n - 2, 4, C.c_void_p(m.data_ptr()), C.c_void_p(m.data_ptr()), s) == -1
    assert lib.psv_get_backbone_adam_state(e._h, -1, 1, C.c_void_p(m.data_ptr()), C.c_void_p(m.data_ptr()), s) == -1
    e.close()
    e16 = _engine(geom, sd, 8, "bf16")
    assert lib.psv_backbone_adam_step(e16._h, C.c_void_p(g.data_ptr()), steps, *args) == -4
    assert lib.psv_get_backbone_params(e16._h, C.c_void_p(bucket.data_ptr()), s) == -4
    with pytest.raises(psv_native.PsvError):
        e16.backbone_adam_step(g, [1] * nt)
    e16.close()


# BackboneTrainer against the drop-in's torch path (model(x), CE, backward, torch.optim.Adam), K steps on DeiT-S at
# batch 16.  The backward accumulates with float atomics, so the two runs differ in the last bits of every gradient and
# Adam, which normalises each gradient, carries that into the update; in the bf16 mode a weight that differs in its last
# fp32 bits can round to another bf16 value in the next forward.  Bars: loss history, max relative difference; final
# weights, Frobenius norm of the difference over that of the update (p_K - p_0), backbone and trained compressors
# together.  Worst values over two runs on a B200 (1000 W), loss / weights: split 8.9e-8 / 1.6e-4, bf16 7.4e-4 / 4.1e-2,
# joint 9.8e-6 / 2.5e-2.
TRAINER_BARS = {"split": (1e-4, 6e-4), "bf16": (3e-3, 0.15), "joint": (1e-4, 8e-2)}


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
def test_backbone_trainer_matches_drop_in(state_dicts, train_precision, joint):
    from main_model_utils import BackboneTrainer
    geom, sd = state_dicts("deits16")
    B, K, lr = 16, 3, 1e-4
    xs = [synth.make_pixels(B, geom, seed=500 + i, kind="randn").cuda() for i in range(K)]
    ys = [torch.randint(0, geom.classes, (B,), generator=torch.Generator().manual_seed(50 + i)).cuda() for i in range(K)]
    ref = _drop_in(geom, sd, train_precision, joint)
    opt = torch.optim.Adam([p for p in ref.parameters() if p.requires_grad], lr=lr, foreach=False)
    ref_hist = []
    for x, y in zip(xs, ys):
        logits = ref(x).logits
        loss = torch.nn.CrossEntropyLoss()(logits, y)
        if joint:
            loss = loss + sum((layer.loss for layer in ref.encoder.layer), 0.0)
        opt.zero_grad()
        loss.backward()
        opt.step()
        ref_hist.append(loss.item())
    model = _drop_in(geom, sd, train_precision, joint)
    eng = model._psv_engine_for(B, xs[0].device)
    tr = BackboneTrainer(eng, mlp_threshold=model.mlp_threshold, lr=lr, joint=joint)
    hist = [float(tr.step(x, y)) for x, y in zip(xs, ys)]
    rel = max(abs(a - b) / abs(b) for a, b in zip(hist, ref_hist))
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
    print(f"{train_precision}{' joint' if joint else ''}: loss rel {rel:.2e} (bar {loss_bar}), "
          f"|dp| / |update| {upd:.2e} (bar {update_bar})")
    assert rel <= loss_bar and upd <= update_bar
    # export_to: the module takes the trained values and its next drop-in forward runs without a reload
    loads = []
    orig = eng.load_state_dict
    eng.load_state_dict = lambda sdict: (loads.append(1), orig(sdict))
    tr.export_to(model)
    model.eval()
    with torch.no_grad():
        got = model(xs[0]).logits
    assert not loads
    assert model._psv_engine is eng
    r = eng.forward(xs[0], model.mlp_threshold, want_n_active=True, use_graph=True)
    assert torch.equal(got, r["logits"])
    for k, v in out.items():
        assert torch.equal(dict(model.named_parameters())[k].detach().reshape(v.shape), v)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs with peer access")
def test_sharded_peer_step_two_gpus():
    """tools/backbone_p2p_check.py at world 2: bit-identical replicas (p2p-fused and nccl), p2p-fused bit-equal to a
    single-process emulation (rank-order fp32 sum + backbone_adam_step), p2p-fused against nccl within a bar, and a
    world-2 checkpoint loaded into a world-1 trainer with equal moments."""
    from conftest import ROOT
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tools", "backbone_p2p_check.py"), "--steps", "3",
           "--batch", "16", "--geom", "deits16"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:], r.stderr[-1500:])
    res = json.loads(lines[-1])
    assert res["ok"], res
