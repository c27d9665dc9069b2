"""Mixed-precision backbone fine-tuning (psv_set_train_precision(PSV_TRAIN_BF16) on fp32 handles) against float64
references that round to bf16 where the kernels round (oracle/bf16_train_reference.py, straight-through roundings).

Stages and bars, as in test_gpu_bf16_fp64.py: each test prints the worst error per stage and geometry, and the bars
sit about 3-4x above the worst errors a B200 measured (values beside each bar).  A CPU test plants defects in the
references on the GPU cases' inputs; each defect must move its stage's metric by at least 2x the bar.

What separates the kernels from the rounding-aware reference is the rounding the reference does not model: P rounded
against a running maximum, the fp32 accumulation order, and the bf16 rounding of the upstream gradients that the
backward's GEMMs and the attention backward take as operands (dY, dO, P, dS) -- the reference's gradients are exact.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synth
import test_gpu_bf16_fp64 as B16
import test_gpu_finetune_fp64 as FT
from oracle import bf16_reference as R
from oracle import bf16_train_reference as TR

GEOMS = {"deits16": synth.DEIT_S16, "vitb16": synth.VIT_B16, "vitl16": synth.VIT_L16}
MT = 0.5

# ---- bars, about 3-4x above the worst errors measured on a B200 at 1000 W (in brackets)
# The three attention bars held on a B200 for the single / lengths / mixed cases with each part's own norm as the
# denominator; with the case's whole dqkv as the denominator, and for the dominant / ties / big_v cases, the worst
# errors are printed by test_gpu_attention_hooks_against_rounded_fp64 but not yet recorded here.
LSE_TOL = 1e-4               # |lse - ref|, natural log
ATTN_GRAD_FROB = 1.5e-2      # dQ, dK, dV of one case: ||g - r|| / ||r of the case's whole dqkv||
ATTN_GRAD_MAX = 4e-2         # max |g - r| / max |r of the case's whole dqkv|
STEP_FROB = 5e-2             # whole step, per gradient tensor, vs the rounding-aware reference: ||g - r|| / ||r||
                             # [1.47e-2, uint8 input; 1.11e-2 otherwise]
STEP_MAX = 8e-2              # max |g - r| / max |r|  [2.03e-2, uint8 input; 1.31e-2 otherwise]
KEY_BIAS = 5e-2              # ||d key.bias|| / ||d query.bias||: exactly zero in exact arithmetic  [1.3e-2]
COMP_FROB = 5e-2             # compressor tensors of the joint objective  [1.33e-2]
COMP_MAX = 5e-2              # [1.10e-2]
TRUE_FROB = 5e-2             # against the UNROUNDED fp64 reference: how far mixed precision is from exact  [1.25e-2]
TRUE_MAX = 6e-2              # [1.57e-2]
TRUE_COMP = 1e-1             # compressor tensors, both metrics  [2.66e-2]
MODES_FROB = 5e-2            # bf16 mode vs split mode at batch 256, every token kept  [1.34e-2]
DECISION_BAND = 1.2e-3       # every mask disagreement has |score - mt| below this  [3.0e-4]

ATTN_CASES = ["single", "lengths_x1", "lengths_x4", "mixed", "dominant", "ties", "big_v"]


# ------------------------------------------------------------------------------------------------ references
def attention_case(D, name):
    if name == "single":
        g = torch.Generator().manual_seed(D + 7)
        return torch.randn(197, 3 * D, generator=g, dtype=torch.float64).to(torch.bfloat16), [197]
    return B16.attention_case(D, name)


def attention_reference(qkv, lens, D, dctx, scale=R.SCALE, drop_last_block=False):
    """fp64 autograd of the straight-through rounded attention on the same bf16 inputs:
    (ctx [T, D], lse [T, H], dqkv [T, 3D]); dctx [T, D] is the upstream gradient"""
    H = D // 64
    x = qkv.double().detach().requires_grad_(True)
    ctxs, lses = [], []
    r0 = 0
    for n in lens:
        q, k, v = (x[r0:r0 + n, j * D:(j + 1) * D].reshape(n, H, 64).transpose(0, 1) for j in range(3))
        km = None
        if drop_last_block and n > 32:
            km = torch.ones(1, n, dtype=torch.bool, device=x.device)
            km[:, (n - 1) // 32 * 32:] = False
        ctxs.append(TR.attend(q, k, v, True, km, scale).transpose(0, 1).reshape(n, D))
        s = torch.matmul(q, k.transpose(-1, -2)) * scale
        lses.append(torch.logsumexp(s, -1).transpose(0, 1))
        r0 += n
    ctx = torch.cat(ctxs)
    (dqkv,) = torch.autograd.grad(ctx, [x], dctx.double())
    return ctx.detach(), torch.cat(lses).detach(), dqkv


def attention_manual_grads(qkv, lens, D, dctx, with_di=True):
    """FlashAttention-2's backward written out in fp64 without rounding; with_di=False plants a missing Di term"""
    H = D // 64
    x = qkv.double()
    out = torch.zeros_like(x)
    r0 = 0
    for n in lens:
        q, k, v = (x[r0:r0 + n, j * D:(j + 1) * D].reshape(n, H, 64).transpose(0, 1) for j in range(3))
        do = dctx[r0:r0 + n].double().reshape(n, H, 64).transpose(0, 1)
        p = torch.softmax(torch.matmul(q, k.transpose(-1, -2)) * R.SCALE, -1)
        o = torch.matmul(p, v)
        di = (do * o).sum(-1, keepdim=True) if with_di else 0.0
        ds = p * (torch.matmul(do, v.transpose(-1, -2)) - di)
        for j, t in enumerate((torch.matmul(ds, k) * R.SCALE, torch.matmul(ds.transpose(-1, -2), q) * R.SCALE,
                               torch.matmul(p.transpose(-1, -2), do))):
            out[r0:r0 + n, j * D:(j + 1) * D] = t.transpose(0, 1).reshape(n, D)
        r0 += n
    return out


def _dctx(T, D, seed):
    return torch.randn(T, D, generator=torch.Generator().manual_seed(seed), dtype=torch.float32)


def grad_errors(got, ref, D):
    """per part (dQ, dK, dV): (Frobenius norm, max-abs) of the error over those of the case's whole reference dqkv.
    (Where one key dominates, dQ itself nearly vanishes: dP and Di cancel.  Against its own norm the bf16 rounding of
    O alone is then a large relative error.)"""
    out = {}
    rn, rmax = float(ref.double().norm()), float(ref.double().abs().max())
    for j, name in enumerate(("dq", "dk", "dv")):
        d = got[:, j * D:(j + 1) * D].double() - ref[:, j * D:(j + 1) * D].double()
        out[name] = (float(d.norm()) / rn, float(d.abs().max()) / rmax)
    return out


# ------------------------------------------------------------------------------------------------ CPU
def test_reference_without_rounding_is_the_fp32_finetune_reference(state_dicts):
    """rounding=False: logits and every gradient equal reference_forward's (fp64) to ~1e-12"""
    geom, sd = state_dicts("deits16")
    x = synth.make_pixels(2, geom, seed=3).double()
    p1, p2 = FT.reference_params(sd, "cpu"), FT.reference_params(sd, "cpu")
    a = FT.reference_forward(p1, x, MT, geom.heads, joint=True)
    b = TR.forward(p2, x, MT, geom.heads, joint=True, rounding=False)
    assert torch.equal(a[1], b[1])
    up = torch.randn(a[0].shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    ga = FT.reference_grads(p1, [a[0], a[3]], [up, torch.ones_like(a[3])], True)
    gb = FT.reference_grads(p2, [b[0], b[3]], [up, torch.ones_like(b[3])], True)
    worst = max(float((ga[k] - gb[k]).norm()) / max(float(ga[k].norm()), 1e-300) for k in ga
                if not k.endswith("key.bias"))
    print(f"\nunrounded train reference vs fp64 fine-tune reference: worst relative gradient difference {worst:.1e}")
    assert worst < 1e-10
    assert float((a[0] - b[0]).abs().max()) < 1e-12


def test_reference_forward_is_the_bf16_inference_reference(state_dicts):
    """rounding on, teacher-forced: the training reference's logits are bf16_reference.forward's"""
    geom, sd = state_dicts("deits16")
    x = synth.make_pixels(2, geom, seed=4).double()
    masks = FT.reference_forward(FT.reference_params(sd, "cpu"), x, MT, geom.heads)[1]
    with torch.no_grad():
        ref, _ = R.forward(sd, x, forced_masks=masks)
        got = TR.forward(FT.reference_params(sd, "cpu"), x, MT, geom.heads, forced_masks=masks)[0]
    err = float((got - ref).abs().max())
    print(f"\ntraining reference vs bf16_reference logits: {err:.1e}")
    assert err < 1e-9


def test_rounding_is_straight_through():
    t = torch.tensor([1.0 + 2 ** -10, -3.3], dtype=torch.float64, requires_grad=True)
    y = TR.rnd(t)
    assert torch.equal(y.detach(), t.detach().to(torch.bfloat16).double())
    (g,) = torch.autograd.grad((y * torch.tensor([0.1 + 2 ** -20, 7.0], dtype=torch.float64)).sum(), [t])
    assert g[0] == 0.1 + 2 ** -20 and g[1] == 7.0         # not rounded to bf16


@pytest.mark.parametrize("D", [384, 768, 1024])
def test_attention_bars_catch_planted_defects(D):
    """On the GPU cases' inputs each planted defect moves its stage by at least 2x the bar."""
    qkv, lens = attention_case(D, "lengths_x1")
    dctx = _dctx(qkv.shape[0], D, D)
    _, lse, _ = attention_reference(qkv, lens, D, dctx)
    _, lse_s, _ = attention_reference(qkv, lens, D, dctx, scale=1 / 7.9)
    scale_move = float((lse_s - lse).abs().max())
    clean = attention_manual_grads(qkv, lens, D, dctx)
    no_di = grad_errors(attention_manual_grads(qkv, lens, D, dctx, with_di=False), clean, D)
    _, _, ref = attention_reference(qkv, lens, D, dctx)
    _, _, dropped = attention_reference(qkv, lens, D, dctx, drop_last_block=True)
    drop = grad_errors(dropped, ref, D)
    swapped = ref.clone()
    swapped[:, D:2 * D], swapped[:, 2 * D:] = ref[:, 2 * D:], ref[:, D:2 * D]
    swap = grad_errors(swapped, ref, D)
    moves = {"scale 1/7.9 (lse)": scale_move / LSE_TOL,
             "missing Di (dQ)": no_di["dq"][0] / ATTN_GRAD_FROB,
             "dropped last key block (dV)": drop["dv"][0] / ATTN_GRAD_FROB,
             "dK / dV swapped (dK)": swap["dk"][0] / ATTN_GRAD_FROB}
    print(f"\nD={D} defect / bar: " + ", ".join(f"{k} {v:.1f}x" for k, v in moves.items()))
    for k, v in moves.items():
        assert v >= 2.0, (k, v)


# ------------------------------------------------------------------------------------------------ GPU helpers
def _engine(geom, sd, max_batch, mode="bf16"):
    import psv_native
    e = psv_native.Engine(geom, "fp32", max_batch)
    e.load_state_dict(sd)
    e.set_train_precision(mode)
    return e


@pytest.fixture(scope="module")
def sds():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = synth.make_state_dict(GEOMS[name], seed=42)
        return GEOMS[name], cache[name]
    return get


def _compare(got, ref, frob, mx, comp_frob, comp_mx, label):
    """per-tensor relative Frobenius and max-abs / max|ref|; returns the worst (rel-Frobenius, max-abs) and the failures"""
    worst = {"frob": (0.0, ""), "max": (0.0, ""), "cfrob": (0.0, ""), "cmax": (0.0, "")}
    fails = []
    for k, r in ref.items():
        g = got[k].detach().double().reshape(r.shape)
        r = r.double()
        if k.endswith("attention.attention.key.bias"):      # exactly zero in exact arithmetic
            qb = float(ref[k.replace("key.bias", "query.bias")].norm())
            if float(g.norm()) > KEY_BIAS * qb + 1e-12:
                fails.append((k, "abs", float(g.norm()), qb))
            continue
        rn, rmax = float(r.norm()), float(r.abs().max())
        if rn == 0.0:
            continue
        d = g - r
        rf, ma = float(d.norm()) / rn, float(d.abs().max()) / rmax
        c = "mlp_layer" in k
        kf, km = ("cfrob", "cmax") if c else ("frob", "max")
        if rf > worst[kf][0]:
            worst[kf] = (rf, k)
        if ma > worst[km][0]:
            worst[km] = (ma, k)
        if rf > (comp_frob if c else frob) or ma > (comp_mx if c else mx):
            fails.append((k, rf, ma))
    print(f"[{label}] worst rel-Frobenius {worst['frob'][0]:.2e} ({worst['frob'][1]}), max-abs {worst['max'][0]:.2e} "
          f"({worst['max'][1]})" + (f"; compressors {worst['cfrob'][0]:.2e} / {worst['cmax'][0]:.2e}"
                                    if worst["cmax"][1] else ""))
    return fails


def _step(e, geom, sd, B, mt, upstream, joint=False, pixels=None, seed=1234, label=""):
    x = synth.make_pixels(B, geom, seed=seed, kind="randn").cuda() if pixels is None else pixels
    gen = torch.Generator().manual_seed(seed)
    out = e.backbone_forward_train(x, mt, with_layer_losses=joint)
    logits = out[0] if joint else out
    masks = e.backbone_train_masks()
    if upstream == "ce":
        labels = torch.randint(0, geom.classes, (B,), generator=gen).cuda()
        lg = logits.detach().clone().requires_grad_(True)
        F.cross_entropy(lg, labels).backward()
        dlogits = lg.grad
    else:
        dlogits = torch.randn(B, geom.classes, generator=gen).cuda()
    dlosses = torch.rand(geom.layers, generator=gen).cuda() * 2 + 0.25 if joint else None
    res = e.backbone_backward(dlogits, dlosses)
    torch.cuda.synchronize()
    flat, cflat = res if joint else (res, None)
    got = FT._flat_to_dict(flat, e.backbone_grad_slices())
    if joint:
        got.update(FT._comp_to_dict(cflat, geom))
    return x, logits, masks, dlogits, dlosses, got


def _reference_grads(sd, geom, x, mt, masks, dlogits, dlosses, rounding):
    p = FT.reference_params(sd, "cuda")
    rl, _, rs, rlosses = TR.forward(p, x.double(), mt, geom.heads, forced_masks=masks, joint=dlosses is not None,
                                    rounding=rounding)
    outs, ups = [rl], [dlogits.double()]
    if dlosses is not None:
        outs.append(rlosses)
        ups.append(dlosses.double())
    return rl.detach(), rs, FT.reference_grads(p, outs, ups, dlosses is not None)


# ------------------------------------------------------------------------------------------------ GPU: attention hooks
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GEOMS))
def test_gpu_attention_hooks_against_rounded_fp64(name, sds):
    geom, sd = sds(name)
    D = geom.hidden
    e = _engine(geom, sd, 48)
    try:
        worst = {"ctx_rms": 0.0, "ctx_bar": 0.0, "lse": 0.0, "frob": 0.0, "max": 0.0}
        fails = []
        for case in ATTN_CASES:
            qkv, lens = attention_case(D, case)
            q = qkv.cuda()
            cu = B16._cu(lens, "cuda")
            dctx = _dctx(q.shape[0], D, 11 + D)
            ctx, lse = e.attention_train_forward(q, cu)
            dqkv = e.attention_backward(q, cu, ctx, lse, dctx.cuda())
            dqkv2 = e.attention_backward(q, cu, ctx, lse, dctx.cuda())
            torch.cuda.synchronize()
            assert torch.equal(dqkv, dqkv2), "two runs differ"
            rctx, rlse, rd = attention_reference(q, lens, D, dctx.cuda())
            dist = (ctx.double() - rctx).abs()
            bar = B16.attention_bar(rctx, q, lens, D)
            worst["ctx_bar"] = max(worst["ctx_bar"], float((dist / bar).max()))
            worst["ctx_rms"] = max(worst["ctx_rms"], float(B16.attention_rms(dist, q, lens, D)))
            worst["lse"] = max(worst["lse"], float((lse.double() - rlse).abs().max()))
            errs = grad_errors(dqkv, rd, D)
            lse_err = float((lse.double() - rlse).abs().max())
            print(f"\n[{name} {case}] lse {lse_err:.2e}, ctx max dist/bar {float((dist / bar).max()):.2f}; "
                  + ", ".join(f"{k} {rf:.2e} / {ma:.2e}" for k, (rf, ma) in errs.items()))
            for part, (rf, ma) in errs.items():
                worst["frob"] = max(worst["frob"], rf)
                worst["max"] = max(worst["max"], ma)
                if rf >= ATTN_GRAD_FROB or ma >= ATTN_GRAD_MAX:
                    fails.append((case, part, rf, ma))
            if not bool((dist <= bar).all()) or float(B16.attention_rms(dist, q, lens, D)) >= B16.ATTN_RMS:
                fails.append((case, "ctx"))
            if lse_err >= LSE_TOL:
                fails.append((case, "lse", lse_err))
        print(f"\n[{name}] attention hooks: ctx max dist/bar {worst['ctx_bar']:.2f}, ctx rms/max|v| {worst['ctx_rms']:.2e}, "
              f"lse {worst['lse']:.2e}, grads rel-Frobenius {worst['frob']:.2e}, max-abs {worst['max']:.2e}")
        assert not fails, fails
    finally:
        e.close()


@pytest.mark.gpu
def test_gpu_attention_backward_does_not_depend_on_the_batch(sds):
    """An image's dqkv is bit-identical alone and inside a mixed batch."""
    geom, sd = sds("vitb16")
    D = geom.hidden
    e = _engine(geom, sd, 48)
    try:
        qkv, lens = attention_case(D, "mixed")
        q = qkv.cuda()
        dctx = _dctx(q.shape[0], D, 5).cuda()
        cu = B16._cu(lens, "cuda")
        ctx, lse = e.attention_train_forward(q, cu)
        full = e.attention_backward(q, cu, ctx, lse, dctx)
        r0 = 0
        for b, n in enumerate(lens[:12]):
            one = B16._cu([n], "cuda")
            c1, l1 = e.attention_train_forward(q[r0:r0 + n].contiguous(), one)
            d1 = e.attention_backward(q[r0:r0 + n].contiguous(), one, c1, l1, dctx[r0:r0 + n].contiguous())
            assert torch.equal(c1, ctx[r0:r0 + n]) and torch.equal(l1, lse[r0:r0 + n]), b
            assert torch.equal(d1, full[r0:r0 + n]), b
            r0 += n
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: whole steps
STEP_CASES = [("deits16", 16, "ce", False), ("deits16", 16, "randn", False), ("deits16", 16, "ce", True),
              ("vitb16", 16, "ce", False), ("vitb16", 16, "randn", False), ("vitb16", 16, "ce", True),
              ("vitl16", 8, "ce", False)]


@pytest.mark.gpu
@pytest.mark.parametrize("name, B, upstream, joint", STEP_CASES)
def test_gpu_step_against_rounded_fp64(name, B, upstream, joint, sds):
    geom, sd = sds(name)
    e = _engine(geom, sd, B)
    try:
        label = f"{name} B={B} {upstream}{' joint' if joint else ''}"
        x, logits, masks, dl, dls, got = _step(e, geom, sd, B, MT, upstream, joint, label=label)
        rl, rs, ref = _reference_grads(sd, geom, x, MT, masks, dl, dls, True)
        lerr = (logits.double() - rl).abs()
        print(f"\n[{label}] logits max-abs {float(lerr.max()):.2e}, rms {float(lerr.pow(2).mean().sqrt()):.2e}")
        assert float(lerr.max()) < B16.LOGITS_TOL and float(lerr.pow(2).mean().sqrt()) < B16.LOGITS_RMS
        fails = _compare(got, ref, STEP_FROB, STEP_MAX, COMP_FROB, COMP_MAX, label + " vs rounded")
        assert not fails, fails[:8]
        # decisions: every disagreement with the fp64 compressor on the reference's teacher-forced stream lies in a band
        want = rs >= MT
        dis = (masks[:, :, 1:].bool() != want)
        band = float((rs - MT).abs()[dis].max()) if bool(dis.any()) else 0.0
        print(f"[{label}] decisions: {int(dis.sum())} of {dis.numel()} differ, all within |score - mt| <= {band:.2e}")
        assert band < DECISION_BAND
        del ref
        _, _, true = _reference_grads(sd, geom, x, MT, masks, dl, dls, False)
        fails = _compare(got, true, TRUE_FROB, TRUE_MAX, TRUE_COMP, TRUE_COMP, label + " vs unrounded")
        assert not fails, fails[:8]
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uint8", "similarity"])
def test_gpu_step_uint8_and_similarity(kind, sds):
    geom, sd = sds("deits16")
    B = 8
    e = _engine(geom, sd, B)
    try:
        if kind == "uint8":
            img = torch.randint(0, 256, (B, 224, 224, 3), generator=torch.Generator().manual_seed(3), dtype=torch.uint8)
            e.set_u8_input(224, 224)
            x = img.cuda()
            # 224 x 224 sources: the resize is the identity; x / 255, then (x - 0.5) / 0.5 in fp32 as the kernel does
            pix = ((img.permute(0, 3, 1, 2).float() * (1.0 / 255.0) - 0.5) / 0.5).contiguous()
        else:
            e.set_skip_criterion("similarity", 0.9)
            x = synth.make_pixels(B, geom, seed=77, kind="randn").cuda()
            pix = x
        _, logits, masks, dl, _, got = _step(e, geom, sd, B, MT, "ce", pixels=x, label=kind)
        rl, _, ref = _reference_grads(sd, geom, pix.cuda(), MT, masks, dl, None, True)
        print(f"\n[{kind}] logits max-abs {float((logits.double() - rl).abs().max()):.2e}")
        assert float((logits.double() - rl).abs().max()) < B16.LOGITS_TOL
        fails = _compare(got, ref, STEP_FROB, STEP_MAX, COMP_FROB, COMP_MAX, kind)
        assert not fails, fails[:8]
    finally:
        e.close()


@pytest.mark.gpu
def test_gpu_bf16_mode_against_split_mode_at_batch_256(sds):
    """mt 0.0 keeps every token, so both modes have the same masks by construction."""
    geom, sd = sds("vitb16")
    B = 256
    e = _engine(geom, sd, B, "split")
    try:
        x = synth.make_pixels(B, geom, seed=9, kind="randn").cuda()
        dl = torch.randn(B, geom.classes, generator=torch.Generator().manual_seed(2)).cuda()
        e.backbone_forward_train(x, 0.0)
        split = FT._flat_to_dict(e.backbone_backward(dl).clone(), e.backbone_grad_slices())
        e.set_train_precision("bf16")
        e.backbone_forward_train(x, 0.0)
        assert bool(e.backbone_train_masks().bool().all())
        mixed = FT._flat_to_dict(e.backbone_backward(dl), e.backbone_grad_slices())
        torch.cuda.synchronize()
        fails = _compare(mixed, split, MODES_FROB, 1e9, 1e9, 1e9, "vitb16 B=256 bf16 vs split")
        assert not fails, fails[:8]
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ GPU: plumbing
@pytest.mark.gpu
def test_gpu_mode_is_recorded_with_the_forward(sds):
    """Switching the mode between forward and backward changes nothing.  (The bias and LayerNorm gradients sum with
    float atomics, so two runs agree to rounding, not bit for bit.)"""
    def rel(u, v):
        return float((u - v).norm() / v.norm())
    geom, sd = sds("deits16")
    e = _engine(geom, sd, 4)
    try:
        x = synth.make_pixels(4, geom, seed=5, kind="randn").cuda()
        dl = torch.randn(4, geom.classes, generator=torch.Generator().manual_seed(1)).cuda()
        for first, other in (("bf16", "split"), ("split", "bf16")):
            e.set_train_precision(first)
            e.backbone_forward_train(x, MT)
            a = e.backbone_backward(dl).clone()
            e.backbone_forward_train(x, MT)
            e.set_train_precision(other)
            b = e.backbone_backward(dl)
            torch.cuda.synchronize()
            assert rel(b, a) < 1e-5, (first, rel(b, a))
            if first == "bf16":
                mixed = a
        print(f"\nbf16 vs split gradient, relative norm of the difference: {rel(mixed, a):.2e}")
        assert rel(mixed, a) > 1e-3                          # the modes do differ
    finally:
        e.close()


@pytest.mark.gpu
def test_gpu_refusals(sds):
    import psv_native
    from psv_native import _ptr, _stream, lib
    geom, sd = sds("deits16")
    e = _engine(geom, sd, 2)
    b = psv_native.Engine(geom, "bf16", 2)
    try:
        assert lib.psv_set_train_precision(b._h, 1) == -4                  # PSV_ERR_UNSUPPORTED on a bf16 handle
        assert lib.psv_set_train_precision(e._h, 7) == -1                  # PSV_ERR_INVALID
        x = synth.make_pixels(2, geom, seed=5, kind="randn").cuda()
        logits = torch.empty(2, geom.classes, device="cuda")
        e.set_kv_mode("all")
        rc = lib.psv_backbone_forward_train(e._h, _ptr(x), 0, 2, MT, _ptr(logits), None, _stream(e.device))
        assert rc == -4, rc
        e.set_kv_mode("active")
        e.set_train_precision("split")
        q = torch.zeros(4, 3 * geom.hidden, device="cuda", dtype=torch.bfloat16)
        with pytest.raises(psv_native.PsvError):                          # hooks need PSV_TRAIN_BF16
            e.attention_train_forward(q, B16._cu([4], "cuda"))
    finally:
        e.close()
        b.close()


def _model(geom, sd, precision):
    import model_utils
    from transformers.models.vit.modeling_vit import ViTConfig
    cfg = ViTConfig(hidden_size=geom.hidden, num_attention_heads=geom.heads, intermediate_size=geom.ffn,
                    num_hidden_layers=geom.layers)
    cfg.num_labels = geom.classes
    model = model_utils.ModifiedViTModel(cfg, 0.9, MT, 0)
    model.load_state_dict(sd, strict=False)
    model = model.to("cuda")
    model.psv_precision = "fp32"
    model.psv_train_precision = precision
    return model


@pytest.mark.gpu
def test_gpu_drop_in_grads_are_the_engine_slices(sds):
    geom, sd = sds("deits16")
    model = _model(geom, sd, "bf16")
    model.train()
    model.vit_train()
    x = synth.make_pixels(4, geom, seed=21, kind="randn").cuda()
    labels = torch.tensor([1, 2, 3, 4], device="cuda")
    torch.nn.CrossEntropyLoss()(model(x).logits, labels).backward()
    e = _engine(geom, sd, 4)
    try:
        logits = e.backbone_forward_train(x, MT)
        lg = logits.detach().clone().requires_grad_(True)
        torch.nn.CrossEntropyLoss()(lg, labels).backward()
        flat = FT._flat_to_dict(e.backbone_backward(lg.grad), e.backbone_grad_slices())
        torch.cuda.synchronize()
        params = dict(model.named_parameters())
        scale = max(float(g.abs().max()) for g in flat.values())
        for k, g in flat.items():                            # to the float-atomic rounding of two runs
            assert torch.allclose(params[k].grad.reshape(g.shape), g, rtol=1e-4, atol=1e-6 * scale), k
    finally:
        e.close()


@pytest.mark.gpu
def test_gpu_drop_in_trains_in_bf16(sds):
    from main_model_utils import synthetic_loader, train
    geom, sd = sds("deits16")
    model = _model(geom, sd, "bf16")
    loader = synthetic_loader(8, 8, geom=geom, seed=5, kind="randn", pin_memory=False)
    hist = train(model, loader, None, "cuda", num_epochs=20, loss_type="classification", lr=1e-4)
    print(f"\nbf16 drop-in, 20 Adam steps on one batch of 8: loss {hist[0]:.4f} -> {hist[-1]:.4f}")
    assert all(np.isfinite(h) for h in hist)
    assert hist[-1] < hist[0]
