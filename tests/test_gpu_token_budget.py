"""GPU (B200): the per-layer token budget (psv_set_token_budget) on every path that follows it.

The rule itself is pinned on the CPU in test_token_budget.py; here the library's masks must be exactly that rule
applied to the scores it returns, the budgeted forward must match the fp32 oracle deciding by the same rule, the
documented bit-identities must hold, and fine-tuning under a budget must match the fp64 references with those masks.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import synth
import test_gpu_finetune_bf16 as BF
import test_gpu_finetune_fp64 as FT
from oracle import token_budget as TB
from oracle import vit_skip_oracle as O
from test_gpu_finetune_kv_all import reference_forward_kv_all

pytestmark = pytest.mark.gpu

GEOMS = {"deits16": synth.DEIT_S16, "vitb16": synth.VIT_B16}
MT = 0.5
P = 196
PER_LAYER = [0, 196, 24, 49, 98, 147, 5, 190, 1, 195, 64, 0]
BUDGETS = [("exact", 49), ("cap", 64), ("exact", PER_LAYER), ("cap", PER_LAYER)]
ERR_INVALID, ERR_UNSUPPORTED = -1, -4


@pytest.fixture(scope="module")
def sds():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = synth.make_state_dict(GEOMS[name], seed=42)
        return GEOMS[name], cache[name]
    return get


def _engine(sds, name, precision="fp32", max_batch=8, kv="active"):
    import psv_native
    geom, sd = sds(name)
    e = psv_native.Engine(geom, precision, max_batch)
    e.load_state_dict(sd)
    if kv != "active":
        e.set_kv_mode(kv)
    return e


def _keep(k, L=12):
    return [k] * L if isinstance(k, int) else list(k)


def _check_rule(r, keep, mode, label):
    """masks_out == rule(scores_out) bit for bit, n_active == mask sums (== k + 1 under exact)."""
    masks = r["masks"].cpu().numpy().astype(bool)
    want = TB.budget_masks(r["scores"].cpu().numpy(), keep, mode, MT)
    assert np.array_equal(masks, want), f"{label}: {int((masks != want).sum())} decisions differ from the rule"
    n = r["n_active"].cpu().numpy()
    assert np.array_equal(n, masks.sum(-1)), label
    if mode == "exact":
        assert np.array_equal(n, np.broadcast_to(np.array(keep)[:, None] + 1, n.shape)), label


# ------------------------------------------------------------------------------------------------ 1. the rule on the GPU
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kv", ["active", "all"])
def test_masks_are_the_rule_of_the_returned_scores(sds, precision, kv):
    e = _engine(sds, "deits16", precision, 256, kv)
    try:
        geom, _ = sds("deits16")
        for B in (1, 7, 256):
            x = synth.make_pixels(B, geom, seed=100 + B).cuda()
            for mode, k in BUDGETS:
                keep = _keep(k)
                e.set_token_budget(keep, mode)
                for use_graph in (False, True, True):
                    r = e.forward(x, MT, want_masks=True, want_scores=True, want_n_active=True, use_graph=use_graph)
                    torch.cuda.synchronize()
                    _check_rule(r, keep, mode, f"{precision} kv={kv} B={B} {mode} {k} graph={use_graph}")
                # the per-layer entry point decides the same way
                h = e.embed(x)
                for l in range(geom.layers):
                    m, s, n = e.layer_forward(l, h, MT)
                    torch.cuda.synchronize()
                    want = TB.budget_mask(s.cpu().numpy(), keep[l], mode, MT)
                    assert np.array_equal(m.cpu().numpy().astype(bool), want), (precision, kv, B, mode, l)
                    assert np.array_equal(n.cpu().numpy(), want.sum(-1)), (precision, kv, B, mode, l)
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 2. fp32 against the oracle
def _first_flips(gpu_masks, ref_masks):
    """per image, the first layer whose mask differs (or -1): later layers of that image see another stream"""
    diff = (np.asarray(gpu_masks) != np.asarray(ref_masks)).any(-1)          # [L, B]
    return np.where(diff.any(0), diff.argmax(0), -1)


@pytest.mark.parametrize("name, B", [("deits16", 6), ("vitb16", 3)])
@pytest.mark.parametrize("mode, k", BUDGETS)
def test_fp32_forward_matches_the_oracle_with_its_own_budget(sds, name, B, mode, k):
    geom, sd = sds(name)
    keep = _keep(k)
    e = _engine(sds, name, "fp32", B)
    try:
        e.set_token_budget(keep, mode)
        x = synth.make_pixels(B, geom, seed=7 + B)
        r = e.forward(x.cuda(), MT, want_masks=True, want_scores=True, want_n_active=True)
        torch.cuda.synchronize()
        with torch.no_grad():
            logits, rmasks, rscores = TB.forward(sd, x, keep, mode, MT)
        gm = r["masks"].cpu().numpy().astype(bool)
        first = _first_flips(gm, rmasks.numpy())
        near = np.stack([TB.near_cut(rscores[l].numpy(), keep[l], mode, MT) for l in range(geom.layers)])   # [L, B]
        for b in np.flatnonzero(first >= 0):
            assert near[first[b], b], f"image {b} decided differently at layer {first[b]} outside the 1e-4 band"
        clean = first < 0
        print(f"\n[{name} {mode} {k}] {int((~clean).sum())} of {B} images flipped inside the band "
              f"({int(near.any(0).sum())} have a near cut)")
        assert clean.sum() >= (B + 1) // 2
        assert float((r["logits"].cpu()[clean] - logits[clean]).abs().max()) < 1e-4
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 3. bf16 teacher-forced
@pytest.mark.parametrize("mode, k", [("exact", 49), ("cap", PER_LAYER)])
def test_bf16_layers_teacher_forced_against_the_oracle(sds, mode, k):
    geom, sd = sds("vitb16")
    keep = _keep(k)
    B = 4
    e = _engine(sds, "vitb16", "bf16", B)
    try:
        e.set_token_budget(keep, mode)
        x = synth.make_pixels(B, geom, seed=21)
        flips = 0
        with torch.no_grad():
            h = O.embed(sd, x)
            for l in range(geom.layers):
                s = O.compressor_scores(sd, l, h)
                want = TB.budget_mask(s.numpy(), keep[l], mode, MT)
                m, sg, _ = e.layer_forward(l, h.cuda().contiguous(), MT)
                torch.cuda.synchronize()
                got = m.cpu().numpy().astype(bool)
                assert np.array_equal(got, TB.budget_mask(sg.cpu().numpy(), keep[l], mode, MT))
                near = TB.near_cut(s.numpy(), keep[l], mode, MT)
                bad = (got != want).any(-1)
                assert not (bad & ~near).any(), f"layer {l}: masks differ outside the band"
                flips += int(bad.sum())
                h, _, _ = O.layer_forward(sd, l, h, MT, forced_mask=torch.from_numpy(want))
        print(f"\n[bf16 {mode} {k}] {flips} image-layers decided differently inside the band")
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 4. bit-identical anchors
def _fwd(e, x, mt, use_graph=False):
    r = e.forward(x, mt, want_masks=True, want_scores=True, want_n_active=True, use_graph=use_graph)
    torch.cuda.synchronize()
    return {k: r[k].clone() for k in ("logits", "masks", "scores", "n_active")}


def _same(a, b, label):
    for key in ("logits", "masks", "scores", "n_active"):
        assert torch.equal(a[key], b[key]), f"{label}: {key} differs"


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_anchors(sds, precision):
    geom, _ = sds("deits16")
    B = 16
    x = synth.make_pixels(B, geom, seed=3).cuda()
    fresh = _engine(sds, "deits16", precision, B)
    e = _engine(sds, "deits16", precision, B)
    try:
        for use_graph in (False, True):
            base = _fwd(fresh, x, MT, use_graph)
            dense = _fwd(fresh, x, 0.0, use_graph)
            e.set_token_budget(P, "cap")
            _same(_fwd(e, x, MT, use_graph), base, f"cap N-1 vs no budget, graph={use_graph}")
            e.set_token_budget(P, "exact")
            _same(_fwd(e, x, 0.7, use_graph), dense, f"exact N-1 vs mt=0, graph={use_graph}")
            e.set_token_budget(49, "exact")
            _fwd(e, x, MT, use_graph)
            e.set_token_budget(None)
            _same(_fwd(e, x, MT, use_graph), base, f"budget then off vs fresh, graph={use_graph}")
    finally:
        e.close()
        fresh.close()


@pytest.mark.parametrize("mode, k", [("exact", 49), ("cap", PER_LAYER)])
def test_one_call_equals_per_layer_and_batch_independence(sds, mode, k):
    geom, _ = sds("deits16")
    keep = _keep(k)
    B = 7
    e = _engine(sds, "deits16", "fp32", B)
    try:
        e.set_token_budget(keep, mode)
        x = synth.make_pixels(B, geom, seed=5).cuda()
        r = _fwd(e, x, MT)
        h = e.embed(x)
        masks = []
        for l in range(geom.layers):
            m, _, _ = e.layer_forward(l, h, MT)
            masks.append(m)
        logits = e.head(h)
        torch.cuda.synchronize()
        assert torch.equal(torch.stack(masks), r["masks"]) and torch.equal(logits, r["logits"])
        for b in (0, 3, 6):
            one = _fwd(e, x[b:b + 1].contiguous(), MT)
            assert torch.equal(one["logits"][0], r["logits"][b]), b
            assert torch.equal(one["masks"][:, 0], r["masks"][:, b]), b
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 5. precedence and graphs
def test_forced_masks_override_and_graphs_are_dropped(sds):
    geom, _ = sds("deits16")
    B = 8
    e = _engine(sds, "deits16", "bf16", B)
    try:
        x = synth.make_pixels(B, geom, seed=9).cuda()
        base = _fwd(e, x, MT, True)                                      # captured without a budget
        e.set_token_budget(49, "exact")
        r = _fwd(e, x, MT, True)
        assert (r["n_active"] == 50).all(), "a graph captured before the budget change was replayed"
        assert not torch.equal(r["masks"], base["masks"])
        g = torch.Generator().manual_seed(4)
        forced = (torch.rand(geom.layers, B, geom.tokens, generator=g) < 0.4).to(torch.uint8)
        forced[:, :, 0] = 1
        for use_graph in (False, True):
            rf = e.forward(x, MT, forced_masks=forced.cuda(), want_masks=True, want_n_active=True, use_graph=use_graph)
            torch.cuda.synchronize()
            assert torch.equal(rf["masks"].cpu(), forced)
            assert torch.equal(rf["n_active"].cpu().long(), forced.long().sum(-1))
        m, _, _ = e.layer_forward(3, e.embed(x), MT, forced_mask=forced[3].cuda())
        torch.cuda.synchronize()
        assert torch.equal(m.cpu(), forced[3])
    finally:
        e.close()


def test_profile_reports_the_budget_kernel(sds):
    geom, _ = sds("deits16")
    e = _engine(sds, "deits16", "bf16", 8)
    try:
        x = synth.make_pixels(8, geom, seed=2).cuda()
        e.set_token_budget(49, "exact")
        e.forward(x, MT, use_graph=True)              # the warm-up that sets the graph's hints, outside the profile
        e.profile_begin()
        e.forward(x, MT, use_graph=True)
        kinds = [k for k, _ in e.profile_end()]
        assert kinds.count("budget_mask") == geom.layers
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 6. fine-tuning
def _check_train_masks(masks, rscores, keep, label):
    """k + 1 tokens per image, and the rule on the reference's teacher-forced scores outside the near-cut band"""
    m = masks.cpu().numpy().astype(bool)
    assert np.array_equal(m.sum(-1), np.broadcast_to(np.array(keep)[:, None] + 1, m.shape[:2])), label
    rs = rscores.detach().cpu().float().numpy()
    bad = 0
    for l in range(len(keep)):
        want = TB.budget_mask(rs[l], keep[l], "exact", MT)
        near = TB.near_cut(rs[l], keep[l], "exact", MT)
        diff = (m[l] != want).any(-1)
        assert not (diff & ~near).any(), f"{label}: layer {l} differs from the rule outside the band"
        bad += int(diff.sum())
    print(f"[{label}] {bad} image-layers inside the band decided differently")


# the joint objective's pos_weight is mean / (1 - mean): a layer keeping everything would weigh its loss by 1e16
JOINT_KEEP = [98, 49, 147, 24, 98, 64, 120, 49, 98, 30, 160, 98]


@pytest.mark.parametrize("kv, joint", [("active", False), ("all", False), ("active", True)])
def test_split_finetuning_under_exact_budget(sds, kv, joint):
    geom, sd = sds("deits16")
    B, keep = 16, (JOINT_KEEP if joint else PER_LAYER)
    e = _engine(sds, "deits16", "fp32", B, kv)
    try:
        e.set_token_budget(keep, "exact")
        x = synth.make_pixels(B, geom, seed=31, kind="randn").cuda()
        gen = torch.Generator().manual_seed(31)
        out = e.backbone_forward_train(x, MT, with_layer_losses=joint)
        logits = out[0] if joint else out
        masks = e.backbone_train_masks()
        labels = torch.randint(0, geom.classes, (B,), generator=gen).cuda()
        lg = logits.detach().clone().requires_grad_(True)
        torch.nn.functional.cross_entropy(lg, labels).backward()
        dlosses = torch.rand(geom.layers, generator=gen).cuda() * 2 + 0.25 if joint else None
        res = e.backbone_backward(lg.grad, dlosses)
        torch.cuda.synchronize()
        flat, cflat = res if joint else (res, None)
        got = FT._flat_to_dict(flat, e.backbone_grad_slices())
        if joint:
            got.update(FT._comp_to_dict(cflat, geom))
        p = FT.reference_params(sd, "cuda")
        ref_fwd = reference_forward_kv_all if kv == "all" else FT.reference_forward
        rl, _, rs, rlosses = ref_fwd(p, x.double(), MT, geom.heads, forced_masks=masks, joint=joint)
        outs, ups = [rl], [lg.grad.double()]
        if joint:
            outs.append(rlosses)
            ups.append(dlosses.double())
        ref = FT.reference_grads(p, outs, ups, joint)
        label = f"split kv={kv}{' joint' if joint else ''}"
        assert float((logits.double() - rl.detach()).abs().max()) < 1e-4
        _check_train_masks(masks, rs, keep, label)
        FT._compare(got, ref, label)
    finally:
        e.close()


def test_bf16_finetuning_under_exact_budget(sds):
    geom, sd = sds("deits16")
    # no k = 0 layer: with one token per image the q / k gradients are zero in exact arithmetic, and the rounded
    # reference's are rounding noise that a relative bar cannot compare
    B, keep = 16, [98, 49, 147, 24, 196, 64, 120, 5, 98, 30, 160, 1]
    e = _engine(sds, "deits16", "fp32", B)
    try:
        e.set_train_precision("bf16")
        e.set_token_budget(keep, "exact")
        x, logits, masks, dl, dls, got = BF._step(e, geom, sd, B, MT, "ce", seed=33)
        rl, rs, ref = BF._reference_grads(sd, geom, x, MT, masks, dl, dls, True)
        lerr = (logits.double() - rl).abs()
        assert float(lerr.max()) < BF.B16.LOGITS_TOL and float(lerr.pow(2).mean().sqrt()) < BF.B16.LOGITS_RMS
        fails = BF._compare(got, ref, BF.STEP_FROB, BF.STEP_MAX, BF.COMP_FROB, BF.COMP_MAX, "bf16 exact budget")
        assert not fails, fails[:8]
        m = masks.cpu().numpy().astype(bool)
        assert np.array_equal(m.sum(-1), np.broadcast_to(np.array(keep)[:, None] + 1, m.shape[:2]))
        # the bf16 stream departs from fp64 by more than 1e-4: check the rule where the cut is clear of that
        rs = rs.detach().cpu().float().numpy()
        for l in range(geom.layers):
            want = TB.budget_mask(rs[l], keep[l], "exact", MT)
            near = TB.near_cut(rs[l], keep[l], "exact", MT, band=BF.DECISION_BAND)
            assert not ((m[l] != want).any(-1) & ~near).any(), l
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 7. refusals
def test_refusals(sds):
    import psv_native
    lib = psv_native.lib
    geom, _ = sds("deits16")
    e = _engine(sds, "deits16", "fp32", 4)
    try:
        h = e._h
        arr = (C.c_int32 * 12)(*([49] * 12))
        assert lib.psv_set_token_budget(h, 3, arr) == ERR_INVALID
        assert lib.psv_set_token_budget(h, -1, arr) == ERR_INVALID
        assert lib.psv_set_token_budget(h, 1, None) == ERR_INVALID
        for bad in (-1, 197):
            a = (C.c_int32 * 12)(*([49] * 11 + [bad]))
            assert lib.psv_set_token_budget(h, 2, a) == ERR_INVALID
        assert lib.psv_set_token_budget(h, 0, None) == 0
        x = synth.make_pixels(4, geom, seed=1).cuda()
        e.set_token_budget(49, "exact")
        with pytest.raises(psv_native.PsvError, match=r"\(-4\)"):
            e.compressor_grads(x, MT)
        e.set_skip_criterion("similarity", 0.9)
        with pytest.raises(psv_native.PsvError, match=r"\(-4\)"):
            e.forward(x, MT)
        with pytest.raises(psv_native.PsvError, match=r"\(-4\)"):
            e.forward_host(x.cpu().pin_memory(), MT)
        with pytest.raises(psv_native.PsvError, match=r"\(-4\)"):
            e.backbone_forward_train(x, MT)
        # with forced masks the similarity criterion is not consulted: allowed
        forced = torch.ones(geom.layers, 4, geom.tokens, dtype=torch.uint8)
        r = e.forward(x, MT, forced_masks=forced, want_n_active=True)
        torch.cuda.synchronize()
        assert (r["n_active"] == geom.tokens).all()
        # the per-layer label entry points take masks and do not depend on the budget
        hid = e.embed(x)
        m, s, _ = e.layer_forward(0, hid.clone(), MT)
        e.layer_stats(0, hid, m, s, 0.9)
        e.similarity_mask(0, hid, 0.9)
        e.compressor_layer_grads(0, hid, m, s)
        e.set_skip_criterion("mlp", 0.9)
        e.set_token_budget(None)
        e.compressor_grads(x, MT)
        torch.cuda.synchronize()
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------ 8. the drop-in
def _drop_in(sd, geom):
    import model_utils
    from transformers.models.vit.modeling_vit import ViTConfig
    cfg = ViTConfig(hidden_size=geom.hidden, num_attention_heads=geom.heads, intermediate_size=geom.ffn)
    cfg.num_labels = geom.classes
    model = model_utils.ModifiedViTModel(cfg, 0.9, MT, 0)
    model.load_state_dict(sd, strict=False)
    return model.to("cuda")


def test_drop_in_routes(sds):
    geom, sd = sds("deits16")
    model = _drop_in(sd, geom).eval()
    x = synth.make_pixels(5, geom, seed=12).cuda()
    model.token_budget = PER_LAYER
    with torch.no_grad():
        one = model(x, output_mask=True)
        per = model(x, output_mask=True, output_hidden_states=True)
    for l, (a, b) in enumerate(zip(one.boolean_masks, per.boolean_masks)):
        assert (a.sum(1) == PER_LAYER[l] + 1).all(), l
        assert torch.equal(a, b), l
    assert torch.equal(one.n_active.cpu(), torch.tensor(PER_LAYER)[:, None].int().expand(-1, 5) + 1)
    assert float((one.logits - per.logits).abs().max()) < 1e-5
    model.token_budget, model.token_budget_mode = 10, "cap"
    with torch.no_grad():
        cap = model(x, output_mask=True)
    for m in cap.boolean_masks:
        assert (m.sum(1) <= 11).all()
    model.token_budget = None
    with torch.no_grad():
        plain = model(x)
    assert model._psv_engine._token_budget is None and torch.isfinite(plain.logits).all()


def test_drop_in_trains_under_a_budget(sds):
    from main_model_utils import synthetic_loader, train
    geom, sd = sds("deits16")
    model = _drop_in(sd, geom)
    model.psv_precision = "fp32"
    model.token_budget = 98
    loader = synthetic_loader(8, 8, geom=geom, seed=5, kind="randn", pin_memory=False)
    hist = train(model, loader, None, "cuda", num_epochs=8, loss_type="classification", lr=1e-4)
    print(f"\nexact budget 98: loss {hist[0]:.4f} -> {hist[-1]:.4f}")
    assert all(np.isfinite(h) for h in hist) and hist[-1] < hist[0]
    import psv_native
    with pytest.raises(psv_native.PsvError, match=r"\(-4\)"):          # native compressor training refuses a budget
        model._psv_engine.compressor_grads(next(iter(loader))[0].cuda(), MT)
