"""The bf16 inference path against a float64 reference that rounds to bf16 where the kernels round
(``oracle/bf16_reference.py``), from single kernels up to the logits, on DeiT-S, ViT-B and ViT-L.

The other bf16 tests compare against the fp32 oracle, so their bars (3e-2 per layer, 2e-2 on the logits and on
psv_attention) must also absorb the bf16 weight and activation rounding, and defects of a few 1e-3 pass them.  Here
the reference rounds the same way, so what is left is the kernels' own arithmetic: fp32 accumulation order, ex2.approx,
the fast erf-GELU, and bf16 rounding flips at ties that fp32 noise moves.

* CPU: with ``rounding=False`` the reference equals the fp64 oracle.  Defects planted in the reference (softmax scale
  1/7.9, tanh-GELU, a dropped first or last key, an unwritten last query row, the second query tile left unnormalised,
  a skipped last k-block) must move the output, on the GPU cases' own inputs, by at least 2x one of the stage's bars:
  the max-abs bar at some element, or the rms bar.  Each defect is caught this way at the kernel stage it lives in;
  the layer and logits bars cannot see a softmax scale of 1/7.9 or tanh-GELU (CAUGHT_ELSEWHERE says why and names the
  stage that does).  The test prints each defect's margin and whether the older bar would have caught it.
* GPU: psv_gemm (all epilogues, GELU, ragged M, tail waves), psv_attention (tc / mma / pk; boundary lengths, mixed
  batches, the tcgen05 kernel's lazy rescale, dominant and tied keys, |v| ~ 100, q / k scaled x1 / x2 / x4 / x8),
  psv_layer_forward teacher-forced on four mask patterns in both kv modes (this is the only way to reach the unit table
  that the compaction kernel builds and the keep-all-keys mma path), and teacher-forced logits.

The GPU tests print the worst error per stage and geometry; the bars below sit about 3-4x above what a B200 measured.
"""
import math

import pytest
import torch

import synth
from oracle import bf16_reference as R
from oracle import vit_skip_oracle as O

GEOMS = {"deits16": synth.DEIT_S16, "vitb16": synth.VIT_B16, "vitl16": synth.VIT_L16}
MT = 0.5

# ---------------------------------------------------------------------------------------------------------------- bars
# Worst errors measured on a B200 (1000 W) are next to each bar.  A bar may sit less than 4x above its measurement when
# that is what keeps it 2x under a planted defect; the runs are deterministic (fixed seeds, deterministic kernels).
# psv_gemm, bf16 output: |out - bf16(ref)| <= ulp(bf16(ref)) + GEMM_ACC * 2^-24 * S (+ GELU_FLOOR with GELU), where
# S = sum_k |a w| + |bias| bounds what fp32 accumulation can lose; fp32 output: |out - ref| <= GEMM_ACC * 2^-24 * S,
# with |residual| or |base| added to S.  Measured: bf16 outputs at most 1 ulp (err / bar 0.999), fp32 outputs
# 11 * 2^-24 * S (FC2 at D = 1024).
GEMM_ACC = 48.0
GELU_FLOOR = 4e-6            # gelu_erf_fast is within 1.1e-6 of the exact GELU
# psv_attention: |ctx - ref| <= ulp(ref) + ATTN_V * max |v| of the (image, head); measured err / bar 0.40 (tc kernel)
ATTN_V = 8e-3
# rms over all elements of |ctx - ref| / max |v| of the (image, head); measured 2.5e-4 (tc), 1.4e-4 (pk), 1.2e-4 (mma).
# The softmax-scale defect moves it by 1.57e-3, so the bar stays at 3x the measurement.
ATTN_RMS = 7.5e-4
# psv_layer_forward, max-abs over every row (active and keep-all-keys mode) and rms over the active rows; measured
# 2.9e-3 max-abs (a CLS row) and 6.3e-4 rms (keep-all-keys mode)
LAYER_TOL = 1.2e-2
LAYER_RMS = 2e-3
# logits, max-abs and rms; measured 1.17e-2 and 3.2e-3 (ViT-L with the tc kernel, ViT-B with the tc kernel)
LOGITS_TOL = 5e-2
LOGITS_RMS = 1.2e-2

# Defects a stage's bars cannot separate from what remains of the kernels' rounding, and the stage whose bar catches
# them.  The reference rounds P against the final max; the kernels round against a running (mma, pk) or lazily moved
# (tc) max, so every probability differs by up to 2^-9, every ctx element moves by about 1e-4 of max |v|, and ctx then
# rounds to the other bf16 neighbour at a few percent of the elements.  That dense noise (6.3e-4 rms per layer, 3e-3
# on the logits) is as large as what a softmax scale of 1/7.9 (9e-4 rms per layer) or tanh-GELU (1.9e-4) leave.
CAUGHT_ELSEWHERE = {
    "layer": {"scale 1/7.9": "psv_attention (rms)", "tanh-GELU": "psv_gemm (FC1)"},
    "logits": {"scale 1/7.9": "psv_attention (rms)", "tanh-GELU": "psv_gemm (FC1)",
               "last query row unwritten": "psv_attention and layer"},
}

# the bars of the older tests against the fp32 oracle, for the printout
OLD = {"gemm_bf16": "2e-2 * max|ref|", "gemm_fp32": "2e-4 abs", "attention": "2e-2 abs", "layer": "3e-2 abs (kv_all 6e-2)",
       "logits": "2e-2 abs"}

WORST = {}


def _record(stage, geom, err):
    key = (stage, geom)
    WORST[key] = max(WORST.get(key, 0.0), float(err))


@pytest.fixture(scope="module")
def sds(state_dicts):
    """name -> fp32 state dict (seed 42); ViT-L is built here"""
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = state_dicts(name)[1] if name != "vitl16" else synth.make_state_dict(synth.VIT_L16, seed=42)
        return cache[name]
    return get


def ulp_bf16(x):
    """spacing of bf16 values at |x| (normal range)"""
    _, e = torch.frexp(x.abs().to(torch.float64).clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x, dtype=torch.float64), e - 8)


def _margin(dist, bar):
    """max over elements of dist / bar.  NaN -- a dropped key that leaves a one-token image without keys -- is left
    out: such a defect is caught there trivially, the question is whether it is caught on the longer images."""
    return float(torch.nan_to_num(dist / bar, nan=0.0).max())


# ---------------------------------------------------------------------------------------------------------------- defects
def attend_variant(scale=R.SCALE, keys=slice(None), zero_last_row=False, unnormalised_from=None):
    """R.attend with one planted defect"""
    def f(q, k, v, rounding=True):
        k, v = k[:, keys], v[:, keys]
        if k.shape[1] == 0:                                     # no key left: the output is undefined
            return torch.full((q.shape[1], q.shape[0] * q.shape[2]), math.nan, dtype=q.dtype, device=q.device)
        s = torch.matmul(q, k.transpose(1, 2)) * scale
        e = torch.exp(s - s.amax(-1, keepdim=True))
        den = e.sum(-1, keepdim=True)
        if unnormalised_from is not None:
            den[:, unnormalised_from:] = 1.0
        ctx = R.rnd((torch.matmul(R.rnd(e, rounding), v) / den).transpose(0, 1).reshape(q.shape[1], -1), rounding)
        if zero_last_row:
            ctx[-1] = 0.0
        return ctx
    return f


ATTN_DEFECTS = {
    "scale 1/7.9": attend_variant(scale=1 / 7.9),
    "last key dropped": attend_variant(keys=slice(0, -1)),
    "first key dropped": attend_variant(keys=slice(1, None)),
    "last query row unwritten": attend_variant(zero_last_row=True),
    "2nd query tile unnormalised": attend_variant(unnormalised_from=128),
}
LAYER_DEFECTS = dict(ATTN_DEFECTS, **{"tanh-GELU": "tanh"})


def _layer_variant(sd, l, h, mask, kv_all, defect):
    d = LAYER_DEFECTS[defect]
    if isinstance(d, str):
        return R.layer(sd, l, h, mask, kv_all, gelu=d)
    return R.layer(sd, l, h, mask, kv_all, attend_fn=d)


# ---------------------------------------------------------------------------------------------------------------- inputs
GEMM_KINDS = {
    # name: (N / D, K / D or fixed K, epilogue, gelu)
    "qkv": (3, 1, "bf16", False),
    "fc1": (4, 1, "bf16", True),
    "proj": (1, 1, "red", False),
    "fc2": (1, 4, "red", False),
    "store_res": (1, 1, "store", False),
    "embed": (1, None, "store", False),     # K = 3 * 16 * 16
}
GEMM_MS = (77, 1000, 128 * 150 - 3)          # one ragged tile; a few waves; many waves with a ragged tail


def gemm_case(D, kind, M):
    nmul, kmul, epi, gelu = GEMM_KINDS[kind]
    N, K = nmul * D, (kmul * D if kmul else 768)
    g = torch.Generator().manual_seed(D * 1009 + M * 7 + len(kind))
    a = torch.randn(M, K, generator=g).to(torch.bfloat16)
    w = ((torch.rand(N, K, generator=g) * 2 - 1) * K ** -0.5).to(torch.bfloat16)
    bias = (torch.rand(N, generator=g) * 2 - 1) * K ** -0.5
    extra = torch.randn(M, N, generator=g) if epi != "bf16" else None      # residual (store) or base (red)
    return dict(a=a, w=w, bias=bias, extra=extra, epi=epi, gelu=gelu)


def gemm_reference(c, rows=None, k_drop=0, gelu="none"):
    """(ref fp64, S) on rows `rows`; k_drop: the last k_drop columns of K left out (a planted defect)"""
    a, w = c["a"].double(), c["w"].double()
    if rows is not None:
        a = a[rows]
    dev = a.device
    K = a.shape[1] - k_drop
    ref = a[:, :K] @ w[:, :K].t() + c["bias"].double().to(dev)
    S = a.abs() @ w.abs().t() + c["bias"].double().to(dev).abs()
    if c["gelu"]:
        ref = torch.nn.functional.gelu(ref, approximate=gelu)
    if c["extra"] is not None:
        x = c["extra"].double().to(dev) if rows is None else c["extra"][rows].double().to(dev)
        ref, S = ref + x, S + x.abs()
    return ref, S


def gemm_bar(ref, S, c):
    acc = GEMM_ACC * 2.0 ** -24 * S
    if c["epi"] != "bf16":
        return acc
    return ulp_bf16(R.rnd(ref)) + acc + (GELU_FLOOR if c["gelu"] else 0.0)


LENGTHS = [1, 2, 15, 16, 17, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, 159, 160, 161, 191, 192, 193, 196, 197]
ATTN_CASES = ["lengths_x1", "lengths_x2", "lengths_x4", "lengths_x8", "mixed", "lazy_rescale", "dominant", "ties", "big_v"]


def attention_case(D, name):
    """(qkv bf16 [T, 3D], lengths)"""
    g = torch.Generator().manual_seed(D + 31 * ATTN_CASES.index(name))
    if name.startswith("lengths"):
        lens = LENGTHS
    elif name == "mixed":
        lens = [int(x) for x in torch.randint(1, 198, (48,), generator=g)]
    elif name == "lazy_rescale":
        lens = [33, 64, 65, 97, 129, 160, 197]
    else:
        lens = [1, 17, 64, 128, 129, 197]
    T = sum(lens)
    qkv = torch.randn(T, 3 * D, generator=g, dtype=torch.float64)
    if name.startswith("lengths"):
        qkv[:, :2 * D] *= float(name[-1])
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    H = D // 64
    for b, n in enumerate(lens):
        r0, r1 = cu[b], cu[b + 1]
        for hh in range(H):
            qs, ks, vs = (slice(j * D + hh * 64, j * D + hh * 64 + 64) for j in range(3))
            if name == "lazy_rescale" or name == "dominant":
                # every query shares a direction u; the key at the last real row (lazy_rescale: a late 32-key chunk)
                # or at the middle row (dominant) points along u, so its logit beats the first chunk's maximum by
                # roughly 10..14 log2 units -- past the 8 at which attention_tc.cu moves its reference max
                u = torch.ones(64, dtype=torch.float64)
                qkv[r0:r1, qs] = qkv[r0:r1, qs] * 0.5 + u
                kr = r1 - 1 if name == "lazy_rescale" else r0 + n // 2
                qkv[kr, ks] = u * (1.2 + 0.1 * (hh % 4))
            elif name == "ties":
                qkv[r0:r1, ks] = qkv[r0, ks].clone()                     # every key identical: a uniform softmax
            elif name == "big_v":
                qkv[r0:r1, vs] *= 100.0
    return qkv.to(torch.bfloat16), lens


def _cu(lens, device):
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    return torch.tensor(cu, dtype=torch.int32, device=device)


def _vmax(qkv, lens, D):
    """max |v| of each row's (image, head), per element [T, D]"""
    H = D // 64
    v = qkv[:, 2 * D:].double().abs().reshape(-1, H, 64).amax(-1)            # [T, H]
    vmax = torch.empty_like(v)
    r0 = 0
    for n in lens:
        vmax[r0:r0 + n] = v[r0:r0 + n].amax(0, keepdim=True)
        r0 += n
    return vmax.repeat_interleave(64, dim=1)


def attention_rms(dist, qkv, lens, D):
    """rms over all elements of dist / max |v| of the (image, head); NaN rows (no key left) are left out"""
    r = dist / _vmax(qkv, lens, D)
    r = r[torch.isfinite(r)]
    return r.pow(2).mean().sqrt()


def attention_bar(ref, qkv, lens, D):
    """ulp(ref) + ATTN_V * max |v| of the (image, head), per element"""
    return ulp_bf16(ref) + ATTN_V * _vmax(qkv, lens, D)


LAYER_CASES = ["natural", "all", "cls_only", "crafted"]
CRAFTED = [1, 31, 32, 33, 64, 65, 127, 128, 129, 196, 197]


def layer_case(sd, name, geom, case):
    """(layer index, input h fp32 [B, N, D], mask bool [B, N]); the input is the embedding of synthetic pixels, the
    weights those of the middle layer"""
    l = geom.layers // 2
    B = {"natural": 6, "all": 3, "cls_only": 6, "crafted": len(CRAFTED)}[case]
    x = synth.make_pixels(B, geom, seed=700 + LAYER_CASES.index(case))
    with torch.no_grad():
        h = O.embed(sd, x)
    N = geom.tokens
    if case == "natural":
        mask = O.skip_mask(O.compressor_scores(sd, l, h), MT)
    elif case == "all":
        mask = torch.ones(B, N, dtype=torch.bool)
    elif case == "cls_only":
        mask = torch.zeros(B, N, dtype=torch.bool)
        mask[:, 0] = True
    else:
        g = torch.Generator().manual_seed(5)
        mask = torch.zeros(B, N, dtype=torch.bool)
        mask[:, 0] = True
        for b, n in enumerate(CRAFTED):
            mask[b, torch.randperm(N - 1, generator=g)[:n - 1] + 1] = True
    assert mask[:, 0].all()
    return l, h, mask


E2E_BATCH = {"deits16": 6, "vitb16": 4, "vitl16": 2}


def e2e_pixels(name):
    return synth.make_pixels(E2E_BATCH[name], GEOMS[name], seed=900 + len(name))


# ================================================================================================================ CPU
@pytest.mark.parametrize("name", list(GEOMS))
def test_reference_without_rounding_is_the_oracle(name, sds):
    """rounding=False: embed, layer (both kv modes) and head equal the fp64 oracle (vit_layer, vit_layer_query_pruned)"""
    geom, sd = GEOMS[name], sds(name)
    sd64 = {k: v.double() for k, v in sd.items()}
    x = synth.make_pixels(2, geom, seed=11)
    with torch.no_grad():
        h = R.embed(sd, x, rounding=False)
        assert (h - O.embed(sd64, x.double())).abs().max() < 1e-12
        l = geom.layers - 1
        mask = O.skip_mask(O.compressor_scores(sd, l, h.float()), MT)
        mask[1, 1:60] = True
        assert (R.skip_mask(sd, l, h, MT) == O.skip_mask(O.compressor_scores(sd64, l, h), MT)).all()
        for kv_all in (False, True):
            out = R.layer(sd, l, h, mask, kv_all=kv_all, rounding=False)
            ref = h.clone()
            for b in range(2):
                if kv_all:
                    ref[b][mask[b]] = O.vit_layer_query_pruned(sd64, l, h[b].unsqueeze(0), mask[b])[0]
                else:
                    ref[b][mask[b]] = O.vit_layer(sd64, l, h[b][mask[b]].unsqueeze(0))[0]
            err = float((out - ref).abs().max())
            assert err < 1e-10, f"kv_all={kv_all}: {err}"
            # rounding moves the output by bf16-sized amounts, not more
            dev = float((R.layer(sd, l, h, mask, kv_all=kv_all) - ref).abs().max())
            assert 1e-4 < dev < 3e-2, dev
        assert (R.head(sd, h) - O.head(sd64, h)).abs().max() < 1e-12


def _report(bar_name, bar_text, margins, old_dists, old_bar):
    """margins: defect -> (max over cases of dist / bar); old_dists: defect -> max abs distance (None: no old bar)"""
    elsewhere = CAUGHT_ELSEWHERE.get(old_bar, {})
    print(f"\n[{bar_name}] bar {bar_text}; older bar {OLD[old_bar]}")
    for d, m in margins.items():
        od = old_dists.get(d)
        old = "" if od is None else f"; older bar would have {'caught' if od[0] > od[1] else 'PASSED'} it " \
                                     f"(max abs {od[0]:.2e})"
        where = f"; caught by {elsewhere[d]}" if d in elsewhere else ""
        print(f"    {d:30s} margin {m:9.2f}x{old}{where}")
    low = {d: m for d, m in margins.items() if not m >= 2.0 and d not in elsewhere}
    assert not low, f"[{bar_name}] defects within 2x of the bar: {low}"


@pytest.mark.parametrize("D", [384, 768, 1024])
def test_gemm_bars_catch_planted_defects(D):
    """tanh-GELU (FC1) and a skipped last k-block (every epilogue) against the psv_gemm bars, on the GPU cases' inputs
    (the first 256 and last 64 rows)"""
    margins, old = {}, {}
    for kind in GEMM_KINDS:
        for M in GEMM_MS:
            c = gemm_case(D, kind, M)
            rows = torch.cat((torch.arange(min(256, M)), torch.arange(max(0, M - 64), M))).unique()
            ref, S = gemm_reference(c, rows)
            bar = gemm_bar(ref, S, c)
            ref_out = R.rnd(ref) if c["epi"] == "bf16" else ref
            defects = {"last k-block skipped": dict(k_drop=64)}
            if c["gelu"]:
                defects["tanh-GELU"] = dict(gelu="tanh")
            for dname, kw in defects.items():
                dref, _ = gemm_reference(c, rows, **kw)
                dout = R.rnd(dref) if c["epi"] == "bf16" else dref
                dist = (dout - ref_out).abs()
                key = f"{dname} ({kind})"
                margins[key] = max(margins.get(key, 0.0), _margin(dist, bar))
                old_bar = 2e-2 * float(ref.abs().max()) if c["epi"] == "bf16" else 2e-4
                od = old.get(key, (0.0, old_bar))
                old[key] = (max(od[0], float(dist.max())), old_bar)
    _report(f"psv_gemm D={D}", f"ulp + {GEMM_ACC} * 2^-24 * S (+{GELU_FLOOR} with GELU)", margins, old,
            "gemm_bf16")


@pytest.mark.parametrize("name", list(GEOMS))
def test_attention_bar_catches_planted_defects(name):
    D = GEOMS[name].hidden
    margins, old = {}, {}
    for case in ATTN_CASES:
        qkv, lens = attention_case(D, case)
        cu = _cu(lens, "cpu")
        ref = R.attention(qkv, cu, D // 64)
        bar = attention_bar(ref, qkv, lens, D)
        for dname, fn in ATTN_DEFECTS.items():
            dist = (R.attention(qkv, cu, D // 64, attend_fn=fn) - ref).abs()
            m = max(_margin(dist, bar), float(attention_rms(dist, qkv, lens, D)) / ATTN_RMS)
            margins[dname] = max(margins.get(dname, 0.0), m)
            old[dname] = (max(old.get(dname, (0.0,))[0], float(torch.nan_to_num(dist, nan=0.0).max())), 2e-2)
    _report(f"psv_attention {name}", f"ulp + {ATTN_V} * max|v|, rms {ATTN_RMS} * max|v|", margins, old, "attention")


@pytest.mark.parametrize("name", list(GEOMS))
def test_layer_bar_catches_planted_defects(name, sds):
    geom, sd = GEOMS[name], sds(name)
    margins, old = {}, {}
    with torch.no_grad():
        for case in LAYER_CASES:
            l, h, mask = layer_case(sd, name, geom, case)
            for kv_all in (False, True):
                ref = R.layer(sd, l, h, mask, kv_all)
                for dname in LAYER_DEFECTS:
                    dist = (_layer_variant(sd, l, h, mask, kv_all, dname) - ref).abs()
                    rms = float(torch.nan_to_num(dist[mask], nan=0.0).pow(2).mean().sqrt())
                    m = max(_margin(dist, LAYER_TOL), rms / LAYER_RMS)
                    margins[dname] = max(margins.get(dname, 0.0), m)
                    d = float(torch.nan_to_num(dist, nan=0.0).max())
                    old_bar = 6e-2 if kv_all else 3e-2
                    if d / old_bar > old.get(dname, (0.0, 1.0))[0] / old.get(dname, (0.0, 1.0))[1]:
                        old[dname] = (d, old_bar)
    _report(f"layer {name}", f"{LAYER_TOL} abs, rms {LAYER_RMS}", margins, old, "layer")


@pytest.mark.parametrize("name", list(GEOMS))
def test_logits_bar_catches_planted_defects(name, sds):
    """each defect planted in every layer of the chained reference, on the pixels of the GPU case"""
    sd = sds(name)
    x = e2e_pixels(name)
    margins, old = {}, {}
    with torch.no_grad():
        ref, masks = R.forward(sd, x, MT)
        for dname, d in LAYER_DEFECTS.items():
            kw = dict(gelu=d) if isinstance(d, str) else dict(attend_fn=d)
            logits, _ = R.forward(sd, x, MT, forced_masks=masks, **kw)
            dist = (logits - ref).abs()
            margins[dname] = max(_margin(dist, LOGITS_TOL),
                                 float(torch.nan_to_num(dist, nan=0.0).pow(2).mean().sqrt()) / LOGITS_RMS)
            old[dname] = (float(torch.nan_to_num(dist, nan=0.0).max()), 2e-2)
    _report(f"logits {name}", f"{LOGITS_TOL} abs, rms {LOGITS_RMS}", margins, old, "logits")


# ================================================================================================================ GPU
def _engine(name, sd, max_batch):
    import psv_native
    e = psv_native.Engine(GEOMS[name], "bf16", max_batch)
    e.load_state_dict(sd)
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GEOMS))
def test_gpu_gemm_against_rounded_fp64(name, sds):
    D = GEOMS[name].hidden
    e = _engine(name, sds(name), 4)
    failed = []
    for kind in GEMM_KINDS:
        for M in GEMM_MS:
            c = gemm_case(D, kind, M)
            a, w, bias = c["a"].cuda(), c["w"].cuda(), c["bias"].cuda()
            if c["epi"] == "bf16":
                out = e.gemm(a, w, bias, out_fp32=False, gelu=c["gelu"])
            elif c["epi"] == "store":
                out = e.gemm(a, w, bias, c["extra"].cuda(), out_fp32=True)
            else:
                out = e.gemm(a, w, bias, out_fp32=True, accumulate_into=c["extra"].cuda())
            torch.cuda.synchronize()
            cg = dict(c, a=a, w=w)
            ref, S = gemm_reference(cg)
            bar = gemm_bar(ref, S, c)
            want = R.rnd(ref) if c["epi"] == "bf16" else ref
            err = (out.double() - want).abs()
            ratio = float((err / bar).max())
            _record(f"gemm {kind}", name, ratio)
            worst = int((err / bar).argmax())
            print(f"[gemm {name} {kind} M={M}] worst err / bar {ratio:.3f} (err {float(err.view(-1)[worst]):.3e} at "
                  f"row {worst // out.shape[1]}, col {worst % out.shape[1]}; max-abs {float(err.max()):.3e})")
            if not ratio <= 1.0:
                failed.append(f"{kind} M={M}: err / bar {ratio:.3f}")
            del out, ref, S, bar, err
    e.close()
    assert not failed, failed


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GEOMS))
def test_gpu_attention_against_rounded_fp64(name, sds):
    D = GEOMS[name].hidden
    e = _engine(name, sds(name), 64)
    failed = []
    try:
        for case in ATTN_CASES:
            qkv_cpu, lens = attention_case(D, case)
            qkv = qkv_cpu.cuda()
            cu = _cu(lens, "cuda")
            ref = R.attention(qkv, cu.cpu(), D // 64)
            bar = attention_bar(ref, qkv, lens, D)
            for kind in ("tc", "mma", "pk"):
                e.set_attention_kernel(kind)
                ctx = e.attention(qkv, cu)
                torch.cuda.synchronize()
                err = (ctx.double() - ref).abs()
                r = err / bar
                rms = float(attention_rms(err, qkv, lens, D))
                _record(f"attention rms {kind}", name, rms)
                if not rms <= ATTN_RMS:
                    failed.append(f"{case} {kind}: rms / max|v| {rms:.3e}")
                ratio = float(torch.nan_to_num(r, nan=math.inf).max())
                _record(f"attention {kind}", name, ratio)
                i = int(torch.nan_to_num(r, nan=math.inf).argmax())
                row, col = i // D, i % D
                img = next(b for b in range(len(lens)) if int(cu[b + 1]) > row)
                print(f"[attention {name} {case} {kind}] rms / max|v| {rms:.3e}; worst err / bar {ratio:.3f} (image {img} n={lens[img]}, "
                      f"query {row - int(cu[img])}, head {col // 64}; err {float(err.view(-1)[i]):.3e}, "
                      f"max-abs {float(err.max()):.3e})")
                if not ratio <= 1.0:
                    failed.append(f"{case} {kind}: image {img} (n={lens[img]}) query {row - int(cu[img])} "
                                  f"head {col // 64}: err / bar {ratio:.3f}")
    finally:
        e.set_attention_kernel("auto")
        e.close()
    assert not failed, failed


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GEOMS))
def test_gpu_layers_against_rounded_fp64(name, sds):
    """psv_layer_forward teacher-forced on the reference's input: every row against the reference, skipped rows
    bit-identical, in active mode with each attention kernel and in keep-all-keys mode"""
    geom, sd = GEOMS[name], sds(name)
    e = _engine(name, sd, 16)
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    failed = []
    try:
        for case in LAYER_CASES:
            l, h, mask = layer_case(sd, name, geom, case)
            hg, mg = h.cuda(), mask.cuda()
            for kv_all in (False, True):
                ref = R.layer(sd_gpu, l, hg, mg, kv_all)
                e.set_kv_mode("all" if kv_all else "active")
                for kind in (("tc", "mma", "pk", "auto") if not kv_all else ("auto",)):
                    e.set_attention_kernel(kind)
                    out = hg.clone()
                    _, _, n_active = e.layer_forward(l, out, MT, forced_mask=mg.to(torch.uint8))
                    torch.cuda.synchronize()
                    assert torch.equal(n_active.cpu().long(), mask.sum(1))
                    assert torch.equal(out[~mg], hg[~mg]), "skipped rows changed"
                    err = (out.double() - ref).abs()
                    worst = float(err.max())
                    rms = float(err[mg].pow(2).mean().sqrt())
                    mode = "kv_all" if kv_all else kind
                    _record(f"layer {mode}", name, worst)
                    _record(f"layer rms {mode}", name, rms)
                    if not rms <= LAYER_RMS:
                        failed.append(f"{case} {mode}: rms {rms:.3e}")
                    i = int(err.argmax())
                    b, t = i // (geom.tokens * geom.hidden), (i // geom.hidden) % geom.tokens
                    print(f"[layer {name} {case} {mode}] rms {rms:.3e}; max-abs err {worst:.3e} (image {b}, token {t}, "
                          f"{int(mask[b].sum())} active)")
                    if not worst <= LAYER_TOL:
                        failed.append(f"{case} {mode}: image {b} token {t}: {worst:.3e}")
    finally:
        e.set_kv_mode("active")
        e.set_attention_kernel("auto")
        e.close()
    assert not failed, failed


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GEOMS))
def test_gpu_logits_against_rounded_fp64(name, sds):
    """the whole forward teacher-forced with the chained reference's masks: automatic kernel choice through the
    CUDA graph and eagerly, and each kernel forced"""
    sd = sds(name)
    e = _engine(name, sd, E2E_BATCH[name])
    x = e2e_pixels(name).cuda()
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    with torch.no_grad():
        ref, masks = R.forward(sd_gpu, x, MT)
    forced = masks.to(torch.uint8)
    failed = []
    try:
        for kind, graph in (("auto", True), ("auto", False), ("tc", False), ("mma", False), ("pk", False)):
            e.set_attention_kernel(kind)
            r = e.forward(x, MT, forced_masks=forced, want_masks=True, use_graph=graph)
            torch.cuda.synchronize()
            assert torch.equal(r["masks"].bool(), masks)
            err = float((r["logits"].double() - ref).abs().max())
            rms = float((r["logits"].double() - ref).pow(2).mean().sqrt())
            _record("logits", name, err)
            _record("logits rms", name, rms)
            print(f"[logits {name} {kind} graph={graph}] rms {rms:.3e}; max-abs err {err:.3e}")
            if not rms <= LOGITS_RMS:
                failed.append(f"{kind} graph={graph}: rms {rms:.3e}")
            if not err <= LOGITS_TOL:
                failed.append(f"{kind} graph={graph}: {err:.3e}")
    finally:
        e.set_attention_kernel("auto")
        e.close()
    assert not failed, failed


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["tc", "pk"])
def test_gpu_fresh_engine_on_dirty_memory(kind, sds):
    """The tcgen05 and packed attention kernels multiply V rows past the last image's last token by P = 0, and the QKV
    GEMM computes those rows from the LN1 rows past the last active row.  A handle created on memory that a previous
    allocation filled with NaN bit patterns must still give finite logits (it did not while act_a was left
    uninitialised at psv_create)."""
    name = "deits16"
    geom, sd = GEOMS[name], sds(name)
    dirty = torch.full((1 << 28,), -1, dtype=torch.int32, device="cuda")   # 1 GiB of 0xffffffff: NaN as fp32 and bf16
    torch.cuda.synchronize()
    del dirty
    torch.cuda.empty_cache()                                               # back to the driver, for psv_create to reuse
    e = _engine(name, sd, 6)
    x = synth.make_pixels(6, geom, seed=77).cuda()
    mask = torch.zeros(geom.layers, 6, geom.tokens, dtype=torch.uint8, device="cuda")
    mask[..., :100] = 1
    try:
        e.set_attention_kernel(kind)
        r = e.forward(x, MT, forced_masks=mask)
        torch.cuda.synchronize()
        assert torch.isfinite(r["logits"]).all(), r["logits"]
    finally:
        e.close()


@pytest.mark.gpu
def test_gpu_print_worst_errors():
    """summary of the worst errors of this module's GPU tests (gemm / attention: err / bar; layer / logits: max-abs)"""
    for (stage, geom), v in sorted(WORST.items()):
        print(f"WORST {stage:20s} {geom:8s} {v:.3e}")
