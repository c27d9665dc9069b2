"""ORACLE -- test infrastructure, NOT product code.

float64 restatement of the bf16 inference path (``PSV_BF16`` handles) that rounds to bf16 (round to nearest even) at
exactly the points where the CUDA path rounds, and nowhere else:

* embed     : im2col pixels -> bf16, patch weights bf16, fp32 output + bias + position embedding (enqueue_embed);
              the CLS row is cls_token + position embedding in fp32 (cls_rows_kernel)
* LN1       : output -> bf16 (gather_ln on the active rows; keep-all-keys mode: ln_rows over all batch x N rows)
* Q/K/V     : bf16 weights, bias added before the bf16 rounding of the output
* attention : P rounded to bf16, ctx -> bf16
* proj, FC2 : bf16 weights, fp32 accumulation into the residual stream (red.add epilogue)
* LN2       : output -> bf16
* FC1       : bf16 weights, GELU applied before the bf16 rounding
* head      : fp32 math (head_kernel), evaluated here in fp64

With ``rounding=False`` every function is exact fp64 math and equals ``oracle.vit_skip_oracle`` evaluated in fp64.
The fp32 storage of the residual stream (about 2^-24 relative) is not modelled.

Attention: the kernels differ in how they get to bf16 P.  attention_mma.cu / attention_pk.cu round P against the
running max and sum the unrounded p; attention_tc.cu rounds against a lazily updated max and sums the rounded P.  This
reference rounds p = exp(s - final max) and normalises by the unrounded sum; what separates it from each kernel is a
per-probability noise of about 2^-9, which the test bars absorb (no kernel's chunking is emulated).

GELU: the exact erf form.  The tensor-core epilogue (gelu_erf_fast in gemm_tc.cu) stays within 1.1e-6 absolute of it
over [-12, 12] but is many bf16 ulps off in relative terms far in the negative tail, so bars comparing GELU outputs
need an absolute floor.

Every function takes the reference-keyed fp32 state dict as it is (any device) and works on the device of its
activation argument, so the same code runs on the CPU and, much faster, on the GPU.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.vit_skip_oracle import LN_EPS, compact

SCALE = 0.125           # 1 / sqrt(64): every supported geometry has 64-wide heads


def rnd(t: torch.Tensor, rounding: bool = True) -> torch.Tensor:
    """round to bf16 (RN-even) and back to fp64; identity without rounding"""
    return t.to(torch.bfloat16).to(torch.float64) if rounding else t.to(torch.float64)


def _p(sd, key, like):
    return sd[key].to(device=like.device, dtype=torch.float64)


def _w(sd, key, like, rounding):
    """a GEMM weight as the bf16 path holds it"""
    return rnd(sd[key].to(like.device), rounding)


def _ln(x, sd, prefix):
    return F.layer_norm(x, (x.shape[-1],), _p(sd, prefix + ".weight", x), _p(sd, prefix + ".bias", x), LN_EPS)


def _qkv_weights(sd, p, like, rounding):
    w = torch.cat([_w(sd, p + f"attention.attention.{n}.weight", like, rounding) for n in ("query", "key", "value")], 0)
    b = torch.cat([_p(sd, p + f"attention.attention.{n}.bias", like) for n in ("query", "key", "value")], 0)
    return w, b


# ----------------------------------------------------------------------------- embeddings
def embed(sd, pixel_values: torch.Tensor, rounding: bool = True) -> torch.Tensor:
    """pixel_values [B, C, H, W] -> hidden [B, N, D] fp64 (what psv_embed writes, before its fp32 storage)."""
    x = rnd(pixel_values, rounding)
    w = _w(sd, "embeddings.patch_embeddings.projection.weight", x, rounding)
    y = F.conv2d(x, w, _p(sd, "embeddings.patch_embeddings.projection.bias", x), stride=w.shape[-1])
    y = y.flatten(2).transpose(1, 2)
    cls = _p(sd, "embeddings.cls_token", x).expand(y.shape[0], -1, -1)
    return torch.cat((cls, y), dim=1) + _p(sd, "embeddings.position_embeddings", x)


# ----------------------------------------------------------------------------- attention
def attend(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, rounding: bool = True) -> torch.Tensor:
    """One image: q [H, nq, 64], k / v [H, nk, 64] (bf16 values) -> ctx [nq, H * 64].

    p = exp(s - max) with s = q k^T / 8; P = bf16(p); ctx = bf16(P v / sum p)."""
    s = torch.matmul(q, k.transpose(1, 2)) * SCALE
    e = torch.exp(s - s.amax(-1, keepdim=True))
    ctx = torch.matmul(rnd(e, rounding), v) / e.sum(-1, keepdim=True)
    return rnd(ctx.transpose(0, 1).reshape(q.shape[1], -1), rounding)


def _heads_view(t, heads):
    return t.reshape(t.shape[0], heads, -1).transpose(0, 1)


def attention(qkv: torch.Tensor, cu_seqlens, heads: int, rounding: bool = True, attend_fn=attend) -> torch.Tensor:
    """What psv_attention computes: qkv [T, 3D] packed rows of the images delimited by cu_seqlens -> ctx [T, D]."""
    D = qkv.shape[1] // 3
    cu = [int(c) for c in cu_seqlens]
    ctx = torch.zeros(qkv.shape[0], D, dtype=torch.float64, device=qkv.device)
    for b in range(len(cu) - 1):
        r0, r1 = cu[b], cu[b + 1]
        if r1 > r0:
            q, k, v = (_heads_view(qkv[r0:r1, j * D:(j + 1) * D].to(torch.float64), heads) for j in range(3))
            ctx[r0:r1] = attend_fn(q, k, v, rounding)
    return ctx


# ----------------------------------------------------------------------------- one skip layer
def layer(sd, l: int, h: torch.Tensor, mask: torch.Tensor, kv_all: bool = False, heads: int | None = None,
          rounding: bool = True, attend_fn=attend, gelu: str = "none") -> torch.Tensor:
    """psv_layer_forward with a forced mask: h [B, N, D] (fp32 or fp64), mask bool [B, N] -> out [B, N, D] fp64.

    Active rows get the ViT layer over the active tokens of their image (``kv_all``: over all N tokens as keys and
    values); skipped rows keep h.  ``attend_fn`` and ``gelu`` exist so that tests can plant defects."""
    p = f"encoder.layer.{l}."
    h = h.to(torch.float64)
    B, N, D = h.shape
    H = D // 64 if heads is None else heads
    mask = mask.to(h.device).bool()
    idx, cu, _ = compact(mask.cpu())
    idx = idx.long().to(h.device)
    flat = h.reshape(B * N, D)
    x = flat[idx]
    wqkv, bqkv = _qkv_weights(sd, p, h, rounding)
    if kv_all:
        qkv_all = rnd(F.linear(rnd(_ln(flat, sd, p + "layernorm_before"), rounding), wqkv, bqkv), rounding)
        ctx = torch.empty_like(x)
        cu_l = cu.tolist()
        for b in range(B):
            s0, s1 = cu_l[b], cu_l[b + 1]
            if s1 == s0:
                continue
            q = _heads_view(qkv_all[idx[s0:s1], :D], H)
            k, v = (_heads_view(qkv_all[b * N:(b + 1) * N, j * D:(j + 1) * D], H) for j in (1, 2))
            ctx[s0:s1] = attend_fn(q, k, v, rounding)
    else:
        qkv = rnd(F.linear(rnd(_ln(x, sd, p + "layernorm_before"), rounding), wqkv, bqkv), rounding)
        ctx = attention(qkv, cu, H, rounding, attend_fn)
    x1 = x + F.linear(ctx, _w(sd, p + "attention.output.dense.weight", h, rounding),
                      _p(sd, p + "attention.output.dense.bias", h))
    m = rnd(_ln(x1, sd, p + "layernorm_after"), rounding)
    u = F.linear(m, _w(sd, p + "intermediate.dense.weight", h, rounding), _p(sd, p + "intermediate.dense.bias", h))
    u = rnd(F.gelu(u, approximate=gelu), rounding)
    y = x1 + F.linear(u, _w(sd, p + "output.dense.weight", h, rounding), _p(sd, p + "output.dense.bias", h))
    out = flat.clone()
    out[idx] = y
    return out.view(B, N, D)


# ----------------------------------------------------------------------------- compressor decision, head, chain
def skip_mask(sd, l: int, h: torch.Tensor, mlp_threshold: float) -> torch.Tensor:
    """The compressor decision of layer l evaluated in fp64 on h: bool [B, N], CLS forced True (REF:62-68)."""
    p = f"encoder.layer.{l}.mlp_layer."
    h = h.to(torch.float64)
    z = torch.cat((h[:, :1].expand(-1, h.shape[1] - 1, -1), h[:, 1:]), -1)
    z = F.relu(F.linear(z, _p(sd, p + "0.weight", h), _p(sd, p + "0.bias", h)))
    s = torch.sigmoid(F.linear(z, _p(sd, p + "2.weight", h), _p(sd, p + "2.bias", h))).squeeze(-1)
    return torch.cat((torch.ones(h.shape[0], 1, dtype=torch.bool, device=h.device), s >= mlp_threshold), 1)


def head(sd, h: torch.Tensor) -> torch.Tensor:
    """final LayerNorm of the CLS row + classifier, fp64"""
    h = h.to(torch.float64)
    return F.linear(_ln(h[:, 0], sd, "layernorm"), _p(sd, "classifier.weight", h), _p(sd, "classifier.bias", h))


def forward(sd, pixel_values: torch.Tensor, mlp_threshold: float = 0.5, forced_masks: torch.Tensor | None = None,
            kv_all: bool = False, heads: int | None = None, rounding: bool = True, attend_fn=attend,
            gelu: str = "none"):
    """Whole model: returns (logits [B, C] fp64, masks bool [L, B, N]).  Without ``forced_masks`` each layer's mask
    is the fp64 compressor decision on this reference's own hidden state."""
    h = embed(sd, pixel_values, rounding)
    masks = []
    l = 0
    while f"encoder.layer.{l}.layernorm_before.weight" in sd:
        m = skip_mask(sd, l, h, mlp_threshold) if forced_masks is None else forced_masks[l].to(h.device).bool()
        h = layer(sd, l, h, m, kv_all, heads, rounding, attend_fn, gelu)
        masks.append(m)
        l += 1
    return head(sd, h), torch.stack(masks)
