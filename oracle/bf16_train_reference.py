"""ORACLE -- test infrastructure, NOT product code.

Differentiable float64 reference of mixed-precision backbone fine-tuning (``PSV_TRAIN_BF16``): the training forward
rounds to bf16 at exactly the points ``oracle.bf16_reference`` lists (im2col pixels and GEMM weights, the LN1 / LN2
outputs, q|k|v after the bias, P and ctx, the GELU output), and nowhere else; the residual stream, LayerNorm and
softmax statistics, the compressor scores and the layers' compressor losses are exact.

Every rounding is straight-through, ``t + (bf16(t) - t).detach()``: its value is the bf16 value and its derivative is
the identity.  (``t.to(torch.bfloat16)`` would also round the float64 gradients flowing back through it.)  So autograd
through this forward gives the gradients the mixed-precision backward approximates, and with ``rounding=False`` it is
``reference_forward`` of the fp32 fine-tuning tests.

The layers are written in the dense masked form: LN1, q|k|v and the MLP run on all rows, keys of skipped tokens are
at -inf, and h = where(mask, layer(h), h).  For the active rows this is the computation of the packed form row by
row, so with rounding on the logits equal ``bf16_reference.forward(..., forced_masks=...)``.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.bf16_reference import SCALE
from oracle.vit_skip_oracle import LN_EPS


def rnd(t: torch.Tensor, rounding: bool = True) -> torch.Tensor:
    """straight-through bf16 rounding (RN-even): bf16 value, identity derivative"""
    if not rounding:
        return t
    return t + (t.to(torch.bfloat16).to(t.dtype) - t).detach()


def _ln(x, p, prefix):
    return F.layer_norm(x, (x.shape[-1],), p[prefix + ".weight"], p[prefix + ".bias"], LN_EPS)


def attend(q, k, v, rounding=True, key_mask=None, scale=SCALE):
    """q [..., nq, 64], k / v [..., nk, 64] -> ctx [..., nq, 64]: p = exp(s - max), P = bf16(p), ctx = bf16(P v / sum p)
    (as bf16_reference.attend); key_mask bool [..., 1, nk] (False = not a key)."""
    s = torch.matmul(q, k.transpose(-1, -2)) * scale
    if key_mask is not None:
        s = s.masked_fill(~key_mask, float("-inf"))
    e = torch.exp(s - s.amax(-1, keepdim=True).detach())
    return rnd(torch.matmul(rnd(e, rounding), v) / e.sum(-1, keepdim=True), rounding)


def forward(p, pixels, mt, heads, forced_masks=None, joint=False, rounding=True):
    """p: reference-keyed float64 parameters (requires_grad as wanted), pixels [B, 3, H, W] float64.  Returns (logits
    [B, C], masks bool [L, B, N], scores [L, B, N-1], layer losses [L] or None), as reference_forward does."""
    w = rnd(p["embeddings.patch_embeddings.projection.weight"], rounding)
    x = F.conv2d(rnd(pixels, rounding), w, p["embeddings.patch_embeddings.projection.bias"], stride=w.shape[-1])
    x = x.flatten(2).transpose(1, 2)
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
            m = forced_masks[l].to(h.device).bool()
        if joint:
            labels = m[:, 1:].to(s.dtype)
            mean = labels.mean()
            losses.append(F.binary_cross_entropy_with_logits(s, labels, pos_weight=(mean / (1 - mean + 1e-16)).reshape(1)))
        a = rnd(_ln(h, p, q_ + "layernorm_before"), rounding)
        q, k, v = (rnd(F.linear(a, rnd(p[q_ + f"attention.attention.{n}.weight"], rounding),
                                p[q_ + f"attention.attention.{n}.bias"]), rounding)
                   .view(B, N, heads, dh).transpose(1, 2) for n in ("query", "key", "value"))
        ctx = attend(q, k, v, rounding, m[:, None, None, :]).transpose(1, 2).reshape(B, N, D)
        x1 = F.linear(ctx, rnd(p[q_ + "attention.output.dense.weight"], rounding), p[q_ + "attention.output.dense.bias"]) + h
        u = F.linear(rnd(_ln(x1, p, q_ + "layernorm_after"), rounding), rnd(p[q_ + "intermediate.dense.weight"], rounding),
                     p[q_ + "intermediate.dense.bias"])
        u = rnd(F.gelu(u), rounding)
        y = F.linear(u, rnd(p[q_ + "output.dense.weight"], rounding), p[q_ + "output.dense.bias"]) + x1
        h = torch.where(m[..., None], y, h)
        masks.append(m)
        scores.append(s.detach())
    logits = F.linear(_ln(h[:, 0], p, "layernorm"), p["classifier.weight"], p["classifier.bias"])
    return logits, torch.stack(masks), torch.stack(scores), (torch.stack(losses) if joint else None)
