"""Reference rule of the per-layer token budget (psv_set_token_budget, include/psv.h) and the fp32 oracle forward that
decides by it.

For one image with patch scores s_1..s_{N-1}:
    rank(t) = #{u : s_u > s_t, or s_u == s_t and u < t}
ties go to the lower token index; a NaN score ranks below every number and NaNs are ordered among themselves by index.
    exact: mask[t] = rank(t) < k                 cap: mask[t] = (s_t >= mt) and rank(t) < k
CLS (column 0 of the mask) is always kept and is not counted.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import vit_skip_oracle as O

MODES = ("exact", "cap")


def ranks(scores) -> np.ndarray:
    """int64 [..., N-1]: rank(t) of every patch, by the pairwise definition (O(N^2) per image)."""
    s = np.asarray(scores, dtype=np.float32)
    su, st = s[..., :, None], s[..., None, :]                     # [..., u, t]
    n = s.shape[-1]
    u_lt_t = np.arange(n)[:, None] < np.arange(n)[None, :]
    nan_u, nan_t = np.isnan(su), np.isnan(st)
    with np.errstate(invalid="ignore"):
        num = ~nan_u & ((su > st) | ((su == st) & u_lt_t))
    outranks = np.where(nan_t, ~nan_u | u_lt_t, num)
    return outranks.sum(axis=-2)


def budget_mask(scores, k: int, mode: str, mt: float = 0.5) -> np.ndarray:
    """bool [..., N] mask of the rule for scores [..., N-1] and one budget k."""
    if mode not in MODES:
        raise ValueError(mode)
    s = np.asarray(scores, dtype=np.float32)
    keep = ranks(s) < k
    if mode == "cap":
        with np.errstate(invalid="ignore"):
            keep &= s >= np.float32(mt)
    cls = np.ones(s.shape[:-1] + (1,), dtype=bool)
    return np.concatenate((cls, keep), axis=-1)


def budget_masks(scores, keep, mode: str, mt: float = 0.5) -> np.ndarray:
    """bool [L, B, N] for per-layer scores [L, B, N-1] and budgets keep [L]."""
    return np.stack([budget_mask(scores[l], int(keep[l]), mode, mt) for l in range(len(keep))])


def near_cut(scores, k: int, mode: str, mt: float = 0.5, band: float = 1e-4) -> np.ndarray:
    """bool [B]: images whose decision could flip under a score error below ``band``: the k-th and (k+1)-th highest
    scores lie within ``band`` of each other (and, for cap, some score lies within ``band`` of mt)."""
    s = np.asarray(scores, dtype=np.float64)
    srt = -np.sort(-s, axis=-1)
    near = np.zeros(s.shape[0], dtype=bool)
    if 0 < k < s.shape[-1]:
        near |= np.abs(srt[:, k - 1] - srt[:, k]) < band
    if mode == "cap":
        near |= (np.abs(s - mt) < band).any(-1)
    return near


def forward(sd, pixel_values: torch.Tensor, keep, mode: str, mlp_threshold: float = 0.5, kv_all: bool = False):
    """The oracle forward (vit_skip_oracle) with every layer deciding by the budget rule on its own fp32 scores.
    Returns (logits [B, C], masks bool [L, B, N], scores [L, B, N-1])."""
    h = O.embed(sd, pixel_values)
    masks, scores = [], []
    for l in range(O.num_layers(sd)):
        s = O.compressor_scores(sd, l, h)
        m = torch.from_numpy(budget_mask(s.numpy(), int(keep[l]), mode, mlp_threshold))
        h, _, _ = O.layer_forward(sd, l, h, mlp_threshold, forced_mask=m, kv_all=kv_all)
        masks.append(m)
        scores.append(s)
    return O.head(sd, h), torch.stack(masks), torch.stack(scores)
