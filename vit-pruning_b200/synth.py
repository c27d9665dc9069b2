"""Deterministic synthetic weights and inputs for the patch-skip ViT hot path.

There is no network on the build or the GPU box, so every measurement and every
parity test runs on random-init weights of the reference architecture and on
synthetic pixel batches (BASELINE.json: "synthetic CIFAR-100-shaped batch").

The generator is numpy PCG64 so the same bytes come out on every machine and do
not depend on torch's RNG consumption order.  The initialisation scheme mimics what
the reference's constructor produces (reference himanshu/model_utils.py:184-187 builds
the encoder/classifier/compressors *after* HF ``post_init`` so they keep torch's
default ``nn.Linear`` init, while the embeddings keep the HF trunc-normal init):

* embeddings (cls_token, position_embeddings, patch projection): N(0, 0.02) clipped
  to +-2 sigma, zero bias;
* every ``nn.Linear`` in the encoder, the classifier and the compressor
  (``mlp_layer.{0,2}``): weight and bias ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in));
* every LayerNorm: weight 1, bias 0;  pooler: N(0, 0.02), zero bias.

The state-dict keys/shapes are exactly the 250 tensors of the reference's
``ModifiedViTModel.state_dict()`` (SURVEY.md section 8b).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch


@dataclass(frozen=True)
class Geometry:
    """Architecture numbers of the path (ViT-B/16 by default)."""
    hidden: int = 768
    heads: int = 12
    ffn: int = 3072
    layers: int = 12
    classes: int = 100
    image: int = 224
    patch: int = 16
    channels: int = 3
    comp_hidden: int = 64      # reference model_utils.py:28  layer_sizes = [2*hidden, 64, 1]
    ln_eps: float = 1e-12

    @property
    def patches(self) -> int:
        return (self.image // self.patch) ** 2

    @property
    def tokens(self) -> int:
        return self.patches + 1


VIT_B16 = Geometry()
DEIT_S16 = Geometry(hidden=384, heads=6, ffn=1536)
VIT_L16 = Geometry(hidden=1024, heads=16, ffn=4096, layers=24)


def geometry_from_config(config) -> Geometry:
    """Build a Geometry from a transformers ViTConfig-like object."""
    return Geometry(hidden=config.hidden_size, heads=config.num_attention_heads,
                    ffn=config.intermediate_size, layers=config.num_hidden_layers,
                    classes=getattr(config, "num_labels", 2), image=config.image_size,
                    patch=config.patch_size, channels=config.num_channels,
                    ln_eps=config.layer_norm_eps)


def _uniform(rng, shape, bound):
    return torch.from_numpy(rng.uniform(-bound, bound, size=shape).astype(np.float32))


def _trunc_normal(rng, shape, std):
    a = rng.standard_normal(size=shape).astype(np.float32)
    np.clip(a, -2.0, 2.0, out=a)
    return torch.from_numpy(a * np.float32(std))


def make_state_dict(geom: Geometry = VIT_B16, seed: int = 42) -> dict[str, torch.Tensor]:
    """Random-init fp32 state dict with the reference's keys and shapes."""
    rng = np.random.Generator(np.random.PCG64(seed))
    D, F, C = geom.hidden, geom.ffn, geom.classes
    sd: dict[str, torch.Tensor] = {}

    def linear(prefix, out_f, in_f):
        b = 1.0 / math.sqrt(in_f)
        sd[prefix + ".weight"] = _uniform(rng, (out_f, in_f), b)
        sd[prefix + ".bias"] = _uniform(rng, (out_f,), b)

    def layernorm(prefix):
        sd[prefix + ".weight"] = torch.ones(D)
        sd[prefix + ".bias"] = torch.zeros(D)

    sd["embeddings.cls_token"] = _trunc_normal(rng, (1, 1, D), 0.02)
    sd["embeddings.position_embeddings"] = _trunc_normal(rng, (1, geom.tokens, D), 0.02)
    sd["embeddings.patch_embeddings.projection.weight"] = _trunc_normal(
        rng, (D, geom.channels, geom.patch, geom.patch), 0.02)
    sd["embeddings.patch_embeddings.projection.bias"] = torch.zeros(D)
    for i in range(geom.layers):
        p = f"encoder.layer.{i}."
        linear(p + "attention.attention.query", D, D)
        linear(p + "attention.attention.key", D, D)
        linear(p + "attention.attention.value", D, D)
        linear(p + "attention.output.dense", D, D)
        linear(p + "intermediate.dense", F, D)
        linear(p + "output.dense", D, F)
        layernorm(p + "layernorm_before")
        layernorm(p + "layernorm_after")
        linear(p + "mlp_layer.0", geom.comp_hidden, 2 * D)
        linear(p + "mlp_layer.2", 1, geom.comp_hidden)
    layernorm("layernorm")
    sd["pooler.dense.weight"] = _trunc_normal(rng, (D, D), 0.02)
    sd["pooler.dense.bias"] = torch.zeros(D)
    linear("classifier", C, D)
    return sd


def make_pixels(batch: int, geom: Geometry = VIT_B16, seed: int = 1234, kind: str = "randn") -> torch.Tensor:
    """Synthetic ``pixel_values`` [B, C, H, W] fp32.

    ``randn``  : standard normal (SURVEY.md 8d input (i)).
    ``cifar``  : CIFAR-shaped -- uniform [0,1) 32x32 images, bilinear x7 upsample to 224,
                 then (x-0.5)/0.5 as the HF processor the reference uses does
                 (reference himanshu/main_model_utils.py:54-60).
    """
    rng = np.random.Generator(np.random.PCG64(seed))
    if kind == "randn":
        a = rng.standard_normal(size=(batch, geom.channels, geom.image, geom.image)).astype(np.float32)
        return torch.from_numpy(a)
    if kind == "cifar":
        small = torch.from_numpy(rng.random(size=(batch, geom.channels, 32, 32)).astype(np.float32))
        up = torch.nn.functional.interpolate(small, size=(geom.image, geom.image), mode="bilinear",
                                             align_corners=False)
        return (up - 0.5) / 0.5
    raise ValueError(f"unknown synthetic input kind {kind!r}")


def algorithmic_flops_per_image(n_active, geom: Geometry = VIT_B16, kv_all: bool = False) -> float:
    """Skip-scaled algorithmic FLOPs per image (SURVEY.md 8d).

    ``n_active`` : array [L, B] of active tokens per layer per image, CLS included.
    Returns the batch mean of  sum_l [n*24*D^2 + n^2*4*D] + L*F_comp + F_embed + F_head.
    ``kv_all`` (query-only pruning): keys / values are projected for all N tokens and every active query attends
    to all of them: per layer n*20*D^2 + N*4*D^2 + n*N*4*D.
    """
    n = np.asarray(n_active, dtype=np.float64)
    D, L = geom.hidden, geom.layers
    if kv_all:
        per_layer = n * 20.0 * D * D + geom.tokens * 4.0 * D * D + n * geom.tokens * 4.0 * D
    else:
        per_layer = n * 24.0 * D * D + n * n * 4.0 * D
    f_comp = 2.0 * geom.patches * D * geom.comp_hidden + 2.0 * D * geom.comp_hidden + 2.0 * geom.patches * geom.comp_hidden
    f_embed = 2.0 * geom.patches * D * (geom.channels * geom.patch * geom.patch)
    f_head = 2.0 * D * geom.classes
    return float(per_layer.sum(axis=0).mean() + L * f_comp + f_embed + f_head)
