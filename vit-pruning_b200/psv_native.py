"""ctypes binding of the C ABI in include/psv.h (libpsv.so, built in-tree by csrc/Makefile).

There is deliberately no fallback: if the shared library is missing or cannot be loaded the
import raises, and if no CUDA device is present ``psv_create`` fails with PSV_ERR_CUDA.
torch is used only for device memory and the stream; all arithmetic is in libpsv.so.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PSV_LIB", os.path.join(_HERE, "libpsv.so"))

PSV_FP32, PSV_BF16 = 0, 1
PSV_PIXELS_F32, PSV_PIXELS_BF16, PSV_PIXELS_U8_HWC = 0, 1, 2

EXPORTS = [
    "psv_version", "psv_create", "psv_destroy", "psv_last_error", "psv_load_weights", "psv_embed",
    "psv_layer_forward", "psv_get_compaction", "psv_layer_stats", "psv_similarity_mask", "psv_head",
    "psv_forward", "psv_forward_host", "psv_forward_host_submit", "psv_forward_host_wait", "psv_compressor_grads", "psv_compressor_layer_grads",
    "psv_compressor_param_count", "psv_compressor_adam_step", "psv_get_compressor_params",
    "psv_set_compressor_params", "psv_last_launch_count", "psv_gemm", "psv_profile_begin", "psv_profile_end",
    "psv_attention", "psv_set_attention_kernel", "psv_set_u8_input", "psv_set_kv_mode",
    "psv_compressor_peer_reduce_adam_step", "psv_get_compressor_adam_state", "psv_set_compressor_adam_state",
    "psv_set_loss_variant", "psv_backbone_forward_train", "psv_backbone_backward", "psv_backbone_param_count",
    "psv_backbone_train_masks", "psv_set_skip_criterion", "psv_set_train_precision", "psv_attention_train_forward",
    "psv_attention_backward", "psv_backbone_adam_step", "psv_get_backbone_params", "psv_get_backbone_adam_state",
    "psv_set_backbone_adam_state", "psv_backbone_shard", "psv_backbone_peer_reduce_adam_step",
    "psv_backbone_peer_gather_params", "psv_backbone_adam_step_groups", "psv_backbone_peer_reduce_sqnorm",
    "psv_backbone_peer_adam_step_groups", "psv_compressor_adam_step_clipped",
    "psv_compressor_peer_reduce_adam_step_clipped", "psv_set_token_budget",
]


class PsvError(RuntimeError):
    pass


class PsvConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("hidden", "heads", "ffn", "layers", "tokens", "classes", "image",
                                         "patch", "channels", "comp_hidden", "precision", "max_batch")] + \
               [("ln_eps", C.c_float)]


_LAYER_FIELDS = ("ln1_w", "ln1_b", "q_w", "q_b", "k_w", "k_b", "v_w", "v_b", "o_w", "o_b", "ln2_w", "ln2_b",
                 "fc1_w", "fc1_b", "fc2_w", "fc2_b", "c1_w", "c1_b", "c2_w", "c2_b")


class PsvLayerWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _LAYER_FIELDS]


class PsvWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("cls_token", "pos_emb", "patch_w", "patch_b", "final_ln_w",
                                          "final_ln_b", "cls_w", "cls_b")] + \
               [("layers", C.POINTER(PsvLayerWeights))]


class PsvLayerStats(C.Structure):
    _fields_ = [("loss", C.c_void_p), ("similarity", C.c_void_p), ("accuracy", C.c_void_p),
                ("confusion", C.c_void_p)]


def _load():
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C vit-pruning_b200/csrc`). There is no CPU/PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    lib.psv_version.restype = C.c_char_p
    lib.psv_last_error.restype = C.c_char_p
    lib.psv_last_error.argtypes = [C.c_void_p]
    lib.psv_create.argtypes = [C.POINTER(PsvConfig), C.POINTER(C.c_void_p)]
    lib.psv_destroy.argtypes = [C.c_void_p]
    lib.psv_load_weights.argtypes = [C.c_void_p, C.POINTER(PsvWeights), C.c_void_p]
    lib.psv_embed.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.psv_layer_forward.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_float, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_get_compaction.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_layer_stats.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_float, C.POINTER(PsvLayerStats), C.c_void_p]
    lib.psv_similarity_mask.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_float, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
    lib.psv_head.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.psv_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.psv_forward_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                     C.c_void_p, C.c_void_p]
    lib.psv_forward_host_submit.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_float,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_forward_host_wait.argtypes = [C.c_void_p, C.c_int32]
    lib.psv_compressor_grads.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                         C.c_void_p, C.c_void_p]
    lib.psv_compressor_layer_grads.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                               C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
    lib.psv_compressor_param_count.restype = C.c_int64
    lib.psv_compressor_param_count.argtypes = [C.c_void_p]
    lib.psv_compressor_adam_step.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                             C.c_int32, C.c_float, C.c_void_p]
    lib.psv_get_compressor_params.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_set_compressor_params.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_get_compressor_adam_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_set_compressor_adam_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_last_launch_count.restype = C.c_int32
    lib.psv_last_launch_count.argtypes = [C.c_void_p]
    lib.psv_profile_begin.argtypes = [C.c_void_p]
    lib.psv_profile_end.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.psv_gemm.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                             C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.psv_set_attention_kernel.argtypes = [C.c_void_p, C.c_int32]
    lib.psv_set_kv_mode.argtypes = [C.c_void_p, C.c_int32]
    lib.psv_set_skip_criterion.argtypes = [C.c_void_p, C.c_int32, C.c_float]
    lib.psv_set_token_budget.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
    lib.psv_set_loss_variant.argtypes = [C.c_void_p, C.c_int32, C.c_float]
    lib.psv_backbone_forward_train.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                               C.c_void_p, C.c_void_p]
    lib.psv_backbone_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_backbone_param_count.argtypes = [C.c_void_p]
    lib.psv_backbone_param_count.restype = C.c_int64
    lib.psv_backbone_train_masks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_compressor_peer_reduce_adam_step.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_float,
                                                         C.c_float, C.c_float, C.c_float, C.c_int32, C.c_float,
                                                         C.c_void_p]
    lib.psv_set_u8_input.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_attention.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.psv_set_train_precision.argtypes = [C.c_void_p, C.c_int32]
    lib.psv_attention_train_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                                C.c_void_p, C.c_void_p]
    lib.psv_attention_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_backbone_adam_step.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_float, C.c_float,
                                           C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
    lib.psv_get_backbone_params.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_get_backbone_adam_state.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_set_backbone_adam_state.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_backbone_shard.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.psv_backbone_peer_reduce_adam_step.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_int32,
                                                       C.c_int32, C.POINTER(C.c_int32), C.c_float, C.c_float, C.c_float,
                                                       C.c_float, C.c_float, C.c_float, C.c_void_p]
    lib.psv_backbone_peer_gather_params.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_int32,
                                                    C.c_void_p]
    lib.psv_backbone_adam_step_groups.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_float),
                                                  C.POINTER(C.c_float), C.c_float, C.c_float, C.c_float, C.c_float,
                                                  C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.psv_backbone_peer_reduce_sqnorm.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_int32,
                                                    C.POINTER(C.c_int32), C.c_float, C.POINTER(C.c_void_p), C.c_void_p,
                                                    C.c_void_p]
    lib.psv_backbone_peer_adam_step_groups.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_int32,
                                                       C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_float),
                                                       C.POINTER(C.c_float), C.c_float, C.c_float, C.c_float, C.c_float,
                                                       C.c_float, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]
    lib.psv_compressor_adam_step_clipped.argtypes = lib.psv_compressor_adam_step.argtypes
    lib.psv_compressor_peer_reduce_adam_step_clipped.argtypes = lib.psv_compressor_peer_reduce_adam_step.argtypes
    return lib


lib = _load()


def backbone_shard(n, world, rank):
    """[lo, hi) of the flat backbone vector (n floats) that ``rank`` of ``world`` reduces and updates in the sharded
    peer-memory step: contiguous, bounds multiples of 4, the last rank takes the tail (psv_backbone_shard)."""
    lo, hi = C.c_int64(), C.c_int64()
    rc = lib.psv_backbone_shard(int(n), int(world), int(rank), C.byref(lo), C.byref(hi))
    if rc != 0:
        raise PsvError(f"psv_backbone_shard({n}, {world}, {rank}) failed ({rc})")
    return lo.value, hi.value


def _ptrs(addrs):
    """Host array of device addresses (ints or tensors); None stays None."""
    if addrs is None:
        return None
    return (C.c_void_p * len(addrs))(*[a.data_ptr() if isinstance(a, torch.Tensor) else int(a) for a in addrs])


def _ptr(t):
    if t is None:
        return None
    assert t.is_contiguous(), "psv needs contiguous tensors"
    return C.c_void_p(t.data_ptr())


def _stream(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    """One PsvHandle: geometry + precision + max_batch, bound to the current CUDA device."""

    def __init__(self, geom, precision: str = "fp32", max_batch: int = 64, device=None):
        if not torch.cuda.is_available():
            raise PsvError("psv needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.geom = geom
        self.precision = precision
        self.max_batch = int(max_batch)
        cfg = PsvConfig(hidden=geom.hidden, heads=geom.heads, ffn=geom.ffn, layers=geom.layers,
                        tokens=geom.tokens, classes=geom.classes, image=geom.image, patch=geom.patch,
                        channels=geom.channels, comp_hidden=geom.comp_hidden,
                        precision={"fp32": PSV_FP32, "bf16": PSV_BF16}[precision], max_batch=self.max_batch,
                        ln_eps=geom.ln_eps)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            rc = lib.psv_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise PsvError(f"psv_create failed ({rc}): {lib.psv_last_error(None).decode()}")
        self._weights_keepalive = None
        self.train_forwards = 0          # training forwards so far: each one replaces the state a pending backward reads
        self._train_batch = 0

    # -- plumbing
    def _check(self, rc, what):
        if rc != 0:
            raise PsvError(f"{what} failed ({rc}): {lib.psv_last_error(self._h).decode()}")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib.psv_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def last_launch_count(self) -> int:
        return int(lib.psv_last_launch_count(self._h))

    # -- weights
    def load_state_dict(self, sd):
        """sd: reference-keyed state dict (any device/dtype); cast to fp32 on this device."""
        g = self.geom
        dev = self.device

        def t(key):
            return sd[key].detach().to(device=dev, dtype=torch.float32).contiguous()

        keep = []

        def p(key):
            x = t(key)
            keep.append(x)
            return x.data_ptr()

        layers = (PsvLayerWeights * g.layers)()
        for i in range(g.layers):
            pre = f"encoder.layer.{i}."
            names = {
                "ln1_w": "layernorm_before.weight", "ln1_b": "layernorm_before.bias",
                "q_w": "attention.attention.query.weight", "q_b": "attention.attention.query.bias",
                "k_w": "attention.attention.key.weight", "k_b": "attention.attention.key.bias",
                "v_w": "attention.attention.value.weight", "v_b": "attention.attention.value.bias",
                "o_w": "attention.output.dense.weight", "o_b": "attention.output.dense.bias",
                "ln2_w": "layernorm_after.weight", "ln2_b": "layernorm_after.bias",
                "fc1_w": "intermediate.dense.weight", "fc1_b": "intermediate.dense.bias",
                "fc2_w": "output.dense.weight", "fc2_b": "output.dense.bias",
                "c1_w": "mlp_layer.0.weight", "c1_b": "mlp_layer.0.bias",
                "c2_w": "mlp_layer.2.weight", "c2_b": "mlp_layer.2.bias",
            }
            for f, k in names.items():
                setattr(layers[i], f, p(pre + k))
        w = PsvWeights(cls_token=p("embeddings.cls_token"), pos_emb=p("embeddings.position_embeddings"),
                       patch_w=p("embeddings.patch_embeddings.projection.weight"),
                       patch_b=p("embeddings.patch_embeddings.projection.bias"),
                       final_ln_w=p("layernorm.weight"), final_ln_b=p("layernorm.bias"),
                       cls_w=p("classifier.weight"), cls_b=p("classifier.bias"), layers=layers)
        with torch.cuda.device(dev):
            self._check(lib.psv_load_weights(self._h, C.byref(w), _stream(dev)), "psv_load_weights")
            torch.cuda.current_stream(dev).synchronize()     # sources may be freed after this
        del keep

    # -- hot path
    @staticmethod
    def _pixel_type(x):
        if x.dtype == torch.float32:
            return PSV_PIXELS_F32
        if x.dtype == torch.bfloat16:
            return PSV_PIXELS_BF16
        if x.dtype == torch.uint8:
            return PSV_PIXELS_U8_HWC                 # raw [B, H, W, 3] images, see set_u8_input
        raise PsvError(f"pixel_values dtype {x.dtype} not supported (float32, bfloat16 or uint8 HWC)")

    def embed(self, pixels):
        B = pixels.shape[0]
        hidden = torch.empty(B, self.geom.tokens, self.geom.hidden, device=self.device, dtype=torch.float32)
        self._check(lib.psv_embed(self._h, _ptr(pixels), self._pixel_type(pixels), B, _ptr(hidden),
                                  _stream(self.device)), "psv_embed")
        return hidden

    def layer_forward(self, layer, hidden, mt, forced_mask=None, want_mask=True, want_scores=True):
        """In place on ``hidden`` [B,N,D] fp32.  Returns (mask uint8 [B,N] | None, scores | None, n_active)."""
        B, N = hidden.shape[0], self.geom.tokens
        mask = torch.empty(B, N, device=self.device, dtype=torch.uint8) if want_mask else None
        scores = torch.empty(B, N - 1, device=self.device, dtype=torch.float32) if want_scores else None
        n_active = torch.empty(B, device=self.device, dtype=torch.int32)
        if forced_mask is not None:
            forced_mask = forced_mask.to(device=self.device, dtype=torch.uint8).contiguous()
        self._check(lib.psv_layer_forward(self._h, layer, _ptr(hidden), B, float(mt), _ptr(forced_mask), _ptr(mask),
                                          _ptr(scores), _ptr(n_active), _stream(self.device)), "psv_layer_forward")
        return mask, scores, n_active

    def get_compaction(self, batch):
        idx = torch.empty(batch * self.geom.tokens, device=self.device, dtype=torch.int32)
        cu = torch.empty(batch + 1, device=self.device, dtype=torch.int32)
        self._check(lib.psv_get_compaction(self._h, batch, _ptr(idx), _ptr(cu), _stream(self.device)),
                    "psv_get_compaction")
        return idx, cu

    def layer_stats(self, layer, hidden_in, mask, scores, st):
        B, N = hidden_in.shape[0], self.geom.tokens
        loss = torch.empty(1, device=self.device, dtype=torch.float32)
        sim = torch.empty(B, N - 1, device=self.device, dtype=torch.float32)
        acc = torch.empty(B, N - 1, device=self.device, dtype=torch.uint8)
        conf = torch.empty(2, 2, device=self.device, dtype=torch.int64)
        out = PsvLayerStats(loss=loss.data_ptr(), similarity=sim.data_ptr(), accuracy=acc.data_ptr(),
                            confusion=conf.data_ptr())
        self._check(lib.psv_layer_stats(self._h, layer, _ptr(hidden_in), B, _ptr(mask), _ptr(scores), float(st),
                                        C.byref(out), _stream(self.device)), "psv_layer_stats")
        return loss, sim, acc.bool(), conf

    def similarity_mask(self, layer, hidden_in, st):
        B, N = hidden_in.shape[0], self.geom.tokens
        mask = torch.empty(B, N, device=self.device, dtype=torch.uint8)
        sim = torch.empty(B, N - 1, device=self.device, dtype=torch.float32)
        self._check(lib.psv_similarity_mask(self._h, layer, _ptr(hidden_in), B, float(st), _ptr(mask), _ptr(sim),
                                            _stream(self.device)), "psv_similarity_mask")
        return mask, sim

    def head(self, hidden):
        B = hidden.shape[0]
        logits = torch.empty(B, self.geom.classes, device=self.device, dtype=torch.float32)
        self._check(lib.psv_head(self._h, _ptr(hidden), B, _ptr(logits), _stream(self.device)), "psv_head")
        return logits

    def forward(self, pixels, mt, forced_masks=None, want_masks=False, want_scores=False, want_n_active=False,
                use_graph=False, out=None):
        """Whole-model forward.  Returns dict(logits, masks, scores, n_active)."""
        g = self.geom
        B = pixels.shape[0]
        out = out or {}
        logits = out.get("logits")
        if logits is None:
            logits = torch.empty(B, g.classes, device=self.device, dtype=torch.float32)
        masks = out.get("masks")
        if masks is None and want_masks:
            masks = torch.empty(g.layers, B, g.tokens, device=self.device, dtype=torch.uint8)
        scores = out.get("scores")
        if scores is None and want_scores:
            scores = torch.empty(g.layers, B, g.tokens - 1, device=self.device, dtype=torch.float32)
        n_active = out.get("n_active")
        if n_active is None and want_n_active:
            n_active = torch.empty(g.layers, B, device=self.device, dtype=torch.int32)
        if forced_masks is not None:
            forced_masks = forced_masks.to(device=self.device, dtype=torch.uint8).contiguous()
        self._check(lib.psv_forward(self._h, _ptr(pixels), self._pixel_type(pixels), B, float(mt), _ptr(forced_masks),
                                    _ptr(logits), _ptr(masks), _ptr(scores), _ptr(n_active), int(use_graph),
                                    _stream(self.device)), "psv_forward")
        return {"logits": logits, "masks": masks, "scores": scores, "n_active": n_active,
                "_keep": (pixels, forced_masks)}

    def forward_host(self, host_pixels, mt, host_logits=None, host_n_active=None):
        """End-to-end: pinned host pixels in, host logits out (synchronises the stream)."""
        g = self.geom
        B = host_pixels.shape[0]
        assert host_pixels.device.type == "cpu"
        if host_logits is None:
            host_logits = torch.empty(B, g.classes, dtype=torch.float32).pin_memory()
        self._check(lib.psv_forward_host(self._h, _ptr(host_pixels), self._pixel_type(host_pixels), B, float(mt),
                                         _ptr(host_logits), _ptr(host_n_active), _stream(self.device)),
                    "psv_forward_host")
        return host_logits

    def forward_host_submit(self, slot, host_pixels, mt, host_logits, host_n_active=None):
        """Asynchronous end-to-end step (double-buffered): returns immediately; see forward_host_wait."""
        assert host_pixels.device.type == "cpu" and host_logits.device.type == "cpu"
        self._check(lib.psv_forward_host_submit(self._h, int(slot), _ptr(host_pixels), self._pixel_type(host_pixels),
                                                host_pixels.shape[0], float(mt), _ptr(host_logits),
                                                _ptr(host_n_active), _stream(self.device)), "psv_forward_host_submit")

    def forward_host_wait(self, slot):
        self._check(lib.psv_forward_host_wait(self._h, int(slot)), "psv_forward_host_wait")

    def gemm(self, a, w, bias=None, residual=None, out_fp32=True, gelu=False, accumulate_into=None, out=None):
        m, k = a.shape
        n = w.shape[0]
        if out is None:
            out = accumulate_into if accumulate_into is not None else \
                torch.empty(m, n, device=self.device, dtype=torch.float32 if out_fp32 else torch.bfloat16)
        self._check(lib.psv_gemm(self._h, _ptr(a), _ptr(w), _ptr(bias), _ptr(residual), _ptr(out), int(out_fp32),
                                 m, n, k, int(gelu), int(accumulate_into is not None), _stream(self.device)),
                    "psv_gemm")
        return out

    def set_u8_input(self, height, width, mean=None, std=None):
        """Accept raw uint8 [B, height, width, 3] images: Pillow-exact bilinear resize to the model size, 1/255
        rescale and (x - mean) / std (default 0.5 / 0.5, the ViT processor) are fused into the patch embedding."""
        key = (int(height), int(width), tuple(mean) if mean is not None else None,
               tuple(std) if std is not None else None)
        if getattr(self, "_u8_key", None) == key:          # unchanged: keep the captured graphs (the C side checks too)
            return
        m = (C.c_float * 3)(*mean) if mean is not None else None
        s = (C.c_float * 3)(*std) if std is not None else None
        self._check(lib.psv_set_u8_input(self._h, int(height), int(width), m, s, _stream(self.device)),
                    "psv_set_u8_input")
        self._u8_key = key

    ATTENTION_KERNELS = {"auto": 0, "mma": 1, "tc": 2, "pk": 3}

    def set_attention_kernel(self, kind: str):
        """'auto' (per-layer choice by sequence length), 'mma' (warp-level mma.sync) or 'tc' (tcgen05/TMEM)."""
        self._check(lib.psv_set_attention_kernel(self._h, self.ATTENTION_KERNELS[kind]), "psv_set_attention_kernel")

    # -- backbone fine-tuning (fp32 engines)
    def backbone_forward_train(self, pixels, mt, with_layer_losses=False):
        """fp32 patch-skip forward that keeps what the backward needs; returns logits [B, C], or (logits, the L layers'
        compressor losses) for the joint objective of loss_type "both".  ``pixels``: fp32 pixel_values or raw uint8
        [B, H, W, 3] images (after set_u8_input).  Runs in the engine's kv mode (set_kv_mode) and skip criterion
        (set_skip_criterion); the matching backbone_backward follows the mode and the uint8 setup of this forward."""
        B = pixels.shape[0]
        logits = torch.empty(B, self.geom.classes, device=self.device, dtype=torch.float32)
        losses = torch.empty(self.geom.layers, device=self.device, dtype=torch.float32) if with_layer_losses else None
        self._check(lib.psv_backbone_forward_train(self._h, _ptr(pixels), self._pixel_type(pixels), B, float(mt),
                                                   _ptr(logits), _ptr(losses) if with_layer_losses else None,
                                                   _stream(self.device)), "psv_backbone_forward_train")
        self._train_pixels = pixels                  # must outlive the backward
        self._train_batch = B
        self.train_forwards += 1
        return (logits, losses) if with_layer_losses else logits

    def backbone_backward(self, dlogits, dlosses=None, out=None, comp_out=None):
        """d loss / d logits -> flat fp32 gradient of every backbone parameter (layout: backbone_grad_slices); with
        dlosses [L] (upstream gradients of the layer losses) -> (backbone gradient, flat compressor gradient).
        Differentiates the LAST backbone_forward_train; other calls on the engine in between do not disturb it.
        ``out`` / ``comp_out``: flat fp32 buffers to write into (e.g. symmetric-memory buckets peers can read)."""
        if tuple(dlogits.shape) != (self._train_batch, self.geom.classes):
            raise PsvError(f"dlogits has shape {tuple(dlogits.shape)}, the last training forward produced "
                           f"({self._train_batch}, {self.geom.classes})")
        n = self.backbone_param_count
        grads = out if out is not None else torch.empty(n, device=self.device, dtype=torch.float32)
        assert grads.numel() == n and grads.dtype == torch.float32 and grads.is_contiguous()
        dlogits = dlogits.to(device=self.device, dtype=torch.float32).contiguous()
        if dlosses is None:
            self._check(lib.psv_backbone_backward(self._h, _ptr(dlogits), None, _ptr(grads), None, _stream(self.device)),
                        "psv_backbone_backward")
            return grads
        dlosses = dlosses.to(device=self.device, dtype=torch.float32).contiguous()
        cgrads = comp_out if comp_out is not None else \
            torch.empty(self.compressor_param_count, device=self.device, dtype=torch.float32)
        assert cgrads.numel() == self.compressor_param_count and cgrads.dtype == torch.float32
        self._check(lib.psv_backbone_backward(self._h, _ptr(dlogits), _ptr(dlosses), _ptr(grads), _ptr(cgrads),
                                              _stream(self.device)), "psv_backbone_backward")
        return grads, cgrads

    def backbone_train_masks(self):
        """The skip masks the last backbone_forward_train decided: uint8 [L, B, N], 1 = processed (test hook)."""
        g = self.geom
        masks = torch.empty(g.layers, self._train_batch, g.tokens, device=self.device, dtype=torch.uint8)
        self._check(lib.psv_backbone_train_masks(self._h, _ptr(masks), _stream(self.device)), "psv_backbone_train_masks")
        return masks

    def backbone_grad_slices(self):
        """reference state-dict key -> (offset, shape) into the flat gradient of backbone_backward."""
        g = self.geom
        D, F, N, C, KP = g.hidden, g.ffn, g.tokens, g.classes, g.channels * g.patch * g.patch
        out, o = {}, 0

        def take(key, *shape):
            nonlocal o
            n = 1
            for d in shape:
                n *= d
            out[key] = (o, shape)
            o += n
        take("embeddings.cls_token", 1, 1, D)
        take("embeddings.position_embeddings", 1, N, D)
        take("embeddings.patch_embeddings.projection.weight", D, g.channels, g.patch, g.patch)
        take("embeddings.patch_embeddings.projection.bias", D)
        for i in range(g.layers):
            p = f"encoder.layer.{i}."
            take(p + "layernorm_before.weight", D); take(p + "layernorm_before.bias", D)
            take(p + "attention.attention.query.weight", D, D); take(p + "attention.attention.key.weight", D, D)
            take(p + "attention.attention.value.weight", D, D)
            take(p + "attention.attention.query.bias", D); take(p + "attention.attention.key.bias", D)
            take(p + "attention.attention.value.bias", D)
            take(p + "attention.output.dense.weight", D, D); take(p + "attention.output.dense.bias", D)
            take(p + "layernorm_after.weight", D); take(p + "layernorm_after.bias", D)
            take(p + "intermediate.dense.weight", F, D); take(p + "intermediate.dense.bias", F)
            take(p + "output.dense.weight", D, F); take(p + "output.dense.bias", D)
        take("layernorm.weight", D); take("layernorm.bias", D)
        take("classifier.weight", C, D); take("classifier.bias", C)
        assert o == int(lib.psv_backbone_param_count(self._h))
        return out

    # -- backbone optimizer (fp32 engines): Adam / AdamW on the handle's own weights
    @property
    def backbone_param_count(self) -> int:
        return int(lib.psv_backbone_param_count(self._h))

    def _steps(self, steps):
        steps = [int(s) for s in steps]
        n = 8 + 16 * self.geom.layers
        if len(steps) != n:
            raise PsvError(f"steps has {len(steps)} entries, the backbone has {n} tensors")
        return (C.c_int32 * n)(*steps)

    def backbone_adam_step(self, grads, steps, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                           grad_scale=1.0):
        """torch.optim.AdamW (weight_decay = 0: Adam) on the engine's backbone weights from a flat gradient (layout:
        backbone_grad_slices).  ``steps``: one 1-based Adam step per backbone tensor in that order, 0 = frozen."""
        assert grads.numel() == self.backbone_param_count and grads.dtype == torch.float32
        self._check(lib.psv_backbone_adam_step(self._h, _ptr(grads), self._steps(steps), float(lr), float(betas[0]),
                                               float(betas[1]), float(eps), float(weight_decay), float(grad_scale),
                                               _stream(self.device)), "psv_backbone_adam_step")

    def backbone_peer_reduce_adam_step(self, peer_grads, param_bucket, rank, steps, lr=1e-3, betas=(0.9, 0.999),
                                       eps=1e-8, weight_decay=0.0, grad_scale=1.0):
        """Sharded data-parallel step over NVLink peer memory: ``peer_grads[r]`` = device address of rank r's gradient
        bucket (own rank included); this rank sums its shard (backbone_shard) in rank order, updates it and publishes
        the new values in ``param_bucket`` (an address or a tensor).  Between cross-rank barriers (see psv.h)."""
        arr = (C.c_void_p * len(peer_grads))(*[int(p) for p in peer_grads])
        bucket = param_bucket.data_ptr() if isinstance(param_bucket, torch.Tensor) else int(param_bucket)
        self._check(lib.psv_backbone_peer_reduce_adam_step(
            self._h, arr, C.c_void_p(bucket), len(peer_grads), int(rank), self._steps(steps), float(lr),
            float(betas[0]), float(betas[1]), float(eps), float(weight_decay), float(grad_scale), _stream(self.device)),
            "psv_backbone_peer_reduce_adam_step")

    def _per_tensor(self, value, what):
        """A scalar, a per-tensor list (flat-layout order) or a per-key dict -> host float array, one entry per tensor."""
        keys = list(self.backbone_grad_slices())
        if isinstance(value, dict):
            unknown = set(value) - set(keys)
            if unknown or len(value) != len(keys):
                raise PsvError(f"{what}: needs exactly the backbone keys ({len(keys)}); unknown {sorted(unknown)[:4]}")
            value = [value[k] for k in keys]
        elif not isinstance(value, (list, tuple)):
            value = [value] * len(keys)
        if len(value) != len(keys):
            raise PsvError(f"{what} has {len(value)} entries, the backbone has {len(keys)} tensors")
        return (C.c_float * len(keys))(*[float(x) for x in value])

    @staticmethod
    def _clip(max_grad_norm):
        return 0.0 if max_grad_norm is None else float(max_grad_norm)

    def backbone_adam_step_groups(self, grads, steps, lr, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8,
                                  grad_scale=1.0, max_grad_norm=None, comp_grads=None, grad_norm_out=None):
        """backbone_adam_step with parameter groups and global-norm clipping (psv_backbone_adam_step_groups).
        ``lr`` / ``weight_decay``: a scalar, a per-tensor list or a per-key dict.  ``max_grad_norm``: clip as
        torch.nn.utils.clip_grad_norm_ (None: no clipping).  ``comp_grads``: the compressor gradient, counted in the norm
        (then compressor_adam_step(..., clipped=True)).  ``grad_norm_out``: float64 device tensor [1] for the norm."""
        assert grads.numel() == self.backbone_param_count and grads.dtype == torch.float32
        assert grad_norm_out is None or (grad_norm_out.dtype == torch.float64 and grad_norm_out.is_cuda)
        self._check(lib.psv_backbone_adam_step_groups(
            self._h, _ptr(grads), self._steps(steps), self._per_tensor(lr, "lr"),
            self._per_tensor(weight_decay, "weight_decay"), float(betas[0]), float(betas[1]), float(eps),
            float(grad_scale), self._clip(max_grad_norm), _ptr(comp_grads), _ptr(grad_norm_out),
            _stream(self.device)), "psv_backbone_adam_step_groups")

    def backbone_peer_reduce_sqnorm(self, peer_grads, rank, steps, sqnorm_slot, grad_scale=1.0, comp_peer_grads=None):
        """First pass of the clipped sharded step (see psv.h): sums this rank's shard of the peers' gradient buckets in
        rank order into its own bucket and writes its fp64 partial sum of squares into ``sqnorm_slot`` (a float64
        device tensor or an address in symmetric memory).  Between barriers B0 and B1."""
        slot = sqnorm_slot.data_ptr() if isinstance(sqnorm_slot, torch.Tensor) else int(sqnorm_slot)
        self._check(lib.psv_backbone_peer_reduce_sqnorm(
            self._h, _ptrs(peer_grads), len(peer_grads), int(rank), self._steps(steps), float(grad_scale),
            _ptrs(comp_peer_grads), C.c_void_p(slot), _stream(self.device)), "psv_backbone_peer_reduce_sqnorm")

    def backbone_peer_adam_step_groups(self, peer_grads, param_bucket, rank, steps, lr, weight_decay=0.0,
                                       betas=(0.9, 0.999), eps=1e-8, grad_scale=1.0, max_grad_norm=None,
                                       peer_sqnorms=None, grad_norm_out=None):
        """Sharded update with parameter groups.  Without ``peer_sqnorms``: the fused reduce + update pass (no clipping).
        With them (every rank's sqnorm slot, after backbone_peer_reduce_sqnorm and barrier B1): the norm from the
        partials in rank order, then the (clipped) update of the reduced shard."""
        bucket = param_bucket.data_ptr() if isinstance(param_bucket, torch.Tensor) else int(param_bucket)
        self._check(lib.psv_backbone_peer_adam_step_groups(
            self._h, _ptrs(peer_grads), C.c_void_p(bucket), len(peer_grads), int(rank), self._steps(steps),
            self._per_tensor(lr, "lr"), self._per_tensor(weight_decay, "weight_decay"), float(betas[0]),
            float(betas[1]), float(eps), float(grad_scale), self._clip(max_grad_norm), _ptrs(peer_sqnorms),
            _ptr(grad_norm_out), _stream(self.device)), "psv_backbone_peer_adam_step_groups")

    def backbone_peer_gather_params(self, peer_params, rank):
        """Copies every other rank's updated shard out of its parameter bucket (``peer_params[r]``) into the weights."""
        arr = (C.c_void_p * len(peer_params))(*[int(p) for p in peer_params])
        self._check(lib.psv_backbone_peer_gather_params(self._h, arr, len(peer_params), int(rank), _stream(self.device)),
                    "psv_backbone_peer_gather_params")

    def get_backbone_params(self):
        """The engine's current backbone weights, flat (layout: backbone_grad_slices)."""
        p = torch.empty(self.backbone_param_count, device=self.device, dtype=torch.float32)
        self._check(lib.psv_get_backbone_params(self._h, _ptr(p), _stream(self.device)), "psv_get_backbone_params")
        return p

    def get_backbone_adam_state(self, lo=0, hi=None):
        """(m, v) of the native backbone optimizer for flat positions [lo, hi) (zeros before the first step)."""
        hi = self.backbone_param_count if hi is None else int(hi)
        m = torch.empty(hi - lo, device=self.device, dtype=torch.float32)
        v = torch.empty_like(m)
        self._check(lib.psv_get_backbone_adam_state(self._h, int(lo), hi - lo, _ptr(m), _ptr(v), _stream(self.device)),
                    "psv_get_backbone_adam_state")
        return m, v

    def set_backbone_adam_state(self, m, v, lo=0):
        m = m.to(device=self.device, dtype=torch.float32).contiguous()
        v = v.to(device=self.device, dtype=torch.float32).contiguous()
        assert m.numel() == v.numel()
        self._check(lib.psv_set_backbone_adam_state(self._h, int(lo), m.numel(), _ptr(m), _ptr(v), _stream(self.device)),
                    "psv_set_backbone_adam_state")

    def export_backbone_state_dict(self, into=None):
        """The engine's CURRENT backbone weights (e.g. after native optimizer steps) as reference-keyed tensors.
        ``into``: an nn.Module (or a state dict) whose matching entries are overwritten in place."""
        flat = self.get_backbone_params()
        out = {}
        for k, (off, shape) in self.backbone_grad_slices().items():
            n = 1
            for d in shape:
                n *= d
            out[k] = flat[off:off + n].reshape(shape).clone()
        if into is not None:
            target = into.state_dict() if hasattr(into, "state_dict") else into
            with torch.no_grad():
                for k, v in out.items():
                    target[k].copy_(v.reshape(target[k].shape).to(target[k].dtype))
        return out

    LOSS_VARIANTS = {"himanshu": 0, "donal": 1}

    def set_loss_variant(self, variant: str, sim_threshold=0.9):
        """'himanshu' (default; reference himanshu/model_utils.py:95-113: labels = the layer's own mask, pos_weight from
        the label mean, similarity blend 0.3) or 'donal' (donal/model_utils.py:68-80: labels = similarity < st, fixed
        pos_weight 1.5, blend 0.5)."""
        self._check(lib.psv_set_loss_variant(self._h, self.LOSS_VARIANTS[variant], float(sim_threshold)),
                    "psv_set_loss_variant")

    KV_MODES = {"active": 0, "all": 1}

    def set_kv_mode(self, mode: str):
        """'active' (reference himanshu/model_utils.py:88-91: attention among the active tokens) or 'all'
        (query-only pruning, reference recap/convprad4.py:99-125: skipped tokens still serve as keys / values).  Inference,
        backbone fine-tuning and compressor_grads all follow it."""
        self._check(lib.psv_set_kv_mode(self._h, self.KV_MODES[mode]), "psv_set_kv_mode")

    SKIP_CRITERIA = {"mlp": 0, "similarity": 1}

    def set_skip_criterion(self, name: str, sim_threshold=0.9):
        """'mlp' (default; reference himanshu/model_utils.py:62-68: compressor score >= mt) or 'similarity' (reference
        pradeep/model_utils.py:73-84: dense pass of each layer, mask = [1, sim < sim_threshold]).  forward, forward_host*
        and backbone_forward_train follow it; layer_forward / layer_stats / similarity_mask do not, and compressor_grads
        raises under 'similarity'."""
        self._check(lib.psv_set_skip_criterion(self._h, self.SKIP_CRITERIA[name], float(sim_threshold)),
                    "psv_set_skip_criterion")

    BUDGET_MODES = {"off": 0, "exact": 1, "cap": 2}

    def set_token_budget(self, keep, mode: str = "exact"):
        """Per-layer token budget on the compressor decision (psv_set_token_budget): layer l keeps the keep[l]
        highest-scoring patches of every image ('exact'; the threshold is ignored) or at most keep[l] of those that pass
        the threshold ('cap'); ties go to the lower token index.  ``keep``: one int for every layer, or a list of
        ``layers`` ints in [0, tokens - 1]; None (or mode 'off') clears the budget.  forward, forward_host*,
        layer_forward and backbone_forward_train follow it; compressor_grads raises while it is set."""
        if keep is None or mode == "off":
            self._check(lib.psv_set_token_budget(self._h, 0, None), "psv_set_token_budget")
            return
        L = self.geom.layers
        ks = [int(keep)] * L if isinstance(keep, int) else [int(k) for k in keep]
        if len(ks) != L:
            raise PsvError(f"keep has {len(ks)} entries, the model has {L} layers")
        arr = (C.c_int32 * L)(*ks)
        self._check(lib.psv_set_token_budget(self._h, self.BUDGET_MODES[mode], arr), "psv_set_token_budget")

    def attention(self, qkv, cu_seqlens, out=None):
        """softmax(q k^T / 8) v per image and head on the packed [T, 3D] activations (test hook)."""
        total, width = qkv.shape
        ctx = out if out is not None else torch.zeros(total, width // 3, device=self.device, dtype=qkv.dtype)
        self._check(lib.psv_attention(self._h, _ptr(qkv), _ptr(cu_seqlens), cu_seqlens.numel() - 1, total,
                                      _ptr(ctx), _stream(self.device)), "psv_attention")
        return ctx

    TRAIN_PRECISIONS = {"split": 0, "bf16": 1}

    def set_train_precision(self, mode: str):
        """Arithmetic of backbone fine-tuning (fp32 engines): 'split' (default; split-bf16 GEMMs, fp32-exact, matches
        fp32 autograd to ~1e-4) or 'bf16' (mixed precision: bf16 operands rounded where the bf16 inference path rounds,
        one tensor-core pass per GEMM, fp32 accumulation, residual stream and statistics).  backbone_forward_train
        records it; the matching backbone_backward follows the recorded mode."""
        self._check(lib.psv_set_train_precision(self._h, self.TRAIN_PRECISIONS[mode]), "psv_set_train_precision")

    def attention_train_forward(self, qkv, cu_seqlens):
        """Mixed-precision training attention (engine in set_train_precision('bf16'); test hook): qkv bf16 [T, 3D] ->
        (ctx bf16 [T, D], lse fp32 [T, H]) with lse = logsumexp(q k^T / 8) per row and head."""
        total, width = qkv.shape
        ctx = torch.zeros(total, width // 3, device=self.device, dtype=torch.bfloat16)
        lse = torch.zeros(total, self.geom.heads, device=self.device, dtype=torch.float32)
        self._check(lib.psv_attention_train_forward(self._h, _ptr(qkv), _ptr(cu_seqlens), cu_seqlens.numel() - 1, total,
                                                    _ptr(ctx), _ptr(lse), _stream(self.device)),
                    "psv_attention_train_forward")
        return ctx, lse

    def attention_backward(self, qkv, cu_seqlens, ctx, lse, dctx):
        """Its backward (test hook): dctx fp32 [T, D] -> dqkv fp32 [T, 3D]."""
        total, width = qkv.shape
        dqkv = torch.zeros(total, width, device=self.device, dtype=torch.float32)
        dctx = dctx.to(device=self.device, dtype=torch.float32).contiguous()
        self._check(lib.psv_attention_backward(self._h, _ptr(qkv), _ptr(cu_seqlens), cu_seqlens.numel() - 1, total,
                                               _ptr(ctx), _ptr(lse), _ptr(dctx), _ptr(dqkv), _stream(self.device)),
                    "psv_attention_backward")
        return dqkv

    # -- profiling (bench roofline leg)
    KERNEL_KINDS = ("score_mask", "compact_gather_ln", "gemm", "attention", "layernorm", "im2col", "cls_rows",
                    "head", "similarity", "label_stats", "train", "other", "cls_half", "budget_mask")

    def profile_begin(self):
        self._check(lib.psv_profile_begin(self._h), "psv_profile_begin")

    def profile_end(self, capacity=4096):
        kinds = (C.c_int32 * capacity)()
        ms = (C.c_float * capacity)()
        count = C.c_int32(0)
        self._check(lib.psv_profile_end(self._h, kinds, ms, capacity, C.byref(count)), "psv_profile_end")
        n = min(count.value, capacity)
        return [(self.KERNEL_KINDS[kinds[i]], float(ms[i])) for i in range(n)]

    # -- compressor training
    @property
    def compressor_param_count(self) -> int:
        return int(lib.psv_compressor_param_count(self._h))

    def compressor_layer_grads(self, layer, hidden_in, mask, scores, grad_scale=1.0):
        per = self.compressor_param_count // self.geom.layers
        grads = torch.empty(per, device=self.device, dtype=torch.float32)
        self._check(lib.psv_compressor_layer_grads(self._h, layer, _ptr(hidden_in), hidden_in.shape[0], _ptr(mask),
                                                   _ptr(scores), float(grad_scale), _ptr(grads),
                                                   _stream(self.device)), "psv_compressor_layer_grads")
        return grads

    def compressor_grads(self, pixels, mt, out=None):
        """Per-layer compressor losses and their gradients in one skip-mode forward, in the engine's kv mode.
        ``out``: flat fp32 gradient bucket to write into (e.g. a symmetric-memory tensor peers can read)."""
        grads = out if out is not None else torch.empty(self.compressor_param_count, device=self.device,
                                                        dtype=torch.float32)
        assert grads.numel() == self.compressor_param_count and grads.dtype == torch.float32
        loss = torch.empty(self.geom.layers, device=self.device, dtype=torch.float32)
        self._check(lib.psv_compressor_grads(self._h, _ptr(pixels), self._pixel_type(pixels), pixels.shape[0],
                                             float(mt), _ptr(grads), _ptr(loss), _stream(self.device)),
                    "psv_compressor_grads")
        return grads, loss

    def compressor_adam_step(self, grads, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, step=1, grad_scale=1.0,
                             clipped=False):
        """``clipped``: also scale by the clip coefficient of the last clipped backbone step whose norm covered the
        compressor gradient (psv_compressor_adam_step_clipped)."""
        fn = lib.psv_compressor_adam_step_clipped if clipped else lib.psv_compressor_adam_step
        self._check(fn(self._h, _ptr(grads), lr, beta1, beta2, eps, step, grad_scale, _stream(self.device)),
                    "psv_compressor_adam_step" + ("_clipped" if clipped else ""))

    def compressor_peer_reduce_adam_step(self, peer_ptrs, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, step=1,
                                         grad_scale=1.0, clipped=False):
        """All-reduce over NVLink peer memory fused with Adam: ``peer_ptrs[r]`` = device address of rank r's gradient
        bucket mapped into this process (own rank included).  The caller brackets the call with cross-rank barriers.
        ``clipped``: as in compressor_adam_step."""
        arr = (C.c_void_p * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        fn = lib.psv_compressor_peer_reduce_adam_step_clipped if clipped else lib.psv_compressor_peer_reduce_adam_step
        self._check(fn(self._h, arr, len(peer_ptrs), lr, beta1, beta2, eps, step, grad_scale, _stream(self.device)),
                    "psv_compressor_peer_reduce_adam_step" + ("_clipped" if clipped else ""))

    def get_compressor_params(self):
        p = torch.empty(self.compressor_param_count, device=self.device, dtype=torch.float32)
        self._check(lib.psv_get_compressor_params(self._h, _ptr(p), _stream(self.device)),
                    "psv_get_compressor_params")
        return p

    def set_compressor_params(self, params):
        self._check(lib.psv_set_compressor_params(self._h, _ptr(params), _stream(self.device)),
                    "psv_set_compressor_params")

    def get_compressor_adam_state(self):
        """(m, v): the native optimizer's moments, flat layout of the parameters (zeros before the first step)."""
        m = torch.empty(self.compressor_param_count, device=self.device, dtype=torch.float32)
        v = torch.empty_like(m)
        self._check(lib.psv_get_compressor_adam_state(self._h, _ptr(m), _ptr(v), _stream(self.device)),
                    "psv_get_compressor_adam_state")
        return m, v

    def set_compressor_adam_state(self, m, v):
        m = m.to(device=self.device, dtype=torch.float32).contiguous()
        v = v.to(device=self.device, dtype=torch.float32).contiguous()
        assert m.numel() == v.numel() == self.compressor_param_count
        self._check(lib.psv_set_compressor_adam_state(self._h, _ptr(m), _ptr(v), _stream(self.device)),
                    "psv_set_compressor_adam_state")

    def export_compressor_state_dict(self, into=None):
        """The handle's CURRENT compressor parameters (e.g. after native training steps) as reference-keyed tensors
        ``encoder.layer.{i}.mlp_layer.{0,2}.{weight,bias}`` (himanshu/model_utils.py:28-37).  ``into``: an nn.Module
        (or a state dict) whose matching entries are overwritten in place, so ``torch.save(model.state_dict())`` -- the
        reference's checkpoint, main_model_utils.py:181-183 -- saves what was trained."""
        g = self.geom
        flat = self.get_compressor_params()
        ch, D = g.comp_hidden, g.hidden
        per = ch * 2 * D + 2 * ch + 1
        stride = (per + 3) // 4 * 4
        out = {}
        for i in range(g.layers):
            blk = flat[i * stride:i * stride + per]
            pre = f"encoder.layer.{i}.mlp_layer."
            out[pre + "0.weight"] = blk[:ch * 2 * D].reshape(ch, 2 * D).clone()
            out[pre + "0.bias"] = blk[ch * 2 * D:ch * 2 * D + ch].clone()
            out[pre + "2.weight"] = blk[ch * 2 * D + ch:ch * 2 * D + 2 * ch].reshape(1, ch).clone()
            out[pre + "2.bias"] = blk[ch * 2 * D + 2 * ch:per].clone()
        if into is not None:
            target = into.state_dict() if hasattr(into, "state_dict") else into
            with torch.no_grad():
                for k, v in out.items():
                    target[k].copy_(v.to(target[k].dtype))
        return out
