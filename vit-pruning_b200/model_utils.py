"""Drop-in for the reference's ``himanshu/model_utils.py`` backed by the B200 C-ABI library.

Same module name, class names, constructor and forward signatures, output object and
``state_dict`` keys as the reference (reference himanshu/model_utils.py:19-300), so
``hi_main.py`` / ``main_model_utils.py`` / ``donal/*.py`` style callers run unchanged:

    model = ModifiedViTModel(config, sim_threshold, mlp_threshold, avg_threshold)
    model.load_state_dict(...); model.to("cuda")
    out = model(pixel_values, compute_cosine=True)       # out.logits, out.boolean_masks
    model.encoder.layer[i].loss / .mlp_accuracy_arr / .mlp_confusion_matrix

The modules only hold parameters (so checkpoints of the reference and HF weights load with
the reference's own key renaming, hi_main.py:130-137).  ALL arithmetic of the forward happens
in libpsv.so (hand-written sm_100a kernels); there is no PyTorch fallback: calling the model
with CPU tensors or without the built library raises.

Deliberate differences from the reference, all to resolve defects listed in SURVEY.md 8b:
* ``output_mask=True`` works (the reference raises at model_utils.py:47) and returns the tuple
  of per-layer ``bool [B, 197]`` masks, as donal/model_utils.py:86-89,136-137 does;
* ``avg_threshold`` is accepted and stored but the neighbour-average pre-step (dead code in
  the reference, model_utils.py:47-51) is not implemented;
* ``head_mask`` / ``output_attentions`` / ``return_dict=False`` / ``bool_masked_pos`` /
  ``interpolate_pos_encoding`` are accepted and ignored or rejected (inert or broken upstream).

Precision: ``model.psv_precision`` is ``"fp32"`` (default for fp32 parameters; the 1e-4 parity
mode) or ``"bf16"`` (tcgen05 tensor cores; default when the parameters are bfloat16, i.e.
after ``model.to(torch.bfloat16)``).  Environment variable PSV_PRECISION overrides the default.
"""
from __future__ import annotations

import numbers
import os
from typing import Optional

import torch
from torch import nn
from transformers.modeling_outputs import BaseModelOutput
from transformers.models.vit.modeling_vit import ViTConfig, ViTEncoder, ViTLayer, ViTModel

import psv_native
from synth import geometry_from_config


class _CompressorLoss(torch.autograd.Function):
    """loss_l as a differentiable function of layer l's compressor parameters.

    forward : the loss value the C-ABI computed (model_utils.py:103-108 of the reference);
    backward: psv_compressor_layer_grads on the saved layer input / mask / scores.
    """

    @staticmethod
    def forward(ctx, c1_w, c1_b, c2_w, c2_b, engine, layer, hidden_in, mask, scores, loss_value):
        ctx.engine, ctx.layer = engine, layer
        ctx.save_for_backward(hidden_in, mask, scores)
        ctx.shapes = (c1_w.shape, c1_b.shape, c2_w.shape, c2_b.shape)
        return loss_value.reshape(()).clone()

    @staticmethod
    def backward(ctx, grad_out):
        hidden_in, mask, scores = ctx.saved_tensors
        flat = ctx.engine.compressor_layer_grads(ctx.layer, hidden_in, mask, scores) * grad_out
        outs, o = [], 0
        for shp in ctx.shapes:
            n = 1
            for d in shp:
                n *= d
            outs.append(flat[o:o + n].reshape(shp))
            o += n
        return (*outs, None, None, None, None, None, None)


class _BackboneTrain(torch.autograd.Function):
    """logits -- and, for the joint objective, the layers' compressor losses -- as differentiable functions of the
    parameters (reference main_model_utils.py:108-165 with loss_type 'classification' / 'both' / 'alternate').

    forward : psv_backbone_forward_train (fp32 patch-skip forward that keeps the packed activations);
    backward: psv_backbone_backward -- d objective / d logits (and d objective / d loss_l) -> the gradient of every
    backbone parameter (and of the compressors).  The skip decisions are constants for the backward (hard thresholds),
    as in the reference's autograd graph; the layer losses reach the backbone through the compressor inputs, which the
    reference does not detach (himanshu/model_utils.py:62-65)."""

    @staticmethod
    def forward(ctx, engine, pixel_values, mlp_threshold, keys, slices, n_comp_layers, *params):
        ctx.engine, ctx.keys, ctx.slices, ctx.n_comp_layers = engine, keys, slices, n_comp_layers
        ctx.needs = [p.requires_grad for p in params]
        ctx.comp_shapes = [tuple(p.shape) for p in params[len(keys):]]
        if n_comp_layers:
            out = engine.backbone_forward_train(pixel_values, mlp_threshold, with_layer_losses=True)
        else:
            out = engine.backbone_forward_train(pixel_values, mlp_threshold)
        ctx.train_forward = engine.train_forwards
        return out

    @staticmethod
    def backward(ctx, dlogits, dlosses=None):
        if ctx.engine.train_forwards != ctx.train_forward:
            # the engine keeps the activations of ONE training forward: a later one replaced what this backward needs
            raise psv_native.PsvError(
                "another training forward ran on this model after the one being differentiated; the engine keeps the "
                "activations of the last training forward only, so call backward() after each training forward "
                "(gradient accumulation: one forward + backward per micro-batch)")
        if ctx.n_comp_layers:
            flat, cflat = ctx.engine.backbone_backward(dlogits, dlosses)
        else:
            flat, cflat = ctx.engine.backbone_backward(dlogits), None
        grads = []
        for key, need in zip(ctx.keys, ctx.needs):
            if not need:
                grads.append(None)
                continue
            off, shape = ctx.slices[key]
            n = 1
            for d in shape:
                n *= d
            grads.append(flat[off:off + n].reshape(shape))
        if ctx.n_comp_layers:
            per = cflat.numel() // ctx.n_comp_layers
            for layer in range(ctx.n_comp_layers):
                o = layer * per
                for shape in ctx.comp_shapes[4 * layer:4 * layer + 4]:      # c1_w, c1_b, c2_w, c2_b
                    n = 1
                    for d in shape:
                        n *= d
                    grads.append(cflat[o:o + n].reshape(shape))
                    o += n
        return (None, None, None, None, None, None, *grads)


class ModifiedViTLayer(ViTLayer):
    """Parameter container + per-layer entry point (reference model_utils.py:19-121)."""

    def __init__(self, config, sim_threshold=0.9, mlp_threshold=0.5, avg_threshold=0.1, mlp_needed=True):
        super().__init__(config)
        self.mlp_needed = mlp_needed
        self.loss = 0
        self._psv_owner = None          # set by ModifiedViTModel: (model, layer index)
        if not self.mlp_needed:
            return
        self.hidden_size = config.hidden_size
        self.mlp_layer = nn.Sequential(nn.Linear(self.hidden_size * 2, 64), nn.ReLU(), nn.Linear(64, 1),
                                       nn.Sigmoid())
        self.sim_threshold = sim_threshold
        self.mlp_threshold = mlp_threshold
        self.avg_threshold = avg_threshold

    def forward(self, hidden_states: torch.Tensor, head_mask=None, output_attentions: bool = False,
                compute_cosine=False, output_mask=False, previous_mask=None):
        """Same contract as the reference: returns ``(output,)`` or ``(output, boolean_mask)``; sets
        ``.loss`` / ``.mlp_accuracy_arr`` / ``.mlp_confusion_matrix`` when training or compute_cosine.
        The input tensor is not modified (the reference clones at model_utils.py:88)."""
        if self._psv_owner is None:
            raise psv_native.PsvError("ModifiedViTLayer must belong to a ModifiedViTModel (it owns the psv engine)")
        model, index = self._psv_owner
        engine = model._psv_engine_for(hidden_states.shape[0], hidden_states.device)
        if hidden_states.dtype != torch.float32:
            hidden_states = hidden_states.float()
        out = hidden_states.contiguous().clone()
        forced = None
        if not self.mlp_needed:
            forced = torch.ones(out.shape[:2], dtype=torch.uint8, device=out.device)
        elif model.skip_criterion == "similarity":
            # oracle/"cosine" criterion of reference pradeep/model_utils.py:73-84
            forced, _ = engine.similarity_mask(index, hidden_states, self.sim_threshold)
        mask, scores, _ = engine.layer_forward(index, out, getattr(self, "mlp_threshold", 0.5), forced_mask=forced)
        self.boolean_mask = mask.bool()                          # donal/model_utils.py:56
        if self.mlp_needed and (self.training or compute_cosine):
            donal = model.loss_variant == "donal"
            if getattr(engine, "_loss_variant", None) != (model.loss_variant, self.sim_threshold):
                engine.set_loss_variant(model.loss_variant, self.sim_threshold)
                engine._loss_variant = (model.loss_variant, self.sim_threshold)
            loss, sim, acc, conf = engine.layer_stats(index, hidden_states, mask, scores, self.sim_threshold)
            if torch.is_grad_enabled() and any(p.requires_grad for p in self.mlp_layer.parameters()):
                m0, m2 = self.mlp_layer[0], self.mlp_layer[2]
                labels = mask
                if donal:      # donal/model_utils.py:76: the targets are (similarity < st), CLS column unused
                    labels = torch.cat((torch.ones_like(mask[:, :1]), (sim < self.sim_threshold).to(torch.uint8)), 1)
                self.loss = _CompressorLoss.apply(m0.weight, m0.bias, m2.weight, m2.bias, engine, index,
                                                  hidden_states, labels.contiguous(), scores, loss)
            else:
                self.loss = loss.reshape(())
            self.mlp_accuracy_arr = acc
            self.similarity_val = sim
            self.mlp_confusion_counts = conf                     # device tensor, no host sync
            self.true_labels = (sim < self.sim_threshold).int().flatten()     # donal/model_utils.py:78-79
            self.pred_labels = ((scores > self.mlp_threshold) if donal else self.boolean_mask[:, 1:]).int().flatten()
            self._confusion_host = None
        else:
            self.loss = 0
        if output_mask:
            return (out, self.boolean_mask)
        return (out,)

    @property
    def mlp_confusion_matrix(self):
        """2x2 numpy array like sklearn's confusion_matrix in the reference (model_utils.py:113);
        fetched from the device lazily (this is the only host sync of the label path)."""
        if getattr(self, "_confusion_host", None) is None:
            self._confusion_host = self.mlp_confusion_counts.cpu().numpy()
        return self._confusion_host


class ModifiedViTEncoder(ViTEncoder):
    """reference model_utils.py:123-181"""

    def __init__(self, config: ViTConfig, sim_threshold=0.9, mlp_threshold=0.5, avg_threshold=0.1):
        super().__init__(config)
        self.layer = nn.ModuleList([ModifiedViTLayer(config, sim_threshold, mlp_threshold, avg_threshold, True)
                                    for _ in range(config.num_hidden_layers)])

    def forward(self, hidden_states: torch.Tensor, head_mask=None, output_attentions: bool = False,
                output_hidden_states: bool = False, return_dict: bool = True, compute_cosine: bool = False,
                output_mask: bool = False):
        all_hidden_states = () if output_hidden_states else None
        all_boolean_mask = () if output_mask else None
        for layer_module in self.layer:
            if output_hidden_states:
                all_hidden_states = all_hidden_states + (hidden_states,)
            layer_outputs = layer_module(hidden_states, None, False, compute_cosine=compute_cosine,
                                         output_mask=bool(output_mask))
            hidden_states = layer_outputs[0]
            if output_mask:
                all_boolean_mask = all_boolean_mask + (layer_outputs[1],)
        if output_hidden_states:
            all_hidden_states = all_hidden_states + (hidden_states,)
        return BaseModelOutput(last_hidden_state=hidden_states, hidden_states=all_hidden_states,
                               attentions=None), all_boolean_mask


class _Output:
    """The reference returns an ad-hoc object with .logits and .boolean_masks (model_utils.py:255-259)."""

    def __init__(self, logits, boolean_masks, hidden_states=None, n_active=None):
        self.logits = logits
        self.boolean_masks = boolean_masks
        self.hidden_states = hidden_states
        self.n_active = n_active


class ModifiedViTModel(ViTModel):
    """reference model_utils.py:183-300"""

    def __init__(self, config: ViTConfig, sim_threshold=0.9, mlp_threshold=0.5, avg_threshold=0.1):
        super().__init__(config)
        self.encoder = ModifiedViTEncoder(config, sim_threshold, mlp_threshold, avg_threshold)
        self.classifier = nn.Linear(config.hidden_size, config.num_labels)
        self.sim_threshold, self.mlp_threshold, self.avg_threshold = sim_threshold, mlp_threshold, avg_threshold
        self.psv_precision: Optional[str] = None       # None = infer from parameter dtype / PSV_PRECISION
        self.psv_use_graph = True
        self.skip_criterion = "mlp"                    # or "similarity" (BASELINE config 4, "type=cosine")
        # "active": attention among the active tokens (reference model_utils.py:88-91); "all": query-only pruning,
        # skipped tokens still serve as keys / values (reference recap/convprad4.py:99-125,191-193)
        self.kv_mode = "active"
        # backbone fine-tuning arithmetic on fp32 models: "split" (fp32-exact split-bf16 GEMMs) or "bf16" (mixed
        # precision: bf16 operands, fp32 accumulation, residual stream and statistics)
        self.psv_train_precision = "split"
        # "himanshu" (reference himanshu/model_utils.py:95-113) or "donal" (donal/model_utils.py:68-80): which loss /
        # labels / accuracy the label path computes when training or compute_cosine
        self.loss_variant = "himanshu"
        # per-layer token budget (DynamicViT / EViT style): None (the threshold decides), an int for every layer or a
        # list with one int per layer in [0, 196]; "exact" keeps that many highest-scoring patches per image, "cap" at
        # most that many of those passing mlp_threshold
        self.token_budget = None
        self.token_budget_mode = "exact"
        self._psv_engine = None
        self._psv_fingerprint = None
        for i, layer in enumerate(self.encoder.layer):
            object.__setattr__(layer, "_psv_owner", (self, i))

    # ------------------------------------------------------------------ engine management
    def _precision(self) -> str:
        if self.psv_precision:
            return self.psv_precision
        env = os.environ.get("PSV_PRECISION")
        if env:
            return env
        return "bf16" if self.classifier.weight.dtype == torch.bfloat16 else "fp32"

    def _fingerprint(self):
        """(address, version counter) of every parameter.  In-place edits through ``p.data`` (``p.data.copy_`` ...) do
        not bump the version counter: call ``psv_sync_weights()`` after such an edit."""
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def psv_sync_weights(self):
        """Force the engine to re-read every parameter from the module at the next forward (needed after edits the
        version counters cannot see, e.g. ``param.data.copy_(...)``)."""
        self._psv_fingerprint = None

    def psv_export_compressors(self):
        """Copy the ENGINE's compressor parameters into the module's ``mlp_layer`` tensors -- after native training
        (``CompressorTrainer`` on ``model._psv_engine``) the module would otherwise save stale values with
        ``torch.save(model.state_dict())`` and overwrite the trained ones at the next weight sync."""
        if self._psv_engine is None:
            return
        self._psv_engine.export_compressor_state_dict(into=self)
        self._psv_fingerprint = self._fingerprint()

    def _token_budget_setting(self):
        """(mode, keep per layer) from ``token_budget`` / ``token_budget_mode``, or None; ValueError if malformed."""
        budget, mode = self.token_budget, self.token_budget_mode
        if budget is None:
            return None
        if mode not in ("exact", "cap"):
            raise ValueError(f"token_budget_mode must be 'exact' or 'cap', not {mode!r}")
        layers, patches = len(self.encoder.layer), (self.config.image_size // self.config.patch_size) ** 2

        def one(k):
            if isinstance(k, bool) or not isinstance(k, numbers.Integral) or not 0 <= k <= patches:
                raise ValueError(f"token_budget entries must be ints in [0, {patches}], got {k!r}")
            return int(k)
        if isinstance(budget, (list, tuple)):
            if len(budget) != layers:
                raise ValueError(f"token_budget has {len(budget)} entries, the model has {layers} layers")
            return mode, tuple(one(k) for k in budget)
        return mode, (one(budget),) * layers

    def _psv_engine_for(self, batch: int, device) -> "psv_native.Engine":
        budget = self._token_budget_setting()
        device = torch.device(device)
        if device.type != "cuda":
            raise psv_native.PsvError(
                "ModifiedViTModel runs on CUDA only (B200, sm_100a): move the model and inputs to the GPU; "
                "there is no CPU fallback in this implementation")
        prec = self._precision()
        e = self._psv_engine
        if e is None or e.precision != prec or e.max_batch < batch or e.device != device:
            if e is not None:
                e.close()
            geom = geometry_from_config(self.config)
            geom = type(geom)(**{**geom.__dict__, "classes": self.classifier.out_features})
            max_batch = max(batch, int(os.environ.get("PSV_MAX_BATCH", "0")), e.max_batch if e else 0)
            with torch.cuda.device(device):
                self._psv_engine = e = psv_native.Engine(geom, prec, max_batch, device)
            self._psv_fingerprint = None
        if getattr(e, "_kv_mode", "active") != self.kv_mode:
            e.set_kv_mode(self.kv_mode)
            e._kv_mode = self.kv_mode
        if getattr(e, "_token_budget", None) != budget:
            e.set_token_budget(None if budget is None else list(budget[1]), "off" if budget is None else budget[0])
            e._token_budget = budget
        if prec == "fp32" and getattr(e, "_train_precision", "split") != self.psv_train_precision:
            e.set_train_precision(self.psv_train_precision)
            e._train_precision = self.psv_train_precision
        # the one-call and training paths decide by the engine's criterion; with differing per-layer thresholds the
        # engine stays on "mlp" and those paths refuse (the per-layer path passes its masks itself)
        st = self._common_sim_threshold()
        criterion = ("similarity", st) if self.skip_criterion == "similarity" and st is not None else ("mlp", None)
        if getattr(e, "_skip_criterion", ("mlp", None)) != criterion:
            e.set_skip_criterion(criterion[0], 0.9 if criterion[1] is None else criterion[1])
            e._skip_criterion = criterion
        fp = self._fingerprint()
        if fp != self._psv_fingerprint:
            e.load_state_dict(self.state_dict())
            self._psv_fingerprint = fp
        return e

    def _common_sim_threshold(self):
        """The layers' sim_threshold when they all agree, else None."""
        sts = {float(layer.sim_threshold) for layer in self.encoder.layer if getattr(layer, "mlp_needed", False)}
        return sts.pop() if len(sts) == 1 else None

    def _check_one_threshold(self):
        if self.skip_criterion == "similarity" and self._common_sim_threshold() is None:
            raise NotImplementedError("the similarity criterion of the one-call and training paths takes one "
                                      "sim_threshold for all layers; the layers' values differ")

    # ------------------------------------------------------------------ forward
    def forward(self, pixel_values: Optional[torch.Tensor] = None, bool_masked_pos=None, head_mask=None,
                output_attentions: Optional[bool] = None, output_hidden_states: Optional[bool] = None,
                interpolate_pos_encoding: Optional[bool] = None, return_dict: Optional[bool] = None,
                compute_cosine=False, output_mask: Optional[bool] = None):
        if pixel_values is None:
            raise ValueError("You have to specify pixel_values")
        if bool_masked_pos is not None or interpolate_pos_encoding:
            raise NotImplementedError("bool_masked_pos / interpolate_pos_encoding are not on the patch-skip path")
        if return_dict is False:
            raise NotImplementedError("return_dict=False is broken in the reference (model_utils.py:231) and not offered")
        engine = self._psv_engine_for(pixel_values.shape[0], pixel_values.device)
        if pixel_values.dtype == torch.uint8 and pixel_values.dim() == 4 and pixel_values.shape[-1] == 3:
            # extension: raw [B, H, W, 3] images; the ViTImageProcessor work of the reference's datasets
            # (main_model_utils.py:54-60) is fused into the patch embedding
            engine.set_u8_input(pixel_values.shape[1], pixel_values.shape[2])
        elif pixel_values.dtype not in (torch.float32, torch.bfloat16):
            pixel_values = pixel_values.float()                 # reference casts to the weight dtype, :223-225
        pixel_values = pixel_values.contiguous()

        # backbone fine-tuning (vit_train / vit_mlp_train / classifier_train): logits carry the autograd edge to the
        # backbone parameters; the compressor losses of the layers (when the compressors train as well) come from the
        # per-layer path below, whose own logits are discarded
        backbone = [(k, p) for k, p in self.named_parameters() if "mlp_layer" not in k and not k.startswith("pooler.")]
        if self.training and torch.is_grad_enabled() and any(p.requires_grad for _, p in backbone):
            if engine.precision != "fp32":
                raise psv_native.PsvError("backbone fine-tuning runs in the fp32 mode: set model.psv_precision = 'fp32'")
            self._check_one_threshold()
            slices = engine.backbone_grad_slices()
            keys = [k for k, _ in backbone]
            comp = [layer.mlp_layer for layer in self.encoder.layer if hasattr(layer, "mlp_layer")]
            compressors_train = any(p.requires_grad for m in comp for p in m.parameters())
            # fp32 pixel_values, or the raw uint8 images as they are (set_u8_input above; the backward re-reads them)
            pixels32 = pixel_values if pixel_values.dtype == torch.uint8 else pixel_values.float().contiguous()
            if compressors_train:
                # loss_type "both": cross-entropy + the layers' losses, one backward through everything
                if len(comp) != len(self.encoder.layer) or self.loss_variant != "himanshu":
                    raise NotImplementedError("the joint objective follows himanshu/model_utils.py: a compressor in "
                                              "every layer, labels = the layer's own mask")
                if getattr(engine, "_loss_variant", ("himanshu",))[0] != "himanshu":
                    engine.set_loss_variant("himanshu")
                    engine._loss_variant = ("himanshu", None)
                cparams = [p for m in comp for p in (m[0].weight, m[0].bias, m[2].weight, m[2].bias)]
                logits, losses = _BackboneTrain.apply(engine, pixels32, self.mlp_threshold, keys, slices, len(comp),
                                                      *[p for _, p in backbone], *cparams)
                for i, layer in enumerate(self.encoder.layer):
                    layer.loss = losses[i]
            else:
                logits = _BackboneTrain.apply(engine, pixels32, self.mlp_threshold, keys, slices, 0,
                                              *[p for _, p in backbone])
                for layer in self.encoder.layer:
                    layer.loss = 0
            return _Output(logits, None)

        per_layer = compute_cosine or self.training or output_hidden_states
        if not per_layer:
            self._check_one_threshold()
            # the hot path: one C-ABI call, no host sync, CUDA-graph replay
            r = engine.forward(pixel_values, self.mlp_threshold, want_masks=bool(output_mask), want_n_active=True,
                               use_graph=self.psv_use_graph)
            masks = tuple(m.bool() for m in r["masks"]) if output_mask else None
            for layer in self.encoder.layer:
                layer.loss = 0
            return _Output(r["logits"], masks, None, r["n_active"])

        hidden = engine.embed(pixel_values)
        enc, masks = self.encoder(hidden, output_hidden_states=bool(output_hidden_states),
                                  compute_cosine=compute_cosine, output_mask=bool(output_mask))
        logits = engine.head(enc.last_hidden_state)
        return _Output(logits, masks, enc.hidden_states)

    # ------------------------------------------------------------------ freeze modes, model_utils.py:261-300
    def vit_mlp_train(self):
        for param in self.parameters():
            param.requires_grad = True

    def vit_train(self):
        for param in self.parameters():
            param.requires_grad = True
        for layer in self.encoder.layer:
            if not hasattr(layer, 'mlp_layer'):
                continue
            for param in layer.mlp_layer.parameters():
                param.requires_grad = False

    def mlp_train(self):
        for param in self.parameters():
            param.requires_grad = False
        for layer in self.encoder.layer:
            if not hasattr(layer, 'mlp_layer'):
                continue
            for param in layer.mlp_layer.parameters():
                param.requires_grad = True

    def classifier_train(self):
        for param in self.parameters():
            param.requires_grad = False
        for param in self.classifier.parameters():
            param.requires_grad = True

    def classifier_mlp_train(self):
        for param in self.parameters():
            param.requires_grad = False
        for param in self.classifier.parameters():
            param.requires_grad = True
        for layer in self.encoder.layer:
            if not hasattr(layer, 'mlp_layer'):
                continue
            for param in layer.mlp_layer.parameters():
                param.requires_grad = True
