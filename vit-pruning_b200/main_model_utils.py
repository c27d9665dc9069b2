"""Callers of the hot path, mirroring the reference's ``himanshu/main_model_utils.py``:

* ``test(model, dataloader, device, log_file, full_testing)``  -- reference :235-300.  Same printed
  report and return values, but the per-layer 2x2 confusion counts are accumulated ON THE DEVICE
  (one host copy at the end instead of a ``.cpu()`` + sklearn call per layer per batch).
* ``train(model, train_loader, test_loader, device, log_file, save_path, num_epochs, loss_type, lr)``
  -- reference :100-191.  ``loss_type="cosine"`` (compressor training on a frozen backbone, BASELINE config 5),
  ``"classification"`` / ``"both"`` / ``"alternate"`` (backbone fine-tuning through the patch-skip forward, fp32 mode).
* ``CompressorTrainer`` -- the native data-parallel form of the same compressor training: every rank
  runs ``psv_compressor_grads`` on its shard of the batch, the flat fp32 gradient (1.18 M floats)
  is all-reduced with NCCL, and every rank applies the same fused Adam step (``psv_compressor_adam_step``).
* ``synthetic_loader`` -- the datasets of the reference need the network (torchvision CIFAR-100
  download, HF image processor); here batches are synthetic CIFAR-100-shaped tensors.

Out of scope (I/O and reporting, not the hot path): CIFAR100Dataset / TinyImageNetDataset,
``get_complexity`` (ptflops), ``FocalLoss`` (imported by the reference's model_utils.py:8 but never used).
"""
from __future__ import annotations

import numpy as np
import torch

import synth


def write_N_print(string, log_file):
    """reference :304-306"""
    print(string)
    if log_file is not None:
        log_file.write(string + "\n")


class _SyntheticDataset(torch.utils.data.Dataset):
    def __init__(self, n, geom, seed, kind):
        self.x = synth.make_pixels(n, geom, seed=seed, kind=kind)
        rng = np.random.Generator(np.random.PCG64(seed + 1))
        self.y = torch.from_numpy(rng.integers(0, geom.classes, size=n))

    def __len__(self):
        return self.x.shape[0]

    def __getitem__(self, i):
        return self.x[i], self.y[i]


def synthetic_loader(n_images, batch_size, geom=synth.VIT_B16, seed=1234, kind="cifar", pin_memory=True):
    """DataLoader over synthetic CIFAR-100-shaped images (pixel_values, label), reference :42-61 stand-in."""
    ds = _SyntheticDataset(n_images, geom, seed, kind)
    return torch.utils.data.DataLoader(ds, batch_size=batch_size, shuffle=False, pin_memory=pin_memory)


def test(model, dataloader, device, log_file=None, full_testing=False):
    """reference :235-300.  Returns accuracy, or (accuracy, mlp_accuracy) with full_testing."""
    model.eval()
    n_layers = len(model.encoder.layer)
    total_correct = torch.zeros((), dtype=torch.int64, device=device)
    total_correct_mlp = torch.zeros(n_layers, 2, 2, dtype=torch.int64, device=device) if full_testing else None
    data_size = len(dataloader.dataset)
    with torch.no_grad():
        for inputs, labels in dataloader:
            inputs = inputs.to(device, non_blocking=True)
            labels = labels.to(device, non_blocking=True)
            outputs = model(inputs, compute_cosine=True) if full_testing else model(inputs)
            predicted = outputs.logits.argmax(dim=-1)
            if full_testing:
                for i, layer in enumerate(model.encoder.layer):
                    if hasattr(layer, 'mlp_confusion_counts'):
                        total_correct_mlp[i] += layer.mlp_confusion_counts       # stays on the device
            total_correct += (predicted == labels).sum()
    accuracy = float(total_correct.item()) / data_size
    if not full_testing:
        return accuracy
    tcm = total_correct_mlp.cpu().float()                                       # the only host copy
    each_layer_skip = (tcm.sum(dim=[1], keepdim=True) / tcm.sum(dim=[1, 2], keepdim=True))[:, 0, 0]
    mlp_accuracy = (tcm[:, 1, 1].sum() + tcm[:, 0, 0].sum()) / (tcm.sum() + 1e-16)
    mlp_accuracy_arr = (tcm[:, 1, 1] + tcm[:, 0, 0]) / tcm.sum(dim=[1, 2])
    write_N_print(f"Skip %: {each_layer_skip.mean():.2%}\nOverall accuracy of MLP: {mlp_accuracy:.2%}", log_file)
    header = "              " + " ".join(f"L{i:>5d}" for i in range(n_layers))
    write_N_print(header, log_file)
    write_N_print("Skip ratio    " + " ".join(f"{100 * v:6.1f}" for v in each_layer_skip.tolist()), log_file)
    write_N_print("MLP accuracy  " + " ".join(f"{100 * v:6.1f}" for v in mlp_accuracy_arr.tolist()), log_file)
    conf = (tcm / (tcm.sum(dim=[-2, -1], keepdim=True) + 1e-16))
    write_N_print("\nConfusion matrix for each layer (rows: true skip/process, cols: predicted):", log_file)
    for r in range(2):
        write_N_print("   ".join(f"{conf[i, r, 0]:.3f} {conf[i, r, 1]:.3f}" for i in range(n_layers)), log_file)
    write_N_print(f"Overall accuracy: {accuracy:.2%}\n", log_file)
    return accuracy, float(mlp_accuracy)


def train(model, train_loader, test_loader, device, log_file=None, save_path=None, num_epochs=10,
          loss_type='cosine', lr=1e-3):
    """reference :100-191.  loss_type: "cosine" (compressors only, ``mlp_train``), "classification" (backbone only,
    ``vit_train``), "both" (``vit_mlp_train``: cross-entropy + the layers' compressor losses) or "alternate" (compressors
    every third epoch, backbone otherwise).  Adam on the trainable parameters, as the reference.  The backbone modes
    need the fp32 mode (``model.psv_precision = "fp32"``); all four train in either ``model.kv_mode``.  The backbone
    modes also train under either ``model.skip_criterion`` ("mlp", or "similarity" with one ``sim_threshold`` for all
    layers) and from raw uint8 ``[B, H, W, 3]`` images as well as from pixel_values."""
    if loss_type not in ("cosine", "classification", "both", "alternate"):
        raise ValueError(f"unknown loss_type {loss_type!r}")
    model.train()
    criterion = torch.nn.CrossEntropyLoss()
    cosine_loss_ratio = 1
    if loss_type == "cosine":
        model.mlp_train()
    elif loss_type == "classification":
        model.vit_train()
    elif loss_type == "both":
        model.vit_mlp_train()
    optimizer = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=lr)
    best_val_accuracy, history = 0.0, []
    for epoch in range(num_epochs):
        model.train()
        if loss_type == "alternate":
            if epoch % 3 == 0:
                model.mlp_train()
            else:
                model.vit_train()
        running = 0.0
        for inputs, labels in train_loader:
            inputs = inputs.to(device, non_blocking=True)
            labels = labels.to(device, non_blocking=True)
            logits = model(inputs).logits
            layer_losses = lambda: sum((layer.loss for layer in model.encoder.layer), 0.0)
            if loss_type == "classification":
                total_loss = criterion(logits, labels)
            elif loss_type == "cosine":
                total_loss = layer_losses()
            elif loss_type == "both":
                total_loss = criterion(logits, labels) + cosine_loss_ratio * layer_losses()
            else:
                total_loss = layer_losses() if epoch % 3 == 0 else criterion(logits, labels)
            optimizer.zero_grad()
            total_loss.backward()
            optimizer.step()
            running += float(total_loss.item())
        history.append(running / max(1, len(train_loader)))
        if test_loader is not None:
            val_accuracy, _ = test(model, test_loader, device, log_file, full_testing=True)
            if val_accuracy > best_val_accuracy:
                best_val_accuracy = val_accuracy
                if save_path:
                    torch.save(model.state_dict(), f"models/{save_path}.pth")
            write_N_print(f"Test accuracy after {epoch + 1} epochs: {val_accuracy:.2%}\n", log_file)
    write_N_print(f"Best accuracy: {best_val_accuracy * 100}%\n", log_file)
    return history


class CompressorTrainer:
    """Data-parallel compressor training on the native path (BASELINE config 5).

    Each rank holds a full engine (weights replicated) and a shard of every batch.  Per step:
    ``psv_compressor_grads`` (forward in skip mode + per-layer loss and gradient, one call, no host
    sync) -> the gradient exchange -> Adam with ``grad_scale = 1 / world_size`` (the same update on every rank keeps
    the replicas bit-identical).  Two exchanges (``collective``):

    * ``"p2p-fused"`` (default when torch symmetric memory can map the peers' buckets, i.e. NVLink/NVSwitch P2P): every
      rank writes its gradients into a symmetric-memory bucket and ONE kernel (``psv_compressor_peer_reduce_adam_step``)
      reads all ranks' buckets over NVLink, sums them in rank order and applies Adam -- the all-reduce and the
      optimizer are a single pass, bracketed by two symmetric-memory barriers;
    * ``"nccl"``: one ``all_reduce(SUM)`` of the flat fp32 bucket (1 181 232 floats, 4.7 MB), then
      ``psv_compressor_adam_step``.

    The reference's ``pos_weight`` is a batch statistic; it is computed per rank (equals the reference at world size
    1; SURVEY.md 8e).  The skip layers run in the engine's kv mode (``engine.set_kv_mode``), as the drop-in's forward.
    """

    def __init__(self, engine, mlp_threshold=0.5, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, process_group=None,
                 collective="auto"):
        self.engine, self.mt, self.lr, self.betas, self.eps = engine, mlp_threshold, lr, betas, eps
        self.group = process_group
        self.step_count = 0
        self.world = torch.distributed.get_world_size(process_group) if self._dist() else 1
        self.collective, self.collective_note = "none", ""
        self._symm = self._hdl = self._peer_ptrs = None
        if self.world > 1:
            self.collective = "nccl"
            if collective in ("auto", "p2p-fused") and self.world <= 16:
                try:
                    self._setup_peer_buckets()
                    self.collective = "p2p-fused"
                except Exception as ex:                       # no P2P mapping on this system: NCCL all-reduce
                    self.collective_note = f"symmetric memory unavailable: {str(ex)[:160]}"
                    if collective == "p2p-fused":
                        raise

    def _setup_peer_buckets(self):
        import torch.distributed._symmetric_memory as symm_mem
        dist = torch.distributed
        n = self.engine.compressor_param_count
        with torch.cuda.device(self.engine.device):
            self._symm = symm_mem.empty(n, dtype=torch.float32, device=self.engine.device)
        group = self.group if self.group is not None else dist.group.WORLD
        self._hdl = symm_mem.rendezvous(self._symm, group)
        self._peer_ptrs = [int(p) for p in self._hdl.buffer_ptrs]
        assert len(self._peer_ptrs) == self.world and self._peer_ptrs[self._hdl.rank] == self._symm.data_ptr()

    @staticmethod
    def _dist():
        return torch.distributed.is_available() and torch.distributed.is_initialized()

    def step(self, pixels):
        """One optimisation step on this rank's shard; returns the per-layer losses (device tensor)."""
        self.step_count += 1
        if self.collective == "p2p-fused":
            _, loss = self.engine.compressor_grads(pixels, self.mt, out=self._symm)
            self._hdl.barrier(channel=0)                  # every rank's bucket is complete
            self.engine.compressor_peer_reduce_adam_step(self._peer_ptrs, lr=self.lr, beta1=self.betas[0],
                                                         beta2=self.betas[1], eps=self.eps, step=self.step_count,
                                                         grad_scale=1.0 / self.world)
            self._hdl.barrier(channel=1)                  # every rank has read every bucket: safe to overwrite
            return loss
        grads, loss = self.engine.compressor_grads(pixels, self.mt)
        if self.world > 1:
            torch.distributed.all_reduce(grads, op=torch.distributed.ReduceOp.SUM, group=self.group)
        self.engine.compressor_adam_step(grads, lr=self.lr, beta1=self.betas[0], beta2=self.betas[1], eps=self.eps,
                                         step=self.step_count, grad_scale=1.0 / self.world)
        return loss


    # ---- checkpointing (the reference saves model.state_dict(), main_model_utils.py:181-183)
    def export_to(self, model):
        """Write the natively trained compressor parameters into ``model`` (an nn.Module with the reference's keys) so
        that ``torch.save(model.state_dict())`` stores them; also marks the drop-in's engine cache as up to date."""
        out = self.engine.export_compressor_state_dict(into=model)
        if hasattr(model, "psv_sync_weights") and getattr(model, "_psv_engine", None) is self.engine:
            model._psv_fingerprint = model._fingerprint()      # module and engine hold the same values now
        return out

    def state_dict(self):
        """Optimizer state for a resumable checkpoint: step counter and the Adam moments."""
        m, v = self.engine.get_compressor_adam_state()
        return {"step": self.step_count, "exp_avg": m.cpu(), "exp_avg_sq": v.cpu(),
                "params": self.engine.get_compressor_params().cpu()}

    def load_state_dict(self, state):
        self.step_count = int(state["step"])
        self.engine.set_compressor_adam_state(state["exp_avg"], state["exp_avg_sq"])
        self.engine.set_compressor_params(state["params"].to(self.engine.device).float().contiguous())


def shard_bounds(total, world, rank):
    """Contiguous shard [lo, hi) of ``total`` items for ``rank`` of ``world`` (batch sharding, SURVEY.md 8e)."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def flat_compressor_params(state_dict, geom):
    """The handle's flat compressor layout from a reference-keyed state dict:
    per layer [c1_w (64 x 2D) | c1_b (64) | c2_w (64) | c2_b (1) | zero pad to a multiple of 4]."""
    per = geom.comp_hidden * 2 * geom.hidden + 2 * geom.comp_hidden + 1
    stride = (per + 3) // 4 * 4
    out = torch.zeros(geom.layers * stride, dtype=torch.float32)
    for i in range(geom.layers):
        p = f"encoder.layer.{i}.mlp_layer."
        parts = [state_dict[p + "0.weight"].reshape(-1), state_dict[p + "0.bias"].reshape(-1),
                 state_dict[p + "2.weight"].reshape(-1), state_dict[p + "2.bias"].reshape(-1)]
        flat = torch.cat([t.detach().float().cpu() for t in parts])
        out[i * stride:i * stride + per] = flat
    return out
