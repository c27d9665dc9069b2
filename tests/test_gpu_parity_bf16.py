"""GPU parity, bf16 mode (tcgen05 GEMMs, fp32 residual stream).  Free-running bf16 masks are ill-posed
(SURVEY.md 7.3: a flipped mask cascades), so the logits bar -- 2e-2 abs, top-1 agreement -- is checked
with the oracle's masks teacher-forced, and the free-running mask agreement is reported."""
import numpy as np
import pytest
import torch

import synth
from conftest import load_golden
from oracle import vit_skip_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engines(state_dicts):
    import psv_native
    cache = {}

    def get(name):
        if name not in cache:
            geom, sd = state_dicts(name)
            e = psv_native.Engine(geom, "bf16", 8)
            e.load_state_dict(sd)
            cache[name] = e
        return cache[name]
    yield get
    for e in cache.values():
        e.close()


@pytest.mark.parametrize("case,geom_name", [("vitb16_randn_b4", "vitb16"), ("vitb16_cifar_b2", "vitb16"),
                                            ("deits16_randn_b4", "deits16")])
@pytest.mark.parametrize("attention", ["auto", "mma", "tc", "pk"])
def test_bf16_logits_teacher_forced(case, geom_name, attention, engines, state_dicts):
    """every attention kernel of the bf16 mode (tcgen05 / mma.sync per image / mma.sync per packed row block /
    per-layer automatic choice) meets the bar"""
    g = load_golden(case)
    geom, _ = state_dicts(geom_name)
    e = engines(geom_name)
    e.set_attention_kernel(attention)
    B, mt = int(g["batch"]), float(g["mt"])
    x = synth.make_pixels(B, geom, seed=int(g["seed_pixels"]), kind=str(g["kind"])).cuda()
    forced = torch.from_numpy(g["masks"]).cuda()
    for use_graph in (False, True):
        r = e.forward(x, mt, forced_masks=forced, want_masks=True, want_scores=True, want_n_active=True,
                      use_graph=use_graph)
        torch.cuda.synchronize()
        assert np.array_equal(r["masks"].cpu().numpy(), g["masks"])
        assert np.array_equal(r["n_active"].cpu().numpy(), g["n_active"])
        logits = r["logits"].cpu().numpy()
        err = np.abs(logits - g["logits"]).max()
        print(f"[{case}] attention={attention} graph={use_graph} bf16 teacher-forced logits max-abs err {err:.4f}; scores err "
              f"{np.abs(r['scores'].cpu().numpy() - g['scores']).max():.2e}")
        assert err < 2e-2
        assert (logits.argmax(-1) == g["logits"].argmax(-1)).all()
    free = e.forward(x, mt, want_masks=True)
    torch.cuda.synchronize()
    e.set_attention_kernel("auto")
    agree = (free["masks"].cpu().numpy() == g["masks"]).mean()
    print(f"[{case}] bf16 free-running mask agreement {agree:.4%} (reported, not asserted)")


def test_bf16_layers_teacher_forced(engines, state_dicts):
    geom, sd = state_dicts("vitb16")
    e = engines("vitb16")
    x = synth.make_pixels(3, geom, seed=21)
    with torch.no_grad():
        h = O.embed(sd, x)
        assert (e.embed(x.cuda()).cpu() - h).abs().max() < 2e-2
        worst = 0.0
        for l in range(geom.layers):
            out, mask, scores = O.layer_forward(sd, l, h, 0.5)
            # the compressor runs as split-bf16 tcgen05 MMAs: fp32-class scores, bit-exact masks outside the band
            m_free, s_free, n_free = e.layer_forward(l, h.cuda().contiguous(), 0.5)
            torch.cuda.synchronize()
            s_err = float((s_free.cpu() - scores).abs().max())
            assert s_err < 2e-5, f"layer {l}: score err {s_err}"
            diff = m_free.cpu().bool() != mask
            in_band = torch.cat((torch.zeros(3, 1, dtype=torch.bool), (scores - 0.5).abs() < 1e-4), 1)
            assert not (diff & ~in_band).any(), f"layer {l}: mask flips outside the band"
            assert torch.equal(n_free.cpu().long(), m_free.cpu().long().sum(1))
            idx_gpu, cu_gpu = e.get_compaction(3)
            idx, cu, _ = O.compact(m_free.cpu().bool())
            assert torch.equal(cu_gpu.cpu(), cu) and torch.equal(idx_gpu.cpu()[:int(cu[-1])], idx)
            hg = h.cuda().contiguous()
            e.layer_forward(l, hg, 0.5, forced_mask=mask.to(torch.uint8).cuda())
            torch.cuda.synchronize()
            err = float((hg.cpu() - out).abs().max())
            worst = max(worst, err)
            assert err < 3e-2, f"layer {l}: {err}"
            assert torch.equal(hg.cpu()[~mask], h[~mask])
            h = out
    print(f"bf16 per-layer teacher-forced worst abs err {worst:.4f}")


def test_host_paths_agree_with_device_path(engines, state_dicts):
    """psv_forward_host (blocking) and psv_forward_host_submit/_wait (double-buffered) = psv_forward."""
    geom, _ = state_dicts("deits16")
    e = engines("deits16")
    # one fixed attention kernel: under "auto" the graph path may pick another kernel per layer than the eager
    # reference (same results within tolerance, not the same bits)
    e.set_attention_kernel("tc")
    xs = [synth.make_pixels(6, geom, seed=50 + i) for i in range(3)]
    ref = [e.forward(x.cuda(), 0.5, want_n_active=True) for x in xs]
    torch.cuda.synchronize()
    pinned = [x.pin_memory() for x in xs]
    for i, x in enumerate(pinned):
        nact = torch.empty(geom.layers, 6, dtype=torch.int32).pin_memory()
        logits = e.forward_host(x, 0.5, host_n_active=nact)
        # bit-equal: the forward is deterministic (one fp32 red.add per element per GEMM; stream-K is off by default)
        assert torch.equal(logits, ref[i]["logits"].cpu()) and torch.equal(nact, ref[i]["n_active"].cpu())
    outs = [torch.empty(6, geom.classes).pin_memory() for _ in range(3)]
    for i, x in enumerate(pinned):
        e.forward_host_submit(i & 1, x, 0.5, outs[i])
        if i >= 1:
            e.forward_host_wait((i - 1) & 1)
    e.forward_host_wait(0)
    for i in range(3):
        assert torch.equal(outs[i], ref[i]["logits"].cpu())
    with pytest.raises(Exception):
        e.forward_host_wait(1)                       # nothing in flight
    e.set_attention_kernel("auto")


@pytest.mark.parametrize("attention", ["mma", "tc"])
@pytest.mark.parametrize("batch,mt", [(1, 0.0), (1, 1.5), (5, 0.0), (5, 1.5)])
def test_bf16_edge_batches_and_masks(attention, batch, mt, engines, state_dicts):
    """ragged / extreme cases of the packed path: a single image, every token active (mt = 0: 197 rows per image,
    two query tiles) and every patch skipped (mt > 1: only the CLS row of each image is packed, T = batch)."""
    geom, sd = state_dicts("deits16")
    e = engines("deits16")
    e.set_attention_kernel(attention)
    x = synth.make_pixels(batch, geom, seed=300 + batch)
    with torch.no_grad():
        ref = O.forward(sd, x, mt, 0.9)
    want_active = geom.tokens if mt == 0.0 else 1
    assert int(ref.masks.sum()) == geom.layers * batch * want_active
    for use_graph in (False, True):
        r = e.forward(x.cuda(), mt, want_masks=True, want_n_active=True, use_graph=use_graph)
        torch.cuda.synchronize()
        assert torch.equal(r["masks"].cpu().bool(), ref.masks)
        assert (r["n_active"].cpu() == want_active).all()
        err = float((r["logits"].cpu() - ref.logits).abs().max())
        assert err < 2e-2, f"B={batch} mt={mt} attention={attention}: logits err {err}"
    e.set_attention_kernel("auto")

