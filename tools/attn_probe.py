"""Attention kernel time vs tokens per image (psv_attention hook, CUDA events, B images of n tokens each).
usage: [PSV_ATTENTION_MMA=1] python tools/attn_probe.py [batch] [n ...]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vit-pruning_b200"), ROOT]
import torch, psv_native, synth
B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
ns = [int(a) for a in sys.argv[2:]] or [4, 16, 32, 33, 48, 64, 70, 100, 128, 150, 183, 197]
geom = synth.VIT_B16
eng = psv_native.Engine(geom, "bf16", B)
eng.load_state_dict(synth.make_state_dict(geom, 42))
kind = "mma.sync" if os.environ.get("PSV_ATTENTION_MMA") else "tcgen05"
eng.set_attention_kernel("mma" if kind == "mma.sync" else "tc")
for n in ns:
    total = B * n
    qkv = torch.randn(total, 3 * geom.hidden, device="cuda").to(torch.bfloat16)
    cu = (torch.arange(B + 1, device="cuda") * n).to(torch.int32)
    ctx = torch.zeros(total, geom.hidden, device="cuda", dtype=torch.bfloat16)
    reps = 20
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):
            eng.attention(qkv, cu, out=ctx)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()                 # device-side time: no host launch gaps between the calls
    with torch.cuda.graph(graph, stream=side):
        for _ in range(reps):
            eng.attention(qkv, cu, out=ctx)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / reps * 1e3
    flops = 4.0 * n * n * 64 * geom.heads * B
    print(f"{kind:9s} B={B} n={n:4d}: {us:8.1f} us   {flops / us * 1e-6:7.1f} TFLOP/s")
