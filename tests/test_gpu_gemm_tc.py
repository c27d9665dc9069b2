"""GPU: the tcgen05/TMEM/TMA bf16 GEMM (gemm_tc.cu) through the psv_gemm hook against an fp64 torch
reference computed from the same bf16 operands.  fp32 accumulation => error is bounded by output
rounding (bf16 out) or ~1e-6 relative per term (fp32 out)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine(state_dicts):
    import psv_native
    geom, sd = state_dicts("deits16")
    e = psv_native.Engine(geom, "bf16", 4)
    e.load_state_dict(sd)
    yield e
    e.close()


SHAPES = [
    # m, n, k, gelu, residual, out_fp32
    (128, 256, 64, False, False, True),        # one tile, one k-block
    (128, 128, 128, False, False, True),       # BN=128 path
    (200, 768, 768, False, True, True),        # ragged M tail, residual epilogue (proj GEMM shape)
    (77, 2304, 768, False, False, False),      # QKV shape, bf16 out
    (333, 3072, 768, True, False, False),      # FC1 + GELU
    (1000, 768, 3072, False, True, True),      # FC2, long K (48 k-blocks: ring wraps many times)
    (300, 1152, 384, False, False, False),     # DeiT-S QKV (BN=128)
    (128 * 170 + 5, 768, 768, False, True, True),   # more tiles than SMs: persistent loop + TMEM double buffer
    (128 * 150, 2304, 768, False, False, False),    # 675 pair tiles = 9 full waves + 9 (tail wave of half tiles), bf16 out
    (128 * 150 - 3, 3072, 768, True, False, False), # 900 pair tiles = 12 full waves + 12, GELU epilogue
]


@pytest.mark.parametrize("m,n,k,gelu,use_res,out_fp32", SHAPES)
def test_gemm_tc_matches_torch(engine, m, n, k, gelu, use_res, out_fp32):
    torch.manual_seed(m * 7 + n)
    a = torch.randn(m, k, device="cuda").to(torch.bfloat16)
    w = (torch.randn(n, k, device="cuda") * (k ** -0.5)).to(torch.bfloat16)
    bias = torch.randn(n, device="cuda")
    res = torch.randn(m, n, device="cuda") if use_res else None
    out = engine.gemm(a, w, bias, res, out_fp32=out_fp32, gelu=gelu)
    torch.cuda.synchronize()
    if out_fp32 and not gelu:
        # the accumulate epilogue (fp32 red.global.add into the residual stream): out = base + A.W^T + bias
        base = torch.randn(m, n, device="cuda")
        acc = engine.gemm(a, w, bias, None, out_fp32=True, accumulate_into=base.clone())
        torch.cuda.synchronize()
        ref_acc = base.double() + a.double() @ w.double().t() + bias.double()
        assert float((acc.double() - ref_acc).abs().max()) < 2e-4
    ref = a.double() @ w.double().t() + bias.double()
    if gelu:
        ref = torch.nn.functional.gelu(ref)
    if use_res:
        ref = ref + res.double()
    err = (out.double() - ref).abs()
    tol = 2e-4 if out_fp32 else 2e-2 * max(1.0, float(ref.abs().max()))
    assert float(err.max()) < tol, f"max err {float(err.max())} at {int(err.argmax())} (tol {tol})"
