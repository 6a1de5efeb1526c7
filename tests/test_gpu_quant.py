"""-m gpu: the quantized linears through the C ABI against the oracle / golden vectors.

Bars: integer work (unpack, dequant in a given dtype, re-tiling) bit-exact; linear outputs
normwise within 1e-3 of exact arithmetic (north_star) and within the reference's own bf16
tolerance (tests/test_model.py:133) of the reference's CPU forward."""
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

from oracle import llama_oracle as O  # noqa: E402


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _module(case, dev, dtype):
    from lit_llama_b200.quantization import ColBlockQuantizedLinear

    out_f, in_f = case["w"].shape
    lin = ColBlockQuantizedLinear(in_f, out_f, False, bits=case["bits"], tile_cols=case["groupsize"]).to(dev)
    lin.load_state_dict({"quant_weight": case["quant_weight"], "scales": case["scales"].to(dtype), "zeros": case["zeros"].to(dtype)})
    lin.scales = lin.scales.to(dtype)
    lin.zeros = lin.zeros.to(dtype)
    return lin


def test_dequant_bit_exact_vs_reference(dev):
    for c in load_golden("quant_cases.pt"):
        lin = _module(c, dev, torch.float32)
        assert tuple(lin.quant_weight.stride()) == c["qw_stride"]
        assert torch.equal(lin.get_weight(torch.float32).cpu(), c["deq_f32"])
        assert torch.equal(lin.get_weight(torch.bfloat16).cpu(), c["deq_bf16"])


def test_linear_vs_reference_forward(dev):
    for c in load_golden("quant_cases.pt"):
        lin = _module(c, dev, torch.bfloat16)
        x = c["x"].bfloat16().to(dev)
        y = lin(x).float().cpu()
        # reference's CPU bf16 forward (dense branch, every weight rounded to bf16): within one bf16 ulp
        torch.testing.assert_close(y, c["y_bf16"].float(), rtol=2.0 ** -7, atol=5e-3)
        # exact arithmetic on the same stored parameters
        tc = c["w"].shape[1] if c["groupsize"] == -1 else c["groupsize"]
        exact = O.qlinear_exact(x.cpu().float(), c["quant_weight"], c["scales"].bfloat16(), c["zeros"].bfloat16(), c["bits"], tc)
        assert (y - exact).norm() / exact.norm() < 1e-3 + 2.0 ** -9


def test_tile_roundtrip_bit_exact(dev):
    from gpu_util import rand_q4, tile
    from lit_llama_b200 import _lib as L

    for N, K in [(128, 64), (130, 256), (96, 128), (4096, 4096), (11008, 4096)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=N)
        qt = tile(L, qw, N, K)
        back = torch.empty_like(qw)
        L.check(L.lib().b2l_q4_untile(qt.data_ptr(), back.data_ptr(), N, K, L.stream_ptr()), "untile")
        assert torch.equal(back, qw)
        # documented layout, decoded independently on the host for a few words
        w = qt.view(torch.int32).reshape(-1, K // 32, 128, 4).cpu()
        lvc = lv.cpu()
        for (nt, ks, r, i) in [(0, 0, 0, 0), (0, K // 32 - 1, 5, 3), ((N - 1) // 128, 1 % (K // 32), (N - 1) % 128, 2)]:
            word = int(w[nt, ks, r, i]) & 0xFFFFFFFF
            for s in range(8):
                k = ks * 32 + 8 * i + (2 * s if s < 4 else 2 * (s - 4) + 1)
                assert ((word >> (4 * s)) & 0xF) == int(lvc[nt * 128 + r, k])


@pytest.mark.parametrize("N,K,M,S", [(128, 64, 1, 1), (128, 96, 1, 1), (128, 256, 3, 1), (128, 256, 1, 2), (256, 512, 1, 4),
                                     (256, 1024, 8, 8), (130, 256, 2, 2), (128, 1024, 16, 2), (384, 4096, 1, 0)])
def test_tc_linear_small(dev, N, K, M, S):
    from gpu_util import rand_q4, ref_linear, relerr, tc_call, tile
    from lit_llama_b200 import _lib as L

    lv, qw, sc, z = rand_q4(N, K, dev, seed=N + K + M)
    qt = tile(L, qw, N, K)
    x = torch.randn(M, K, device=dev).bfloat16()
    y, err = tc_call(L, x, qt, sc, z, N, K, split_k=S)
    torch.cuda.synchronize()
    assert err is None, err
    want = ref_linear(x, lv, sc, z)
    assert relerr(y, want) < 1e-3 + 2.0 ** -9  # bf16 output rounding alone is up to 2^-9 normwise
    # against the exact result rounded to bf16: at most 1 ulp apart, almost everywhere equal
    wb = want.float().bfloat16()
    assert float((y == wb).float().mean()) > 0.98


@pytest.mark.parametrize("N,K,grid", [(16, 64, 0), (16, 128, 0), (32, 2048, 0), (48, 4096, 0), (130, 256, 0), (4096, 4096, 0),
                                       (4096, 4096, 7), (4096, 4096, 100), (128, 6400, 0), (112, 11008, 3), (4096, 11008, 0),
                                       (4096, 11008, 77)])
def test_gemv_small_and_ragged(dev, N, K, grid):
    """Batch-1 kernel: odd block counts (pairs + a single), padded rows, short last stage, forced tiny grids."""
    from gpu_util import assert_q4_linear_close, gemv_call, rand_q4, tile_i8, tile_mma
    from lit_llama_b200 import _lib as L

    lv, qw, sc, z = rand_q4(N, K, dev, seed=N + K)
    qt = tile_i8(L, qw, N, K)
    back = torch.empty_like(qw)
    L.check(L.lib().b2l_q4_untile_i8(qt.data_ptr(), back.data_ptr(), N, K, L.stream_ptr()), "untile_i8")
    assert torch.equal(back, qw)  # the re-tiling is a pure permutation of nibbles
    back.zero_()
    L.check(L.lib().b2l_q4_untile_mma(tile_mma(L, qw, N, K).data_ptr(), back.data_ptr(), N, K, L.stream_ptr()), "untile_mma")
    assert torch.equal(back, qw)  # and so is the f16-fragment tiling of the 2..8-row kernel
    x = torch.randn(1, K, device=dev).bfloat16()
    y, err = gemv_call(L, x, qt, sc, z, N, K, grid=grid)
    torch.cuda.synchronize()
    assert err is None, err
    assert_q4_linear_close(y, x, lv, sc, z, min_equal=0.995)  # exact integer contraction: only double rounding differs


def test_gemv_prologue_epilogue_and_determinism(dev):
    from gpu_util import gemv_call, rand_q4, ref_linear, relerr, tile_i8
    from lit_llama_b200 import _lib as L

    torch.manual_seed(11)
    N, K = 512, 1024
    lv, qw, sc, z = rand_q4(N, K, dev, seed=5)
    qt = tile_i8(L, qw, N, K)
    x = (torch.randn(1, K, device=dev) * 0.7).bfloat16()
    g = (1 + 0.1 * torch.randn(K, device=dev)).bfloat16()
    xn = g * (x * torch.rsqrt(torch.mean(x * x, dim=-1, keepdim=True) + 1e-5))  # model.py:270-277 in bf16 on this device
    y, err = gemv_call(L, x, qt, sc, z, N, K, prologue=1, norm_scale=g)
    assert err is None, err
    assert relerr(y, ref_linear(xn, lv, sc, z)) < 1e-3 + 2.0 ** -9
    res = torch.randn(1, N, device=dev).bfloat16()
    y, err = gemv_call(L, x, qt, sc, z, N, K, epilogue=1, res=res)
    want = ref_linear(x, lv, sc, z).float().bfloat16() + res
    # exact contraction: only the fp32 -> bf16 double rounding can differ from the correctly rounded result
    assert err is None and float((y == want).float().mean()) > 0.99
    assert relerr(y, want) < 2.0 ** -9
    buf = res.clone()
    _, err = gemv_call(L, x, qt, sc, z, N, K, epilogue=1, res=buf, y=buf)
    assert err is None and torch.equal(buf, y)
    full = ref_linear(x, lv, sc, z).float().bfloat16().reshape(1, N // 16, 2, 8)
    a, b = full[:, :, 0].reshape(1, -1), full[:, :, 1].reshape(1, -1)
    y, err = gemv_call(L, x, qt, sc, z, N, K, epilogue=2, n_out=N // 2)
    want = torch.nn.functional.silu(a) * b
    assert err is None and float((y == want).float().mean()) > 0.97 and relerr(y, want) < 2.0 ** -8
    # bit-identical across runs and grid sizes (integer accumulation: the result does not depend on any order)
    y0, _ = gemv_call(L, x, qt, sc, z, N, K)
    for grid in (0, 5, 32, 100):
        y1, _ = gemv_call(L, x, qt, sc, z, N, K, grid=grid)
        assert torch.equal(y0, y1)


@pytest.mark.parametrize("N,K,M,grid", [(4096, 4096, 8, 0), (4096, 11008, 5, 0), (22016, 4096, 2, 0), (130, 256, 3, 0), (48, 4096, 8, 2),
                                         (16, 64, 1, 0), (5120, 13824, 8, 0), (4096, 4096, 7, 100)])
def test_gemv_batch_vs_exact_and_vs_batch1(dev, N, K, M, grid):
    """The 2..8-row kernel (f16 MMA, fp32 accumulation): every row against exact arithmetic, and within one bf16
    ulp of the batch-1 kernel (exact integer contraction) on that row, equal almost everywhere."""
    from gpu_util import assert_q4_linear_close, gemv_batch_call, gemv_call, rand_q4, relerr, tile_i8, tile_mma
    from lit_llama_b200 import _lib as L

    lv, qw, sc, z = rand_q4(N, K, dev, seed=N + K + M)
    qt, q8 = tile_mma(L, qw, N, K), tile_i8(L, qw, N, K)
    x = torch.randn(M, K, device=dev).bfloat16()
    y, err = gemv_batch_call(L, x, qt, sc, z, N, K, grid=grid)
    assert err is None, err
    assert_q4_linear_close(y, x, lv, sc, z)
    for m in range(M):
        y1, err = gemv_call(L, x[m : m + 1].contiguous(), q8, sc, z, N, K, grid=grid)
        assert err is None, err
        assert float((y[m : m + 1] == y1).float().mean()) > 0.85 and relerr(y[m : m + 1], y1) < 2.0 ** -9, m


def test_gemv_batch_prologue_epilogue(dev):
    from gpu_util import gemv_batch_call, gemv_call, rand_q4, relerr, tile_i8, tile_mma
    from lit_llama_b200 import _lib as L

    N, K, M = 512, 1024, 6
    lv, qw, sc, z = rand_q4(N, K, dev, seed=5)
    qt, q8 = tile_mma(L, qw, N, K), tile_i8(L, qw, N, K)
    x = (torch.randn(M, K, device=dev) * 0.7).bfloat16()
    g = (1 + 0.1 * torch.randn(K, device=dev)).bfloat16()
    res = torch.randn(M, N, device=dev).bfloat16()
    for kw in (dict(prologue=1, norm_scale=g), dict(epilogue=1, res=res), dict(prologue=1, norm_scale=g, epilogue=2, n_out=N // 2)):
        y, err = gemv_batch_call(L, x, qt, sc, z, N, K, **kw)
        assert err is None, err
        for m in range(M):   # the batch-1 kernel (itself checked against the reference formulas) row by row
            kw1 = dict(kw)
            if "res" in kw1:
                kw1["res"] = res[m : m + 1].contiguous()
            y1, err = gemv_call(L, x[m : m + 1].contiguous(), q8, sc, z, N, K, **kw1)
            assert err is None, err
            # f16-MMA batch kernel vs exact batch-1 kernel: 1-ulp flips only (SwiGLU multiplies two such values)
            assert float((y[m : m + 1] == y1).float().mean()) > 0.85 and relerr(y[m : m + 1], y1) < 2.0 ** -8, (kw.keys(), m)
    # in place on the residual stream (x + h with y aliasing res), twice the same result
    buf = res.clone()
    y, _ = gemv_batch_call(L, x, qt, sc, z, N, K, epilogue=1, res=res)
    _, err = gemv_batch_call(L, x, qt, sc, z, N, K, epilogue=1, res=buf, y=buf)
    assert err is None and torch.equal(buf, y)
    # argument checks
    _, err = gemv_batch_call(L, torch.zeros(9, K, device=dev, dtype=torch.bfloat16), qt, sc, z, N, K)
    assert err is not None and "M=9" in err


@pytest.mark.parametrize("name,N,K", [("13B c_attn", 15360, 5120), ("13B mlp_proj", 5120, 13824), ("65B c_proj", 8192, 8192),
                                      ("65B mlp_proj", 8192, 22016),
                                      # the shards of tensor-parallel decode (tp.py): 65B over 8 ranks, 7B over 4
                                      ("65B/8 mlp_proj", 8192, 2752), ("65B/8 c_proj", 8192, 1024), ("65B/8 c_attn", 3072, 8192),
                                      ("65B/8 lm_head", 4000, 8192), ("7B/4 c_proj", 4096, 1024)])
def test_gemv_13b_65b_shapes(dev, name, N, K):
    """The other BASELINE model widths through the batch-1 kernel (K = 22016 exercises the wide-row prologue)."""
    from gpu_util import gemv_call, rand_q4, ref_linear, relerr, tile_i8
    from lit_llama_b200 import _lib as L

    lv, qw, sc, z = rand_q4(N, K, dev, seed=N % 97 + K)
    qt = tile_i8(L, qw, N, K)
    x = torch.randn(1, K, device=dev).bfloat16()
    g = (1 + 0.1 * torch.randn(K, device=dev)).bfloat16()
    y, err = gemv_call(L, x, qt, sc, z, N, K)
    assert err is None, err
    assert relerr(y, ref_linear(x, lv, sc, z)) < 1e-3 + 2.0 ** -9
    xn = g * (x * torch.rsqrt(torch.mean(x * x, dim=-1, keepdim=True) + 1e-5))
    y, err = gemv_call(L, x, qt, sc, z, N, K, prologue=1, norm_scale=g)
    assert err is None, err
    assert relerr(y, ref_linear(xn, lv, sc, z)) < 1e-3 + 2.0 ** -9


@pytest.mark.parametrize("M,N,K", [(17, 256, 64), (100, 384, 128), (300, 130, 256), (256, 512, 512), (257, 768, 256), (1000, 4096, 4096),
                                   (64, 32000, 4096), (4096, 15360, 5120), (4096, 5120, 13824)])
def test_q4_gemm_prefill_shapes(dev, M, N, K):
    """The tcgen05 prefill GEMM (M > 16) against the reference's dense branch evaluated by torch in fp32 on the SAME
    bf16-rounded dequantised matrix (quantization.py:392-423: get_weight rounds (level - zero) * scale to bf16, F.linear
    accumulates): ragged M / N tiles, one k stage, the 13B widths of BASELINE configs[3] at M = 8 x 512."""
    import ctypes as C

    from gpu_util import rand_q4, relerr, tile
    from lit_llama_b200 import _lib as L

    lv, qw, sc, z = rand_q4(N, K, dev, seed=M + N + K)
    qt = tile(L, qw, N, K)
    x = torch.randn(M, K, device=dev).bfloat16()
    y = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
    a = L.Q4LinearArgs(x=x.data_ptr(), ldx=K, qw_tiled=qt.data_ptr(), scales=sc.data_ptr(), zeros=z.data_ptr(), sz_dtype=L.sz_dtype_of(sc),
                       y=y.data_ptr(), ldy=N, M=M, N=N, K=K, prologue=0, norm_scale=None, eps=0.0, epilogue=0, res=None, ldres=0,
                       split_k=0, flags=0)
    rc = L.lib().b2l_q4_gemm(C.byref(a), L.stream_ptr())
    assert rc == 0, L.lib().b2l_last_error()
    torch.cuda.synchronize()
    wb = ((lv.to(torch.bfloat16) - z.to(torch.bfloat16)) * sc.to(torch.bfloat16))     # get_weight(bf16), quantization.py:398-410
    want = x.float() @ wb.float().t()
    # fp32 accumulation of exact bf16 products in a different order + one bf16 rounding of the result
    assert relerr(y, want.double()) < 2.0 ** -9, relerr(y, want.double())
    err = (y.float() - want).abs()
    mag = x.float().abs() @ wb.float().abs().t()
    assert bool((err <= want.abs() * 2.0 ** -8 + mag * 2.0 ** -20 + 1e-30).all()), float((err / (want.abs() * 2.0 ** -8 + mag * 2.0 ** -20 + 1e-30)).max())
    assert float((y == want.bfloat16()).float().mean()) > 0.98
    if M * N <= 4096 * 5120:   # and through the module: forward() takes this kernel for M > 16
        from lit_llama_b200.quantization import ColBlockQuantizedLinear
        lin = ColBlockQuantizedLinear(K, N, bias=False, bits=4, tile_cols=-1).to(dev)
        lin.quant_weight.copy_(qw); lin.scales = sc.clone(); lin.zeros = z.clone()
        assert torch.equal(lin(x), y)
        assert torch.equal(lin.get_weight(torch.bfloat16), wb)


@pytest.mark.parametrize("name,N,K", [("c_attn", 12288, 4096), ("c_proj", 4096, 4096), ("c_fc12", 22016, 4096),
                                      ("mlp_proj", 4096, 11008), ("lm_head", 32000, 4096)])
def test_tc_linear_7b_shapes(dev, name, N, K):
    """Full BASELINE sizes: agreement with fp64 math, with the independent generic kernel,
    and linearity y(a+b) = y(a) + y(b) (size-independent property)."""
    from gpu_util import rand_q4, ref_linear, relerr, tc_call, tile
    from lit_llama_b200 import _lib as L

    lv, qw, sc, z = rand_q4(N, K, dev, seed=7)
    qt = tile(L, qw, N, K)
    x = torch.randn(2, K, device=dev).bfloat16()
    y, err = tc_call(L, x, qt, sc, z, N, K)
    assert err is None, err
    want = ref_linear(x, lv, sc, z)
    assert relerr(y, want) < 1e-3 + 2.0 ** -9
    # the batch-1 kernel on the same weights: same exact-arithmetic target
    from gpu_util import gemv_call, tile_i8
    y1, err = gemv_call(L, x[0:1], tile_i8(L, qw, N, K), sc, z, N, K)
    assert err is None, err
    assert relerr(y1, want[0:1]) < 1e-3 + 2.0 ** -9
    # two independent kernels: same bf16 results up to 1-ulp flips (the tcgen05 kernel accumulates (128 + level) * x
    # in fp32, the batch-1 kernel is exact: a percent or two of outputs sit on the other side of a rounding boundary)
    assert float((y1 == want[0:1].float().bfloat16()).float().mean()) > 0.995
    assert float((y1 == y[0:1]).float().mean()) > 0.9
    assert relerr(y1, y[0:1]) < 2.0 ** -9
    yg = torch.empty(2, N, device=dev, dtype=torch.bfloat16)
    rc = L.lib().b2l_q_linear(x.data_ptr(), K, qw.data_ptr(), sc.data_ptr(), z.data_ptr(), L.sz_dtype_of(sc), None, yg.data_ptr(), N, 2, N, K, 4, K, L.stream_ptr())
    assert rc == 0
    assert relerr(y, yg) < 3e-3
    xs = (x[0:1].float() + x[1:2].float()).bfloat16()
    ys, err = tc_call(L, xs, qt, sc, z, N, K)
    assert err is None
    lin = ref_linear(xs, lv, sc, z)
    assert relerr(ys, lin) < 1e-3 + 2.0 ** -9


def test_tc_prologue_epilogue(dev):
    from gpu_util import rand_q4, ref_linear, relerr, tc_call, tile
    from lit_llama_b200 import _lib as L

    N, K, M = 512, 1024, 2
    lv, qw, sc, z = rand_q4(N, K, dev, seed=5)
    qt = tile(L, qw, N, K)
    x = (torch.randn(M, K, device=dev) * 0.7).bfloat16()
    g = (1 + 0.1 * torch.randn(K, device=dev)).bfloat16()
    # the reference formula (model.py:270-277) in bf16 on this device (torch's CPU mean double-rounds, see test_gpu_model)
    xn = g * (x * torch.rsqrt(torch.mean(x * x, dim=-1, keepdim=True) + 1e-5))
    y, err = tc_call(L, x, qt, sc, z, N, K, prologue=1, norm_scale=g, eps=1e-5)
    assert err is None, err
    assert relerr(y, ref_linear(xn, lv, sc, z)) < 1e-3 + 2.0 ** -9
    res = torch.randn(M, N, device=dev).bfloat16()
    y, err = tc_call(L, x, qt, sc, z, N, K, epilogue=1, res=res)
    assert err is None, err
    want = ref_linear(x, lv, sc, z).float().bfloat16() + res
    assert float((y == want).float().mean()) > 0.98 and relerr(y, want) < 2e-3
    buf = res.clone()
    _, err = tc_call(L, x, qt, sc, z, N, K, epilogue=1, res=buf, y=buf)
    assert err is None and torch.equal(buf, y)
    full = ref_linear(x, lv, sc, z).float().bfloat16().reshape(M, N // 128, 2, 64)
    a, b = full[:, :, 0].reshape(M, -1), full[:, :, 1].reshape(M, -1)
    want = torch.nn.functional.silu(a) * b
    y, err = tc_call(L, x, qt, sc, z, N, K, epilogue=2, n_out=N // 2)
    assert err is None, err
    assert relerr(y, want) < 4e-3 and float((y == want).float().mean()) > 0.9


def test_unsupported_shapes_raise(dev):
    from lit_llama_b200.quantization import ColBlockQuantizedLinear

    lin = ColBlockQuantizedLinear(64, 16, False, bits=4, tile_cols=-1).to(dev)
    with pytest.raises(RuntimeError):
        lin(torch.zeros(1, 64, device=dev))  # fp32 activations: no silent fallback
    with pytest.raises(RuntimeError):
        lin(torch.zeros(1, 64, dtype=torch.bfloat16))  # CPU tensor


@pytest.mark.parametrize("N,K,M,outliers", [(48, 256, 1, 0), (48, 256, 1, 3), (130, 1024, 3, 2), (4096, 4096, 1, 0), (4096, 4096, 1, 5),
                                           (4096, 11008, 2, 1), (32000, 4096, 1, 0)])
def test_int8_linear_vs_oracle(dev, N, K, M, outliers):
    """Linear8bitLt (LLM.int8) through the C ABI vs the oracle restatement, with and without
    outlier columns (|a| >= 6), batch-shared outlier mask for M > 1.  Parity unpinned (bitsandbytes
    is not available): this checks the CUDA path against the published algorithm only."""
    import lit_llama_b200 as P

    g = torch.Generator().manual_seed(N + K + M + outliers)
    w = torch.randn(N, K, generator=g) * 0.03
    x = torch.randn(M, K, generator=g)
    for i in range(outliers):
        x[i % M, (37 * i + 11) % K] = 7.5 + i
    lin = P.Linear8bitLt(K, N, bias=False)
    lin.load_state_dict({"weight": w})
    cb, scb = O.int8_quantize_weight(w)
    assert torch.equal(lin.weight.CB, cb) and torch.equal(lin.weight.SCB, scb)
    lin = lin.to(dev)
    xb = x.bfloat16()
    y = lin(xb.to(dev)).float().cpu()
    want = O.int8_linear(xb, cb, scb).float()
    exact = xb.float() @ w.t()
    assert (y - want).norm() / want.norm() < 2e-3, float((y - want).norm() / want.norm())
    torch.testing.assert_close(y, want, rtol=2 ** -6, atol=2e-2 * float(want.abs().max()) * 0.1 + 1e-3)
    assert (y - exact).norm() / exact.norm() < 3e-2  # the int8 scheme itself is ~1% accurate


@pytest.mark.parametrize("n", [4096, 8192, 130])
def test_tp_allreduce_single_rank_is_identity(dev, n):
    """b2l_tp_allreduce with world = 1 (no peers): the multi-CTA indexing, the in-place path and the epoch words that
    advance in device memory -- the sum of one row is that row.  The peer exchange itself needs 2 GPUs
    (tests/test_gpu_decode.py::test_tensor_parallel_matches_single_gpu)."""
    import ctypes as C

    from lit_llama_b200 import _lib as L

    lib = L.lib()
    buf = torch.zeros(lib.b2l_tp_buffer_bytes(1, 8192), dtype=torch.uint8, device=dev)
    words = torch.zeros(32, dtype=torch.int32, device=dev)
    comm = L.TPComm()
    comm.peer_buf[0] = buf.data_ptr()
    comm.rank, comm.world, comm.max_elems = 0, 1, 8192
    comm.epoch, comm.status = words.data_ptr(), words.data_ptr() + 64
    x = torch.randn(n, device=dev).bfloat16()
    y = torch.empty_like(x)
    for step in range(3):
        L.check(lib.b2l_tp_allreduce(C.byref(comm), x.data_ptr(), y.data_ptr(), n, 0, L.stream_ptr()), "b2l_tp_allreduce")
        assert torch.equal(x, y)
    z = x.clone()
    L.check(lib.b2l_tp_allreduce(C.byref(comm), z.data_ptr(), z.data_ptr(), n, L.F_PDL, L.stream_ptr()), "b2l_tp_allreduce")  # in place
    assert torch.equal(x, z)
    n_ctas = (n // 2 + 511) // 512
    assert words[:n_ctas].tolist() == [4] * n_ctas and int(words[16]) == 0
