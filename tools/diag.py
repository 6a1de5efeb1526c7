"""GPU diagnostics: exercises every kernel against torch math and PRINTS errors instead
of asserting, section by section, each in its own subprocess with a timeout (a hung
kernel only loses its section).  Usage on the GPU box:

    python tools/diag.py            # all sections
    python tools/diag.py tc_small   # one section
"""
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SECTIONS = ["generic", "tile", "tc_small", "tc_shapes", "tc_modes", "gemv", "mma_rate", "mma_issuers", "grid_flag", "hmma_rate", "imma_rate", "consumer_rate", "bench_gemm", "trace", "bench_layers", "bench_gemv", "bench_step", "bench_ctx", "bench_13b_b8", "bench_sizes", "batch_debug", "bench_step_int8", "timeline"]


_DLIB = None


def dlib():
    """tools/libb200diag.so (include/b2l_diag.h): the micro-benchmarks live outside the product library."""
    global _DLIB
    if _DLIB is None:
        h = C.CDLL(os.path.join(ROOT, "tools", "libb200diag.so"))
        vp, ci = C.c_void_p, C.c_int
        for name, args in {"b2l_debug_mma_rate": [vp, ci, ci, ci, ci, vp], "b2l_debug_mma_issuers": [vp, ci, ci, vp],
                           "b2l_debug_grid_flag": [vp, vp, ci, ci, vp], "b2l_debug_hmma_rate": [vp, ci, ci, ci, ci, vp],
                           "b2l_debug_imma_rate": [vp, ci, ci, ci, ci, vp],
                           "b2l_debug_consumer_rate": [vp, ci, ci, ci, ci, vp]}.items():
            getattr(h, name).restype = ci
            getattr(h, name).argtypes = args
        h.b2l_diag_last_error.restype = C.c_char_p
        _DLIB = h
    return _DLIB


def dcheck(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {dlib().b2l_diag_last_error().decode()}")


def rand_q4(N, K, dev, seed=0, sz_dtype=None, groups=1, bits=4):
    import torch

    g = torch.Generator(device="cpu").manual_seed(seed)
    sz_dtype = sz_dtype or torch.bfloat16
    maxq = 2**bits - 1
    lv = torch.randint(0, maxq + 1, (N, K), generator=g, dtype=torch.uint8)
    epb = 8 // bits
    qw = torch.zeros((N, K // epb), dtype=torch.uint8)
    for nr in range(epb):
        qw |= lv[:, nr::epb] << (nr * bits)
    qw = qw.t().contiguous().t()
    scales = (torch.rand(N, groups, generator=g) * 0.01 + 0.002).to(sz_dtype)
    zeros = torch.randint(0, maxq + 1, (N, groups), generator=g).to(sz_dtype)
    return lv.to(dev), qw.to(dev), scales.to(dev), zeros.to(dev)


def ref_linear(x, lv, scales, zeros, tile_cols=None):
    import torch

    N, K = lv.shape
    tc = K if tile_cols is None else tile_cols
    ng = scales.shape[1]
    w = lv.double()
    for g in range(ng):
        sl = slice(g * tc, (g + 1) * tc)
        w[:, sl] = (w[:, sl] - zeros[:, g : g + 1].double()) * scales[:, g : g + 1].double()
    return (x.double() @ w.t())


def relerr(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


def tc_call(L, x, qt, scales, zeros, N, K, *, y=None, prologue=0, norm_scale=None, eps=1e-5, epilogue=0, res=None,
            split_k=0, flags=0, n_out=None):
    import torch

    M = x.shape[0]
    n_out = n_out or N
    if y is None:
        y = torch.zeros((M, n_out), device=x.device, dtype=torch.bfloat16)
    a = L.Q4LinearArgs(x=x.data_ptr(), ldx=x.stride(0), qw_tiled=qt.data_ptr(), scales=scales.data_ptr(),
                       zeros=zeros.data_ptr(), sz_dtype=L.sz_dtype_of(scales), y=y.data_ptr(), ldy=y.stride(0), M=M, N=N,
                       K=K, prologue=prologue, norm_scale=None if norm_scale is None else norm_scale.data_ptr(),
                       eps=eps, epilogue=epilogue, res=None if res is None else res.data_ptr(),
                       ldres=0 if res is None else res.stride(0), split_k=split_k, flags=flags)
    rc = L.lib().b2l_q4_linear_tc(C.byref(a), L.stream_ptr())
    if rc != 0:
        return None, f"rc={rc}: {L.lib().b2l_last_error().decode()}"
    return y, None


def tile(L, qw, N, K):
    import torch

    qt = torch.empty(L.lib().b2l_q4_tiled_bytes(N, K), dtype=torch.uint8, device=qw.device)
    L.check(L.lib().b2l_q4_tile(qw.data_ptr(), qt.data_ptr(), N, K, L.stream_ptr()), "tile")
    return qt


def tile_mma(L, qw, N, K):
    import torch

    qt = torch.empty(L.lib().b2l_q4_tiled_mma_bytes(N, K), dtype=torch.uint8, device=qw.device)
    L.check(L.lib().b2l_q4_tile_mma(qw.data_ptr(), qt.data_ptr(), N, K, L.stream_ptr()), "tile_mma")
    return qt


def tile_i8(L, qw, N, K):
    import torch

    qt = torch.empty(L.lib().b2l_q4_tiled_i8_bytes(N, K), dtype=torch.uint8, device=qw.device)
    L.check(L.lib().b2l_q4_tile_i8(qw.data_ptr(), qt.data_ptr(), N, K, L.stream_ptr()), "tile_i8")
    return qt


def gemv_call(L, x, qt, scales, zeros, N, K, *, y=None, prologue=0, norm_scale=None, eps=1e-5, epilogue=0, res=None, grid=0,
              flags=0, n_out=None):
    import torch

    n_out = n_out or N
    if y is None:
        y = torch.zeros((1, n_out), device=x.device, dtype=torch.bfloat16)
    a = L.Q4LinearArgs(x=x.data_ptr(), ldx=K, qw_tiled=qt.data_ptr(), scales=scales.data_ptr(), zeros=zeros.data_ptr(),
                       sz_dtype=L.sz_dtype_of(scales), y=y.data_ptr(), ldy=n_out, M=1, N=N, K=K, prologue=prologue,
                       norm_scale=None if norm_scale is None else norm_scale.data_ptr(), eps=eps, epilogue=epilogue,
                       res=None if res is None else res.data_ptr(), ldres=N, split_k=grid, flags=flags)
    rc = L.lib().b2l_q4_gemv(C.byref(a), L.stream_ptr())
    if rc != 0:
        return None, f"rc={rc}: {L.lib().b2l_last_error().decode()}"
    return y, None


def gemv_batch_call(L, x, qt, scales, zeros, N, K, *, y=None, prologue=0, norm_scale=None, eps=1e-5, epilogue=0, res=None, grid=0,
                    flags=0, n_out=None):
    """b2l_q4_gemv_batch on x (M, K), M <= 8."""
    import torch

    M = x.shape[0]
    n_out = n_out or N
    if y is None:
        y = torch.zeros((M, n_out), device=x.device, dtype=torch.bfloat16)
    ws = torch.zeros(L.lib().b2l_q4_gemv_batch_workspace_bytes(K), dtype=torch.uint8, device=x.device)
    a = L.Q4LinearArgs(x=x.data_ptr(), ldx=x.stride(0), qw_tiled=qt.data_ptr(), scales=scales.data_ptr(), zeros=zeros.data_ptr(),
                       sz_dtype=L.sz_dtype_of(scales), y=y.data_ptr(), ldy=n_out, M=M, N=N, K=K, prologue=prologue,
                       norm_scale=None if norm_scale is None else norm_scale.data_ptr(), eps=eps, epilogue=epilogue,
                       res=None if res is None else res.data_ptr(), ldres=N, split_k=grid, flags=flags, workspace=ws.data_ptr())
    rc = L.lib().b2l_q4_gemv_batch(C.byref(a), L.stream_ptr())
    if rc != 0:
        return None, f"rc={rc}: {L.lib().b2l_last_error().decode()}"
    torch.cuda.synchronize()
    return y, None


def sec_gemv():
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    for (N, K, grid) in [(16, 64, 0), (16, 128, 0), (32, 2048, 0), (48, 4096, 0), (130, 256, 0), (4096, 4096, 0), (4096, 4096, 7),
                         (12288, 4096, 0), (4096, 11008, 0), (32000, 4096, 0), (22016, 4096, 0), (128, 6400, 0)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=N + K)
        qt = tile_i8(L, qw, N, K)
        back = torch.empty_like(qw)
        L.check(L.lib().b2l_q4_untile_i8(qt.data_ptr(), back.data_ptr(), N, K, L.stream_ptr()), "untile_i8")
        x = torch.randn(1, K, device=dev).bfloat16()
        y, err = gemv_call(L, x, qt, sc, z, N, K, grid=grid)
        torch.cuda.synchronize()
        if err:
            print(f"gemv N={N} K={K} grid={grid}: {err}")
            continue
        want = ref_linear(x, lv, sc, z)
        wb = want.float().bfloat16()
        print(f"gemv N={N} K={K} grid={grid}: roundtrip={bool(torch.equal(back, qw))} relerr={relerr(y, want):.3e} "
              f"exact_bf16_frac={float((y == wb).float().mean()):.4f}")
        if N == 16 and K == 64:
            print("   got ", [round(float(v), 4) for v in y[0, :8]])
            print("   want", [round(float(v), 4) for v in want[0, :8]])
    N, K = 512, 1024
    lv, qw, sc, z = rand_q4(N, K, dev, seed=5)
    qt = tile_i8(L, qw, N, K)
    x = (torch.randn(1, K, device=dev) * 0.7).bfloat16()
    g = (1 + 0.1 * torch.randn(K, device=dev)).bfloat16()
    ms = torch.mean(x * x, dim=-1, keepdim=True)
    xn = g * (x * torch.rsqrt(ms + 1e-5))
    y, err = gemv_call(L, x, qt, sc, z, N, K, prologue=1, norm_scale=g)
    torch.cuda.synchronize()
    print("gemv rmsnorm prologue:", err or f"relerr={relerr(y, ref_linear(xn, lv, sc, z)):.3e}")
    res = torch.randn(1, N, device=dev).bfloat16()
    y, err = gemv_call(L, x, qt, sc, z, N, K, epilogue=1, res=res)
    torch.cuda.synchronize()
    want = (ref_linear(x, lv, sc, z).float().bfloat16() + res)
    print("gemv residual:", err or f"relerr={relerr(y, want):.3e} exact={float((y == want).float().mean()):.4f}")
    buf = res.clone()
    y, err = gemv_call(L, x, qt, sc, z, N, K, epilogue=1, res=buf, y=buf)
    torch.cuda.synchronize()
    print("gemv in-place residual:", err or f"relerr={relerr(buf, want):.3e}")
    full = ref_linear(x, lv, sc, z).float().bfloat16().reshape(1, N // 16, 2, 8)
    a, b = full[:, :, 0].reshape(1, -1), full[:, :, 1].reshape(1, -1)
    want = torch.nn.functional.silu(a) * b
    y, err = gemv_call(L, x, qt, sc, z, N, K, epilogue=2, n_out=N // 2)
    torch.cuda.synchronize()
    print("gemv swiglu:", err or f"relerr={relerr(y, want):.3e} exact={float((y == want).float().mean()):.4f}")
    y, err = gemv_call(L, x, qt, sc, z, N, K, flags=1)
    torch.cuda.synchronize()
    print("gemv pdl flag:", err or f"relerr={relerr(y, ref_linear(x, lv, sc, z)):.3e}")


def sec_bench_gemv():
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    lib = L.lib()
    for (name, N, K) in [("c_attn", 12288, 4096), ("c_proj", 4096, 4096), ("fc12", 22016, 4096), ("mlp_proj", 4096, 11008), ("lm_head", 32000, 4096)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=3)
        n_copies = max(4, int(400e6 // (N * K // 2)) + 1)
        qts = [tile_i8(L, qw, N, K) for _ in range(n_copies)]
        x = torch.randn(1, K, device=dev).bfloat16()
        y = torch.zeros(1, N, device=dev, dtype=torch.bfloat16)
        for grid in (0,):
            for flags in (1, 17):
                args = [L.Q4LinearArgs(x=x.data_ptr(), ldx=K, qw_tiled=qt.data_ptr(), scales=sc.data_ptr(), zeros=z.data_ptr(),
                                       sz_dtype=0, y=y.data_ptr(), ldy=N, M=1, N=N, K=K, prologue=0, norm_scale=None, eps=1e-5,
                                       epilogue=0, res=None, ldres=N, split_k=grid, flags=flags) for qt in qts]
                if lib.b2l_q4_gemv(C.byref(args[0]), L.stream_ptr()) != 0:
                    print(f"{name} grid={grid}: {lib.b2l_last_error().decode()[:90]}")
                    continue
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for a in args:
                        lib.b2l_q4_gemv(C.byref(a), L.stream_ptr())
                us = _time(g.replay, iters=10, warm=2) / n_copies
                print(f"gemv {name} N={N} K={K} grid={grid or 296} pdl={flags}: {us:.2f} us/launch  {(N * K / 2) / us / 1e3:.0f} GB/s")
        del qts


def sec_generic():
    import torch
    from lit_llama_b200 import _lib as L
    from lit_llama_b200.quantization import ColBlockQuantizedLinear

    dev = torch.device("cuda")
    for bits, groups, N, K, M in [(4, 1, 24, 64, 3), (4, 4, 24, 128, 1), (8, 1, 16, 64, 5), (8, 3, 8, 96, 2), (4, 1, 130, 256, 1),
                                  (4, 1, 4096, 4096, 1), (4, 1, 12288, 4096, 2)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=bits + N, groups=groups, bits=bits)
        tc = K // groups
        lin = ColBlockQuantizedLinear(K, N, False, bits=bits, tile_cols=tc if groups > 1 else -1).to(dev)
        lin.quant_weight.copy_(qw); lin.scales = sc; lin.zeros = z
        x = torch.randn(M, K, device=dev).bfloat16()
        y = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        rc = L.lib().b2l_q_linear(x.data_ptr(), K, lin.quant_weight.data_ptr(), sc.data_ptr(), z.data_ptr(), L.sz_dtype_of(sc), None,
                                  y.data_ptr(), N, M, N, K, bits, tc, L.stream_ptr())
        torch.cuda.synchronize()
        want = ref_linear(x, lv, sc, z, tc)
        print(f"generic bits={bits} groups={groups} N={N} K={K} M={M}: rc={rc} relerr={relerr(y, want):.2e}")
        for dt in (torch.float32, torch.bfloat16):
            w = lin.get_weight(dt)
            wr = lv.float().to(dt)
            for g in range(groups):
                sl = slice(g * tc, (g + 1) * tc)
                wr[:, sl] -= z[:, g : g + 1]
                wr[:, sl] *= sc[:, g : g + 1]
            print(f"   dequant {dt}: bit-exact={bool(torch.equal(w, wr))}")


def sec_tile():
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    for N, K in [(128, 64), (130, 256), (4096, 4096), (96, 128)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=N)
        qt = tile(L, qw, N, K)
        back = torch.empty_like(qw)
        L.check(L.lib().b2l_q4_untile(qt.data_ptr(), back.data_ptr(), N, K, L.stream_ptr()), "untile")
        torch.cuda.synchronize()
        # independent check of the documented layout on the host
        w = qt.view(torch.int32).reshape(-1, K // 32, 128, 4).cpu()
        lvc = lv.cpu()
        ok = True
        for (nt, ks, r, i) in [(0, 0, 0, 0), (0, K // 32 - 1, 5, 3), ((N - 1) // 128, 1 % (K // 32), (N - 1) % 128, 2)]:
            word = int(w[nt, ks, r, i]) & 0xFFFFFFFF
            o = nt * 128 + r
            for s in range(8):
                k = ks * 32 + 8 * i + (2 * s if s < 4 else 2 * (s - 4) + 1)
                ok &= ((word >> (4 * s)) & 0xF) == int(lvc[o, k])
        print(f"tile N={N} K={K}: roundtrip={bool(torch.equal(back, qw))} layout_spot={ok}")


def sec_tc_small():
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    N, K, M = 128, 64, 1
    lv, qw, sc, z = rand_q4(N, K, dev, seed=1)
    qt = tile(L, qw, N, K)
    x = torch.randn(M, K, device=dev).bfloat16()
    y, err = tc_call(L, x, qt, sc, z, N, K, split_k=1)
    torch.cuda.synchronize()
    print("tc_small first call:", err or "launched")
    want = ref_linear(x, lv, sc, z)
    print(f"  N=128 K=64 M=1 S=1 relerr={relerr(y, want):.3e}")
    print("  got ", [round(float(v), 4) for v in y[0, :6]])
    print("  want", [round(float(v), 4) for v in want[0, :6]])
    # hypotheses if wrong: pair order swapped inside a TMEM column / B rows
    xs = x.clone().reshape(M, K // 2, 2).flip(-1).reshape(M, K)
    print(f"  hypothesis pair-swapped relerr={relerr(y, ref_linear(xs, lv, sc, z)):.3e}")
    xh = x.clone().reshape(M, K // 16, 2, 8).flip(2).reshape(M, K)
    print(f"  hypothesis k-halves-swapped relerr={relerr(y, ref_linear(xh, lv, sc, z)):.3e}")
    for (N, K, M, S) in [(128, 64, 1, 1), (128, 128, 1, 1), (128, 256, 3, 1), (128, 256, 1, 2), (256, 512, 1, 4), (256, 1024, 8, 8),
                         (128, 96, 1, 1), (384, 4096, 1, 4), (130, 256, 2, 2), (128, 1024, 16, 2), (128, 1024, 9, 2)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=N + K)
        qt = tile(L, qw, N, K)
        x = torch.randn(M, K, device=dev).bfloat16()
        for flags in (0, 2):
            if flags == 2 and M > 8:
                continue
            y, err = tc_call(L, x, qt, sc, z, N, K, split_k=S, flags=flags)
            torch.cuda.synchronize()
            if err:
                print(f"  N={N} K={K} M={M} S={S} flags={flags}: {err}")
                continue
            want = ref_linear(x, lv, sc, z)
            wb = want.float().bfloat16()
            print(f"  N={N} K={K} M={M} S={S} flags={flags}: relerr={relerr(y, want):.3e} exact_bf16_frac={float((y == wb).float().mean()):.4f}")


def sec_tc_shapes():
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    for (N, K) in [(12288, 4096), (4096, 4096), (22016, 4096), (4096, 11008), (32000, 4096)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=N % 1000 + K)
        qt = tile(L, qw, N, K)
        for M in (1, 8):
            x = torch.randn(M, K, device=dev).bfloat16()
            for S in (0, 1, 2, 4, 8):
                y, err = tc_call(L, x, qt, sc, z, N, K, split_k=S)
                torch.cuda.synchronize()
                if err:
                    print(f"  N={N} K={K} M={M} S={S}: {err}")
                    continue
                want = ref_linear(x, lv, sc, z)
                print(f"  N={N} K={K} M={M} S={S}: relerr={relerr(y, want):.3e}")
        del lv, qw, qt


def sec_tc_modes():
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    N, K, M = 512, 1024, 2
    lv, qw, sc, z = rand_q4(N, K, dev, seed=5)
    qt = tile(L, qw, N, K)
    x = (torch.randn(M, K, device=dev) * 0.7).bfloat16()
    g = (1 + 0.1 * torch.randn(K, device=dev)).bfloat16()
    # rmsnorm prologue (bf16 rounding points of model.py:270-277 via torch bf16 ops)
    ms = torch.mean(x * x, dim=-1, keepdim=True)
    xn = g * (x * torch.rsqrt(ms + 1e-5))
    y, err = tc_call(L, x, qt, sc, z, N, K, prologue=1, norm_scale=g, eps=1e-5)
    torch.cuda.synchronize()
    print("rmsnorm prologue:", err or f"relerr={relerr(y, ref_linear(xn, lv, sc, z)):.3e}")
    # residual epilogue
    res = torch.randn(M, N, device=dev).bfloat16()
    y, err = tc_call(L, x, qt, sc, z, N, K, epilogue=1, res=res)
    torch.cuda.synchronize()
    want = (ref_linear(x, lv, sc, z).float().bfloat16() + res)
    print("residual epilogue:", err or f"relerr={relerr(y, want):.3e} exact={float((y == want).float().mean()):.4f}")
    # in-place residual
    buf = res.clone()
    y, err = tc_call(L, x, qt, sc, z, N, K, epilogue=1, res=buf, y=buf)
    torch.cuda.synchronize()
    print("in-place residual:", err or f"relerr={relerr(buf, want):.3e}")
    # swiglu: rows interleaved [64 a | 64 b]
    full = ref_linear(x, lv, sc, z).float().bfloat16().reshape(M, N // 128, 2, 64)
    a, b = full[:, :, 0].reshape(M, -1), full[:, :, 1].reshape(M, -1)
    want = torch.nn.functional.silu(a) * b
    y, err = tc_call(L, x, qt, sc, z, N, K, epilogue=2, n_out=N // 2)
    torch.cuda.synchronize()
    print("swiglu epilogue:", err or f"relerr={relerr(y, want):.3e} exact={float((y == want).float().mean()):.4f}")
    # pdl flag outside a chain
    y, err = tc_call(L, x, qt, sc, z, N, K, flags=1)
    torch.cuda.synchronize()
    print("pdl flag:", err or f"relerr={relerr(y, ref_linear(x, lv, sc, z)):.3e}")
    # fp32 scales/zeros
    lv, qw, sc, z = rand_q4(N, K, dev, seed=6, sz_dtype=torch.float32)
    qt = tile(L, qw, N, K)
    y, err = tc_call(L, x, qt, sc, z, N, K)
    torch.cuda.synchronize()
    print("fp32 scales:", err or f"relerr={relerr(y, ref_linear(x, lv, sc, z)):.3e}")


def _time(fn, iters=20, warm=3):
    import torch

    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


def make_args(L, x, qt, scales, zeros, N, K, y, *, prologue=0, norm_scale=None, epilogue=0, res=None, split_k=0, flags=0, trace=None):
    return L.Q4LinearArgs(x=x.data_ptr(), ldx=x.stride(0), qw_tiled=qt.data_ptr(), scales=scales.data_ptr(),
                          zeros=zeros.data_ptr(), sz_dtype=L.sz_dtype_of(scales), y=y.data_ptr(), ldy=y.stride(0), M=x.shape[0], N=N,
                          K=K, prologue=prologue, norm_scale=None if norm_scale is None else norm_scale.data_ptr(), eps=1e-5,
                          epilogue=epilogue, res=None if res is None else res.data_ptr(), ldres=0 if res is None else res.stride(0),
                          split_k=split_k, flags=flags, trace=None if trace is None else trace.data_ptr())


def sec_mma_rate():
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    out = torch.zeros(64 * 3, dtype=torch.int64, device=dev)
    for a_smem in (0, 1):
        for n_acc in (1, 4):
            for n_mma in (1, 4, 16):
                out.zero_()
                dcheck(dlib().b2l_debug_mma_rate(out.data_ptr(), n_mma, n_acc, a_smem, 8, L.stream_ptr()), "mma_rate")
                torch.cuda.synchronize()
                o = out.cpu().reshape(-1, 3)[:8]
                r = o[3:].float().mean(0)  # skip cold rounds
                print(f"A_from_{'smem' if a_smem else 'tmem'} n_acc={n_acc} n_mma={n_mma:3d}: issue={r[0]:.0f} cyc ({r[0] / n_mma:.1f}/mma) "
                      f"commit_issue={r[1]:.0f} total_until_arrive={r[2]:.0f} ({r[2] / n_mma:.1f}/mma)")


def sec_mma_issuers():
    """tcgen05.mma issue from 1..4 threads of one CTA at once (round-2 question: does a multi-issuer kernel scale?)."""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    rounds = 6
    out = torch.zeros(rounds * 8, dtype=torch.int64, device=dev)
    for n in (1, 2, 3, 4):
        out.zero_()
        dcheck(dlib().b2l_debug_mma_issuers(out.data_ptr(), n, rounds, L.stream_ptr()), "mma_issuers")
        torch.cuda.synchronize()
        o = out.view(rounds, 8).cpu()
        print(f"issuers={n}: last round, cycles until commit per warp {o[-1, :n].tolist()}  issue cycles {o[-1, 4:4 + n].tolist()}  "
              f"-> {float(o[-1, :n].max()) / (16 * n):.1f} cycles per MMA overall", flush=True)


def sec_grid_flag():
    """Grid-wide arrive-and-wait through a global counter: the cost of a dependency without a kernel boundary."""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    rounds = 16
    for cps in (1, 2):
        out = torch.zeros(2 * rounds, dtype=torch.int64, device=dev)
        out[rounds:] = 2**62
        counter = torch.zeros(1, dtype=torch.int32, device=dev)
        dcheck(dlib().b2l_debug_grid_flag(out.data_ptr(), counter.data_ptr(), cps, rounds, L.stream_ptr()), "grid_flag")
        torch.cuda.synchronize()
        o = out.cpu()
        print(f"ctas_per_sm={cps}: arrive-and-wait ns per round, max over CTAs {o[:rounds].tolist()}  min {o[rounds:].tolist()}", flush=True)


def sec_hmma_rate():
    """Legacy tensor pipe: cycles per mma.sync.m16n8k16 per SM sub-partition, by warps / chains / unpack."""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    out = torch.zeros(2, dtype=torch.int64, device=dev)
    iters = 512
    for unpack in (0, 1):
        for warps in (4, 8, 16, 20):
            for chains in (1, 2, 4, 8):
                dcheck(dlib().b2l_debug_hmma_rate(out.data_ptr(), warps, chains, iters, unpack, L.stream_ptr()), "hmma_rate")
                torch.cuda.synchronize()
                dcheck(dlib().b2l_debug_hmma_rate(out.data_ptr(), warps, chains, iters, unpack, L.stream_ptr()), "hmma_rate")
                torch.cuda.synchronize()
                cyc = int(out[0])
                per_smsp = (warps / 4) * iters * 8
                print(f"unpack={unpack} warps={warps:2d} chains={chains}: {cyc} cycles, {cyc / (iters * 8):.1f} clk per MMA per warp, "
                      f"{cyc / per_smsp:.2f} clk per MMA per sub-partition", flush=True)


def sec_imma_rate():
    """Legacy integer tensor pipe: cycles per mma.sync.m16n8k32 (u8 x s8) per SM sub-partition, by warps / chains / ALU ops."""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    out = torch.zeros(2, dtype=torch.int64, device=dev)
    iters = 512
    for n_alu in (0, 2, 4):
        for warps in (4, 8, 16, 20):
            for chains in (1, 2, 4, 8):
                for _ in range(2):
                    dcheck(dlib().b2l_debug_imma_rate(out.data_ptr(), warps, chains, iters, n_alu, L.stream_ptr()), "imma_rate")
                    torch.cuda.synchronize()
                cyc = int(out[0])
                per_smsp = (warps / 4) * iters * 8
                print(f"n_alu={n_alu} warps={warps:2d} chains={chains}: {cyc} cycles, {cyc / (iters * 8):.1f} clk per MMA per warp, "
                      f"{cyc / per_smsp:.2f} clk per MMA per sub-partition", flush=True)


def sec_consumer_rate():
    """The decode consumer loop on shared-memory-resident stages: what bounds it -- LDS, IMMA issue, or their sum?"""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    out = torch.zeros(2, dtype=torch.int64, device=dev)
    iters = 200
    names = {1: "weights LDS", 2: "digit LDS", 3: "both LDS", 4: "IMMA only", 5: "weights LDS + IMMA", 7: "all", 15: "all, unused lanes predicated off",
             13: "weights LDS + IMMA + (digits off)"}
    for warps in (16, 8):
        for ctas in (1, 148):
            for mode in (1, 2, 3, 4, 5, 7, 15):
                for _ in range(2):
                    dcheck(dlib().b2l_debug_consumer_rate(out.data_ptr(), warps, iters, mode, ctas, L.stream_ptr()), "consumer_rate")
                    torch.cuda.synchronize()
                cyc = int(out[0]) / (iters * 8)
                print(f"warps={warps:2d} ctas={ctas:3d} mode={mode:2d} ({names.get(mode, '')}): {cyc:.0f} cycles per 16 KB stage  "
                      f"-> {16384 / cyc:.1f} B/clk/SM = {16384 / cyc * 1.965 * 148 / 1e3:.1f} TB/s-equivalent", flush=True)


def sec_bench_gemm():
    """The tcgen05 prefill GEMM at the 13B widths, M = 4096 (BASELINE configs[3] prefill 8 x 512), next to torch.matmul
    (library bf16 GEMM on a dense weight of the same shape) as the tensor-pipe yardstick."""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    M = int(os.environ.get("B2L_GEMM_M", "4096"))
    for (name, N, K) in [("c_attn", 15360, 5120), ("c_proj", 5120, 5120), ("fc1", 13824, 5120), ("mlp_proj", 5120, 13824), ("7B c_attn", 12288, 4096)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=3)
        qt = tile(L, qw, N, K)
        x = torch.randn(M, K, device=dev).bfloat16()
        y = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        a = L.Q4LinearArgs(x=x.data_ptr(), ldx=K, qw_tiled=qt.data_ptr(), scales=sc.data_ptr(), zeros=z.data_ptr(), sz_dtype=0, y=y.data_ptr(), ldy=N,
                           M=M, N=N, K=K, prologue=0, norm_scale=None, eps=0.0, epilogue=0, res=None, ldres=0, split_k=0, flags=0)
        fn = lambda: L.check(L.lib().b2l_q4_gemm(C.byref(a), L.stream_ptr()), "gemm")
        us = _time(fn, iters=10, warm=2)
        w = torch.randn(N, K, device=dev).bfloat16()
        us_t = _time(lambda: torch.matmul(x, w.t()), iters=10, warm=2)
        fl = 2.0 * M * N * K
        print(f"gemm {name} M={M} N={N} K={K}: {us:.0f} us = {fl / us / 1e6:.0f} TFLOP/s   | torch.matmul bf16: {us_t:.0f} us = {fl / us_t / 1e6:.0f} TFLOP/s", flush=True)


def sec_trace():
    """clock64 stamps of CTA 0 of one launch: where does a CTA spend its time?"""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    for (name, N, K, S) in [("c_attn", 12288, 4096, 4), ("c_proj", 4096, 4096, 8), ("mlp_proj", 4096, 11008, 8)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=3)
        qt = tile(L, qw, N, K)
        x = torch.randn(1, K, device=dev).bfloat16()
        g = torch.ones(K, device=dev, dtype=torch.bfloat16)
        y = torch.zeros(1, N, device=dev, dtype=torch.bfloat16)
        tr = torch.zeros(256, dtype=torch.int64, device=dev)
        a = make_args(L, x, qt, sc, z, N, K, y, prologue=1, norm_scale=g, split_k=S, trace=tr)
        for rep in range(2):  # second launch: weights of CTA 0 may be L2-warm, code is warm
            tr.zero_()
            flush = torch.empty(200 * 1024 * 1024, dtype=torch.uint8, device=dev).fill_(1)
            L.check(L.lib().b2l_q4_linear_tc(C.byref(a), L.stream_ptr()), "tc")
            torch.cuda.synchronize()
            t = tr.cpu().tolist()
            t0 = t[0]
            rel = lambda i: (t[i] - t0) if t[i] else None
            nst = (K // 32 // S + 1) // 2
            print(f"{name} S={S} rep={rep} stages={nst}: init_sync={rel(1)} pdl_wait={rel(2)} x_ready={rel(3)} d_full={rel(104)} "
                  f"csync1={rel(105)} epi={rel(106)} end={rel(107)}")
            k = min(nst, 20)
            print("   tma_issue ", [rel(108 + i) for i in range(k)])
            print("   w_full    ", [rel(4 + i) for i in range(k)])
            print("   a_empty   ", [rel(24 + i) for i in range(k)])
            print("   st_done   ", [rel(44 + i) for i in range(k)])
            print("   a_full@mma", [rel(64 + i) for i in range(k)])
            print("   commit    ", [rel(84 + i) for i in range(k)])
            del flush


def sec_bench_layers():
    """GPU time of the int4 linear per 7B shape: `n_copies` launches on distinct weight
    copies (> L2) captured in one CUDA graph, so the host cost of a launch is not in it."""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    lib = L.lib()
    for (name, N, K) in [("c_attn", 12288, 4096), ("c_proj", 4096, 4096), ("fc12", 22016, 4096), ("mlp_proj", 4096, 11008), ("lm_head", 32000, 4096)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=3)
        n_copies = max(4, int(400e6 // (N * K // 2)) + 1)
        qts = [tile(L, qw, N, K) for _ in range(n_copies)]
        x = torch.randn(1, K, device=dev).bfloat16()
        y = torch.zeros(1, N, device=dev, dtype=torch.bfloat16)
        for S in (0, 1, 2, 3, 4, 6, 8):
            for flags in (0,):
                args = [make_args(L, x, qt, sc, z, N, K, y, split_k=S, flags=flags) for qt in qts]
                if lib.b2l_q4_linear_tc(C.byref(args[0]), L.stream_ptr()) != 0:
                    print(f"{name} S={S} flags={flags}: {lib.b2l_last_error().decode()[:90]}")
                    continue
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for a in args:
                        lib.b2l_q4_linear_tc(C.byref(a), L.stream_ptr())
                us = _time(g.replay, iters=10, warm=2) / n_copies
                print(f"{name} N={N} K={K} S={S} flags={flags}: {us:.2f} us/launch  {(N * K / 2) / us / 1e3:.0f} GB/s  ({n_copies} launches/graph)")
        del qts


def sec_bench_step():
    import torch
    import lit_llama_b200 as P
    from lit_llama_b200.utils import quantization
    from bench import build_synthetic_model

    dev = torch.device("cuda")
    model = build_synthetic_model("7B", dev)
    S = 2048
    for pdl in (1, 0):
        for graph_after in (2, 0):
            model.reset_cache()
            model.decode_flags = pdl
            model.graph_after = graph_after
            model.copy_logits = False
            idx = torch.randint(0, 32000, (1, 16), device=dev, dtype=torch.int32)
            with torch.no_grad():
                model(idx, S, torch.arange(16, device=dev))
                tok = torch.randint(0, 32000, (1, 1), device=dev, dtype=torch.int32)
                pos = [torch.tensor([16 + i], device=dev) for i in range(64)]
                for i in range(4):
                    model(tok, S, pos[i])
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(4, 64):
                    model(tok, S, pos[i])
                e1.record()
                torch.cuda.synchronize()
            us = e0.elapsed_time(e1) / 60 * 1e3
            print(f"decode step 7B pos~16-80 pdl={pdl} graph={graph_after > 0}: {us:.1f} us/token  {1e6 / us:.1f} tok/s")


def sec_bench_ctx():
    """Decode step time against context length (graph + PDL): what single-token attention costs."""
    import torch
    from bench import build_synthetic_model

    dev = torch.device("cuda")
    model = build_synthetic_model("7B", dev)
    S = 2048
    model.copy_logits = False
    tok = torch.randint(0, 32000, (1, 1), device=dev, dtype=torch.int32)
    with torch.no_grad():
        model(torch.randint(0, 32000, (1, 16), device=dev, dtype=torch.int32), S, torch.arange(16, device=dev))
        t16 = None
        for p0 in (16, 120, 136, 512, 1024, 1536, 1990):
            pos = [torch.tensor([p0 + i], device=dev) for i in range(48)]
            for i in range(6):
                model(tok, S, pos[i])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(6, 46):
                model(tok, S, pos[i])
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) / 40 * 1e3
            t16 = t16 or us
            print(f"decode step 7B pos~{p0 + 6}-{p0 + 46}: {us:.1f} us/token  (+{(us - t16) / 32:.2f} us per layer over pos 16)")


def _decode_us(model, B, S, dev, p0=512, n=24):
    import torch

    tok = torch.randint(0, 32000, (B, 1), device=dev, dtype=torch.int32)
    pos = [torch.tensor([p0 + i], device=dev) for i in range(n + 6)]
    with torch.no_grad():
        for i in range(6):
            model(tok, S, pos[i])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(6, 6 + n):
            model(tok, S, pos[i])
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


def sec_bench_13b_b8():
    """BASELINE.json configs[3]: LLaMA-13B gptq.int4, batch 8, prefill 512 then decode (ctx 2048)."""
    import torch
    from bench import build_synthetic_model

    dev = torch.device("cuda")
    model = build_synthetic_model("13B", dev)
    model.copy_logits = False
    B, T, S = 8, 512, 2048
    idx = torch.randint(0, 32000, (B, T), device=dev, dtype=torch.int32)
    with torch.no_grad():
        for rep in range(2):
            model.reset_cache()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            model(idx, S, torch.arange(T, device=dev))
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
        print(f"13B gptq.int4 prefill B={B} T={T}: {ms:.1f} ms  ({B * T / ms * 1e3:.0f} tokens/s; tcgen05 tile GEMM for every linear)")
        if os.environ.get("B2L_PREFILL_PROFILE"):
            from torch.profiler import ProfilerActivity, profile
            model.reset_cache()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                model(idx, S, torch.arange(T, device=dev))
                torch.cuda.synchronize()
            print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=14, max_name_column_width=60))
    us = _decode_us(model, B, S, dev, p0=T)
    from lit_llama_b200.quantization import BATCH_GEMV
    print(f"13B gptq.int4 decode B={B} pos~{T}: {us:.0f} us/step  {B * 1e6 / us:.0f} tokens/s  "
          f"({'mma.sync batch kernel' if BATCH_GEMV else 'tcgen05 kernel'}, M={B})")


def sec_bench_sizes():
    """Batch-1 decode of every LLaMA size the reference names (lit_llama/model.py llama_configs)."""
    import torch
    from bench import build_synthetic_model

    dev = torch.device("cuda")
    for name in ("13B", "30B", "65B"):
        model = build_synthetic_model(name, dev)
        model.copy_logits = False
        with torch.no_grad():
            model(torch.randint(0, 32000, (1, 16), device=dev, dtype=torch.int32), 2048, torch.arange(16, device=dev))
        us = _decode_us(model, 1, 2048, dev, p0=16, n=32)
        cfg = model.config
        nh = [m for m in model.transformer.h[0].mlp.modules() if hasattr(m, "quant_weight")][0].quant_weight.shape[0]
        w_bytes = cfg.n_layer * (4 * cfg.n_embd * cfg.n_embd + 3 * cfg.n_embd * nh) // 2 + cfg.padded_vocab_size * cfg.n_embd // 2
        print(f"{name} gptq.int4 decode B=1 pos~16-50: {us:.0f} us/token  {1e6 / us:.1f} tok/s  "
              f"({w_bytes / us / 1e3:.0f} GB/s of packed weights = {w_bytes / us / 1e3 / 6573.2:.3f} of measured HBM peak)")
        del model
        torch.cuda.empty_cache()


def sec_batch_debug():
    """B = 2 decode on the tiny model: batch kernel vs batch-1 kernel, with and without PDL / fast path."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from gpu_util import build_tiny

    dev = torch.device("cuda")
    cfg = dict(block_size=32, vocab_size=96, n_layer=2, n_head=4, n_embd=128)
    idx = torch.tensor([[3, 17, 40], [9, 9, 1]], device=dev)
    for flags in (1, 0):
        for fast in (True, False):
            model, _, _ = build_tiny(dev, cfg)
            model.decode_flags = flags
            model.graph_after = 0
            if not fast:
                model._fast_ok = False
            with torch.no_grad():
                pre2 = model(idx, 16, torch.arange(3, device=dev)).clone()
                both = model(torch.tensor([[5], [60]], device=dev), 16, torch.tensor([3], device=dev)).clone()
                model.reset_cache()
                if not fast:
                    model._fast_ok = False
                pre1 = model(idx[1:], 16, torch.arange(3, device=dev)).clone()
                one = model(torch.tensor([[60]], device=dev), 16, torch.tensor([3], device=dev)).clone()
            print(f"pdl={flags} fast={fast}: prefill row diff {float((pre2[1:].float() - pre1.float()).abs().max()):.4g}  "
                  f"decode row diff {float((both[1:].float() - one.float()).abs().max()):.4g}  (|logits| max {float(one.float().abs().max()):.3g})", flush=True)


def sec_bench_step_int8():
    """LLaMA-7B --quantize llm.int8 decode (BASELINE config 2): module path replayed as a CUDA graph."""
    import torch
    import lit_llama_b200 as P
    from lit_llama_b200.utils import quantization

    dev = torch.device("cuda")
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device(dev), quantization("llm.int8"):
            model = P.LLaMA.from_name("7B")
    finally:
        torch.set_default_dtype(prev)
    model.eval()
    S = 2048
    model.copy_logits = False
    idx = torch.randint(0, 32000, (1, 16), device=dev, dtype=torch.int32)
    with torch.no_grad():
        model(idx, S, torch.arange(16, device=dev))
        tok = torch.randint(0, 32000, (1, 1), device=dev, dtype=torch.int32)
        pos = [torch.tensor([16 + i], device=dev) for i in range(72)]
        for i in range(6):
            model(tok, S, pos[i])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(6, 70):
            model(tok, S, pos[i])
        e1.record()
        torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 64 * 1e3
    W8 = 6.6132e9
    print(f"decode step 7B llm.int8 pos~16-90 graph={model._module_graph['graph'] is not None}: {us:.1f} us/token  {1e6 / us:.1f} tok/s  "
          f"({W8 / us / 1e3:.0f} GB/s of weights = {W8 / us / 1e3 / 6573.2:.3f} of measured HBM peak)")


def sec_timeline():
    """%globaltimer stamps of every launch of one eager decode step (7B): who overlaps whom."""
    import torch
    from bench import build_synthetic_model

    dev = torch.device("cuda")
    model = build_synthetic_model("7B", dev)
    S = 2048
    model.graph_after = 0
    model.copy_logits = False
    pos0 = int(os.environ.get("B2L_TL_POS", "64"))
    with torch.no_grad():
        model(torch.randint(0, 32000, (1, 16), device=dev, dtype=torch.int32), S, torch.arange(16, device=dev))
        tok = torch.randint(0, 32000, (1, 1), device=dev, dtype=torch.int32)
        for pdl in (1, 0):
            model.decode_flags = pdl
            model._decode = None
            for i in range(3):
                model(tok, S, torch.tensor([pos0 + i], device=dev))
            st = model._decode
            n = 5 * model.config.n_layer + 1
            tl = torch.zeros((n, 64), dtype=torch.int64, device=dev)
            tl[:, 0] = 2**62
            tl[:, 60] = 2**62
            tl[:, 61] = 2**62
            st.args.timeline = tl.data_ptr()
            model(tok, S, torch.tensor([pos0 + 3], device=dev))
            torch.cuda.synchronize()
            st.args.timeline = None
            t = tl.cpu()
            names = ["c_attn", "attn", "c_proj", "fc12", "mlp_proj"]
            base = int(t[5 * 4, 0])
            print(f"--- pdl={pdl} pos={pos0 + 3}: layers 4-5, ns relative to layer 4 c_attn start; "
                  "start(min) | wait_done(max) | x_ready(max) | loop_done(max) | end(max) | x_loaded(tid0) | after_ss_bar(tid0)")
            for li in range(5 * 4, 5 * 6 + 1):
                r = [int(v) - base if int(v) not in (0, 2**62) else None for v in t[li, :7]]
                extra = ""
                if li % 5 != 1:
                    extra = f"  | x_ready min..max {int(t[li, 60]) - base}..{r[2]}  loop_done min..max {int(t[li, 61]) - base}..{r[3]}"
                if li % 5 == 1:
                    b1 = int(t[li, 0])
                    extra = "  | CTA(0,0): " + " ".join(str(int(t[li, 8 + i]) - b1) for i in range(24) if int(t[li, 8 + i]))
                print(f"  L{li // 5} {names[li % 5]:9s} {r}{extra}")
            for li in (20, 23):  # layer 4 c_attn and fc12: CTA 0 per-stage stamps
                b0 = int(t[li, 0])
                st = [(int(t[li, 8 + 2 * i]) - b0, int(t[li, 9 + 2 * i]) - b0) for i in range(12) if int(t[li, 8 + 2 * i])]
                pi = [int(t[li, 40 + i]) - b0 for i in range(12) if int(t[li, 40 + i])]
                print(f"  {names[li % 5]} CTA0: wait_done={(int(t[li, 1]) - b0)} x_ready={(int(t[li, 2]) - b0)} stages(full_seen, done)={st} tma_issue={pi}")
            tot = int(t[n - 1, 4]) - int(t[0, 0])
            print(f"  whole step (first start -> lm_head end): {tot / 1e3:.1f} us; layer 4 start -> layer 5 start: "
                  f"{(int(t[25, 0]) - int(t[20, 0])) / 1e3:.2f} us")


def sec_precision():
    """How far the batch-1 kernel's fp32 accumulation is from exact arithmetic, in bf16 ulps of the result:
    fraction of outputs that differ from the correctly rounded fp64 result, and the largest distance."""
    import torch
    from lit_llama_b200 import _lib as L

    dev = torch.device("cuda")
    for N, K in [(4096, 4096), (4096, 11008), (2048, 22016)]:
        lv, qw, sc, z = rand_q4(N, K, dev, seed=3)
        qm, qt = tile_i8(L, qw, N, K), (tile(L, qw, N, K) if K <= 11008 else None)
        g = torch.Generator(device="cpu").manual_seed(5)
        base = torch.randn(1, K, generator=g)
        spike = base.clone(); spike[0, 16 * 7 + 2] = 60.0; spike[0, 16 * 90 + 11] = -45.0
        for name, xf in [("randn", base), ("randn+0.5", base + 0.5), ("|randn|", base.abs()), ("spikes", spike)]:
            x = xf.to(dev).bfloat16()
            want = ref_linear(x, lv, sc, z)
            wb = want.float().bfloat16()
            ulp = torch.maximum(want.abs(), torch.tensor(1e-30, device=dev, dtype=torch.float64)).log2().floor().sub(7).exp2()
            y, err = gemv_call(L, x, qm, sc, z, N, K)
            assert err is None, err
            line = f"N={N} K={K} x={name:10s} gemv: differ {float((y != wb).float().mean()):.4f}  max |y-exact| {float(((y.double() - want).abs() / ulp).max()):.3f} ulp"
            if qt is not None:
                y2, err = tc_call(L, torch.cat([x, x]), qt, sc, z, N, K)
                assert err is None, err
                line += f" | tcgen05: differ {float((y2[0:1] != wb).float().mean()):.4f}  max {float(((y2[0:1].double() - want).abs() / ulp).max()):.3f} ulp"
            print(line, flush=True)


def main():
    which = sys.argv[1:] or SECTIONS
    if len(which) == 1 and os.environ.get("B2L_DIAG_CHILD") == "1":
        globals()["sec_" + which[0]]()
        return
    for s in which:
        print(f"===== {s} =====", flush=True)
        t0 = time.time()
        env = dict(os.environ, B2L_DIAG_CHILD="1")
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), s], env=env, timeout=420, capture_output=True, text=True)
            print(r.stdout[-6000:])
            if r.returncode != 0:
                print(f"[{s}] exit code {r.returncode}\n{r.stderr[-3000:]}")
        except subprocess.TimeoutExpired as e:
            print(f"[{s}] TIMEOUT after 420 s\n{(e.stdout or b'')[-3000:]}")
        print(f"[{s}] {time.time() - t0:.1f} s", flush=True)


if __name__ == "__main__":
    main()
