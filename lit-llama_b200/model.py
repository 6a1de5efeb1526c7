"""Drop-in LLaMA modules (reference: lit_llama/model.py) backed by libb200llama.

Same classes, constructor signatures, parameter/buffer names and forward signatures as
the reference, so `with quantization(mode): model = LLaMA.from_name(name)` followed by
`model.load_state_dict(checkpoint)` and the reference's `generate()` work unchanged.
Every forward runs hand-written sm_100a kernels (include/b2l.h); tensors must be CUDA
bf16 - there is no CPU fallback.

Two execution paths behind `LLaMA.forward`:
  * decode (T == 1 with a KV cache, every Linear a gptq.int4 layer with one (scale, zero) per row):
    one C call enqueues the whole token (`b2l_decode_step`: int8-MMA GEMV kernels for batch 1, f16-MMA for 2..8 rows,
    tcgen05 for 9..16), replayed as a CUDA graph.
  * everything else (prefill on the tcgen05 GEMM, no-cache forward, other Linear kinds): module by module.
"""
import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Optional, Tuple, Union

import torch
import torch.nn as nn
from typing_extensions import Self

from . import _lib as L
from .quantization import WEIGHTS_GENERATION
from .utils import find_multiple

MaskCache = torch.Tensor
RoPECache = torch.Tensor
KVCache = Tuple[torch.Tensor, torch.Tensor]


@dataclass
class LLaMAConfig:
    """model.py:25-40."""
    block_size: int = 2048
    vocab_size: int = 32000
    padded_vocab_size: Optional[int] = None
    n_layer: int = 32
    n_head: int = 32
    n_embd: int = 4096

    def __post_init__(self):
        if self.padded_vocab_size is None:
            self.padded_vocab_size = find_multiple(self.vocab_size, 64)

    @classmethod
    def from_name(cls, name: str) -> Self:
        return cls(**llama_configs[name])


llama_configs = {  # model.py:43-48
    "7B": dict(n_layer=32, n_head=32, n_embd=4096),
    "13B": dict(n_layer=40, n_head=40, n_embd=5120),
    "30B": dict(n_layer=60, n_head=52, n_embd=6656),
    "65B": dict(n_layer=80, n_head=64, n_embd=8192),
}


def _linear(module: nn.Module, x: torch.Tensor) -> torch.Tensor:
    return module(x)


class RMSNorm(nn.Module):
    """model.py:257-277; the kernel keeps the reference's bf16 rounding points."""

    def __init__(self, size: int, dim: int = -1, eps: float = 1e-5) -> None:
        super().__init__()
        self.scale = nn.Parameter(torch.ones(size))
        self.eps = eps
        self.dim = dim

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        L.require_cuda_bf16(x, "RMSNorm.forward")
        if self.dim not in (-1, x.dim() - 1):
            raise RuntimeError("RMSNorm: only dim=-1 is implemented")
        xc = x.contiguous()
        C_ = xc.shape[-1]
        y = torch.empty_like(xc)
        scale = self.scale if self.scale.dtype == torch.bfloat16 else self.scale.to(torch.bfloat16)
        rc = L.lib().b2l_rmsnorm(xc.data_ptr(), scale.data_ptr(), y.data_ptr(), xc.numel() // C_, C_, float(self.eps), L.stream_ptr())
        L.check(rc, "b2l_rmsnorm")
        return y


def build_rope_cache(seq_len: int, n_elem: int, dtype: torch.dtype, device: torch.device, base: int = 10000) -> RoPECache:
    """model.py:280-303.  Table construction is one-time host-side setup (torch ops)."""
    theta = 1.0 / (base ** (torch.arange(0, n_elem, 2, dtype=dtype, device=device) / n_elem))
    seq_idx = torch.arange(seq_len, dtype=dtype, device=device)
    idx_theta = torch.outer(seq_idx, theta).float()
    cache = torch.stack([torch.cos(idx_theta), torch.sin(idx_theta)], dim=-1)
    if dtype in (torch.float16, torch.bfloat16, torch.int8):
        cache = cache.half()
    return cache


def apply_rope(x: torch.Tensor, rope_cache: RoPECache) -> torch.Tensor:
    """model.py:306-323 as a stand-alone op: x (B, T, n_head, hs) -> rotated copy.
    (Inside the model the rotation is fused with the KV append, see b2l_attention.)"""
    L.require_cuda_bf16(x, "apply_rope")
    B, T, nh, hs = x.shape
    qkv = torch.zeros((B, T, 3, nh, hs), device=x.device, dtype=x.dtype)
    qkv[:, :, 0] = x
    rows = rope_cache[:T].float().contiguous()
    y = torch.empty((B, T, nh * hs), device=x.device, dtype=x.dtype)
    work = torch.empty(L.lib().b2l_attn_workspace_bytes(B, nh, hs, T, T) // 4 + 1, device=x.device, dtype=torch.float32)
    rc = L.lib().b2l_attention_nocache(qkv.data_ptr(), rows.data_ptr(), y.data_ptr(), work.data_ptr(), B, T, nh, hs, T, L.stream_ptr())
    L.check(rc, "b2l_attention_nocache")
    return qkv[:, :, 0].contiguous()


class CausalSelfAttention(nn.Module):
    """model.py:171-237."""

    def __init__(self, config: LLaMAConfig) -> None:
        super().__init__()
        assert config.n_embd % config.n_head == 0
        self.c_attn = nn.Linear(config.n_embd, 3 * config.n_embd, bias=False)
        self.c_proj = nn.Linear(config.n_embd, config.n_embd, bias=False)
        self.n_head = config.n_head
        self.n_embd = config.n_embd
        self.block_size = config.block_size
        self._ring: Optional[torch.Tensor] = None  # shared by LLaMA; private when used stand-alone
        self._ring_shared = False

    def forward(
        self,
        x: torch.Tensor,
        rope: RoPECache,
        mask: MaskCache,
        max_seq_length: int,
        input_pos: Optional[torch.Tensor] = None,
        kv_cache: Optional[KVCache] = None,
        *,
        _rope_is_table: bool = False,
    ) -> Tuple[torch.Tensor, Optional[KVCache]]:
        """`mask` is accepted for signature parity and ignored: the kernel derives the
        causal mask from input_pos exactly as model.py:94-96 builds it from tril."""
        L.require_cuda_bf16(x, "CausalSelfAttention.forward")
        B, T, C_ = x.size()
        hs = C_ // self.n_head
        qkv = self.c_attn(x)
        if not qkv.is_contiguous():
            qkv = qkv.contiguous()
        y = torch.empty((B, T, C_), device=x.device, dtype=x.dtype)
        lib = L.lib()
        rope32 = rope if rope.dtype == torch.float32 else rope.float()
        rope32 = rope32.contiguous()
        if kv_cache is None:
            work = torch.empty(lib.b2l_attn_workspace_bytes(B, self.n_head, hs, T, T) // 4 + 1, device=x.device, dtype=torch.float32)
            rows = rope32 if not _rope_is_table else rope32[:T]
            rc = lib.b2l_attention_nocache(qkv.data_ptr(), rows.data_ptr(), y.data_ptr(), work.data_ptr(), B, T,
                                           self.n_head, hs, rows.shape[0], L.stream_ptr())
            L.check(rc, "b2l_attention_nocache")
        else:
            cache_k, cache_v = kv_cache
            S = cache_k.shape[2]
            assert S == max_seq_length and cache_k.is_contiguous() and cache_v.is_contiguous()
            pos = input_pos.reshape(-1).to(torch.int64)
            if self._ring is None or self._ring.device != x.device:
                self._ring = torch.zeros(1, dtype=torch.int32, device=x.device)
            if not self._ring_shared:  # stand-alone use: this module owns the roll state (model.py:214-218)
                L.check(lib.b2l_ring_advance(pos.data_ptr(), T, self._ring.data_ptr(), S, L.stream_ptr()), "b2l_ring_advance")
            work = torch.zeros(lib.b2l_attn_workspace_bytes(B, self.n_head, hs, T, S) // 4 + 1, device=x.device, dtype=torch.float32)
            flags = 0 if _rope_is_table else 4  # B2L_F_ROPE_ROWS
            rc = lib.b2l_attention(qkv.data_ptr(), cache_k.data_ptr(), cache_v.data_ptr(), rope32.data_ptr(), pos.data_ptr(),
                                   self._ring.data_ptr(), y.data_ptr(), work.data_ptr(), B, T, self.n_head, hs, S,
                                   rope32.shape[0], flags, L.stream_ptr())
            L.check(rc, "b2l_attention")
        y = self.c_proj(y)
        return y, kv_cache


class MLP(nn.Module):
    """model.py:240-254."""

    def __init__(self, config: LLaMAConfig) -> None:
        super().__init__()
        hidden_dim = 4 * config.n_embd
        n_hidden = int(2 * hidden_dim / 3)
        n_hidden = find_multiple(n_hidden, 256)
        self.c_fc1 = nn.Linear(config.n_embd, n_hidden, bias=False)
        self.c_fc2 = nn.Linear(config.n_embd, n_hidden, bias=False)
        self.c_proj = nn.Linear(n_hidden, config.n_embd, bias=False)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        L.require_cuda_bf16(x, "MLP.forward")
        a = self.c_fc1(x).contiguous()
        b = self.c_fc2(x).contiguous()
        h = torch.empty_like(a)
        L.check(L.lib().b2l_silu_mul(a.data_ptr(), b.data_ptr(), h.data_ptr(), a.numel(), L.stream_ptr()), "b2l_silu_mul")
        return self.c_proj(h)


def _add(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    a, b = a.contiguous(), b.contiguous()
    y = torch.empty_like(a)
    L.check(L.lib().b2l_add(a.data_ptr(), b.data_ptr(), y.data_ptr(), a.numel(), L.stream_ptr()), "b2l_add")
    return y


class Block(nn.Module):
    """model.py:148-168."""

    def __init__(self, config: LLaMAConfig) -> None:
        super().__init__()
        self.rms_1 = RMSNorm(config.n_embd)
        self.attn = CausalSelfAttention(config)
        self.rms_2 = RMSNorm(config.n_embd)
        self.mlp = MLP(config)

    def forward(
        self,
        x: torch.Tensor,
        rope: RoPECache,
        mask: MaskCache,
        max_seq_length: int,
        input_pos: Optional[torch.Tensor] = None,
        kv_cache: Optional[KVCache] = None,
        **kw,
    ) -> Tuple[torch.Tensor, Optional[KVCache]]:
        h, new_kv_cache = self.attn(self.rms_1(x), rope, mask, max_seq_length, input_pos, kv_cache, **kw)
        x = _add(x, h)
        x = _add(x, self.mlp(self.rms_2(x)))
        return x, new_kv_cache


class _DecodeState:
    """Static buffers + the C argument block of b2l_decode_step for one (B, S)."""

    def __init__(self, model: "LLaMA", B: int, S: int, device: torch.device, idx_dtype: torch.dtype) -> None:
        from .quantization import ColBlockQuantizedLinear

        cfg = model.config
        C_, nh = cfg.n_embd, cfg.n_head
        hs = C_ // nh
        bf = dict(device=device, dtype=torch.bfloat16)
        self.B, self.S = B, S
        self.generation = WEIGHTS_GENERATION[0]   # raw weight pointers below are valid for this generation only
        self.idx = torch.zeros(B, dtype=idx_dtype, device=device)
        self.pos = torch.zeros(1, dtype=torch.int64, device=device)
        self.x = torch.empty((B, C_), **bf)
        self.qkv = torch.empty((B, 3 * C_), **bf)
        self.att = torch.empty((B, C_), **bf)
        n_hidden = model.transformer.h[0].mlp.c_fc1.out_features
        self.hid = torch.empty((B, n_hidden), **bf)
        self.logits = torch.empty((B, 1, cfg.padded_vocab_size), **bf)
        lib = L.lib()
        self.work = torch.zeros(lib.b2l_attn_workspace_bytes(B, nh, hs, 1, S) // 4 + 1, device=device, dtype=torch.float32)
        self.keep = []  # tensors the argument block points into

        from .quantization import BATCH_GEMV, batch_workspace

        # batch 1..8: mma.sync kernels (q4_gemv / q4_gemv_batch) and their tiling; 9..16: tcgen05 kernel and its tiling
        gemv = (B == 1) or (B <= 8 and BATCH_GEMV)
        self.batch_ws = None
        if gemv and B > 1:
            self.batch_ws = batch_workspace(device, max(C_, n_hidden))

        def q4(lin: ColBlockQuantizedLinear) -> L.Q4Weight:
            t = (lin.tiled_i8() if B == 1 else lin.tiled_mma()) if gemv else lin.tiled()
            self.keep.append(t)   # a compacted layer hands out transient tilings: this state owns the ones it points at
            return L.Q4Weight(None if gemv else t.data_ptr(), t.data_ptr() if gemv else None, lin.scales.data_ptr(),
                              lin.zeros.data_ptr(), lin.out_features, lin.in_features)

        def bf16(p: torch.Tensor) -> torch.Tensor:
            t = p.detach()
            if t.dtype != torch.bfloat16:
                t = t.to(torch.bfloat16)
                self.keep.append(t)
            return t

        layers = (L.Layer * cfg.n_layer)()
        for i, blk in enumerate(model.transformer.h):
            fc12 = model._fc12(i, "i8" if B == 1 else ("mma" if gemv else "tc"))
            k, v = model.kv_caches[i]
            layers[i] = L.Layer(
                rms_1=bf16(blk.rms_1.scale).data_ptr(), rms_2=bf16(blk.rms_2.scale).data_ptr(),
                c_attn=q4(blk.attn.c_attn), c_proj=q4(blk.attn.c_proj),
                c_fc12=L.Q4Weight(None if gemv else fc12[0].data_ptr(), fc12[0].data_ptr() if gemv else None,
                                  fc12[1].data_ptr(), fc12[2].data_ptr(), 2 * n_hidden, C_),
                mlp_proj=q4(blk.mlp.c_proj), k_cache=k.data_ptr(), v_cache=v.data_ptr())
        self.layers = layers
        lin0 = model.lm_head
        self.args = L.DecodeArgs(
            n_layer=cfg.n_layer, n_head=nh, n_embd=C_, n_hidden=n_hidden, vocab=cfg.padded_vocab_size, B=B, S=S,
            sz_dtype=L.sz_dtype_of(lin0.scales), eps=float(model.transformer.ln_f.eps), layers=layers,
            wte=bf16(model.transformer.wte.weight).data_ptr(), ln_f=bf16(model.transformer.ln_f.scale).data_ptr(),
            lm_head=q4(lin0), rope=model.rope_cache.data_ptr(), idx=self.idx.data_ptr(),
            idx_is_i64=1 if idx_dtype == torch.int64 else 0, input_pos=self.pos.data_ptr(),
            ring_start=model._ring.data_ptr(), block_size=cfg.block_size, x=self.x.data_ptr(), qkv=self.qkv.data_ptr(),
            att=self.att.data_ptr(), hid=self.hid.data_ptr(), attn_work=self.work.data_ptr(),
            logits=self.logits.data_ptr(), flags=model.decode_flags,
            batch_work=None if self.batch_ws is None else self.batch_ws.data_ptr())
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.calls = 0

    def enqueue(self) -> None:
        L.check(L.lib().b2l_decode_step(C.byref(self.args), L.stream_ptr()), "b2l_decode_step")


class LLaMA(nn.Module):
    """model.py:51-145."""

    #: replay the decode step as a CUDA graph after this many eager steps (0 = never)
    graph_after: int = 2
    #: flags passed to b2l_decode_step (1 = programmatic dependent launch)
    decode_flags: int = 1
    #: return a fresh logits tensor per call like the reference (False: a view of the static buffer)
    copy_logits: bool = True

    def __init__(self, config: LLaMAConfig) -> None:
        super().__init__()
        assert config.padded_vocab_size is not None
        self.config = config

        self.lm_head = nn.Linear(config.n_embd, config.padded_vocab_size, bias=False)
        self.transformer = nn.ModuleDict(
            dict(
                wte=nn.Embedding(config.padded_vocab_size, config.n_embd),
                h=nn.ModuleList(Block(config) for _ in range(config.n_layer)),
                ln_f=RMSNorm(config.n_embd),
            )
        )

        self.rope_cache: Optional[RoPECache] = None
        self.mask_cache: Optional[MaskCache] = None  # kept for attribute parity; never materialised
        self.kv_caches: List[KVCache] = []
        self._ring: Optional[torch.Tensor] = None
        self._kv_store: Optional[torch.Tensor] = None
        self._decode: Optional[_DecodeState] = None
        self._module_graph = None  # CUDA graph of the module-by-module decode step (non-fused Linear kinds)
        self._fast_ok: Optional[bool] = None  # every Linear is a per-row gptq.int4 layer the fused step can run (checked once)
        self._fc12_cache = {}

    def _init_weights(self, module: nn.Module) -> None:
        """model.py:70-74."""
        if isinstance(module, nn.Linear) and hasattr(module, "weight"):
            torch.nn.init.normal_(module.weight, mean=0.0, std=0.02 / math.sqrt(2 * self.config.n_layer))
        elif isinstance(module, nn.Embedding):
            torch.nn.init.normal_(module.weight, mean=0.0, std=0.02 / math.sqrt(2 * self.config.n_layer))

    @classmethod
    def from_name(cls, name: str) -> Self:
        return cls(LLaMAConfig.from_name(name))

    def build_rope_cache(self, idx: torch.Tensor) -> RoPECache:
        """model.py:128-134: called with the integer token tensor, so the table is fp32."""
        return build_rope_cache(seq_len=self.config.block_size, n_elem=self.config.n_embd // self.config.n_head,
                                dtype=idx.dtype, device=idx.device)

    def build_mask_cache(self, idx: torch.Tensor) -> MaskCache:
        """model.py:136-138 (provided for parity; the kernels never read a mask tensor)."""
        ones = torch.ones((self.config.block_size, self.config.block_size), device=idx.device, dtype=torch.bool)
        return torch.tril(ones).unsqueeze(0).unsqueeze(0)

    def reset_cache(self) -> None:
        """model.py:140-145."""
        self.kv_caches.clear()
        self._kv_store = None
        self._decode = None
        self._module_graph = None
        if self._ring is not None:
            self._ring.zero_()

    # ------------------------------------------------------------------ helpers
    def _fc12(self, i: int, kind: str):
        """c_fc1 and c_fc2 of layer i interleaved (8 rows / 8 rows per 16-row block for the
        batch-1 kernel, 64 / 64 per 128-row tile for the tcgen05 kernel) and re-tiled, so one
        tile holds silu's argument and its multiplier and SwiGLU runs in the epilogue."""
        mlp = self.transformer.h[i].mlp
        gemv = kind != "tc"
        hit = self._fc12_cache.get((i, kind))
        if hit is not None and getattr(mlp.c_fc1, "_released", False):
            return hit[1]     # compacted: this copy IS the layer's weights (compact())
        q1, q2 = mlp.c_fc1.reference_quant_weight(), mlp.c_fc2.reference_quant_weight()
        key = (kind, q1.data_ptr(), q1._version, q2.data_ptr(), q2._version)
        if hit is not None and hit[0] == key:
            return hit[1]
        nh, K = mlp.c_fc1.out_features, mlp.c_fc1.in_features
        g = 8 if gemv else 64
        assert nh % g == 0

        def inter(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:  # rows (dim 0) of a, b -> [t][g of a | g of b]
            return torch.stack((a.reshape(nh // g, g, *a.shape[1:]), b.reshape(nh // g, g, *b.shape[1:])), dim=1).reshape(2 * nh, *a.shape[1:])

        qw = inter(q1, q2).t().contiguous().t()  # reference layout (1, 2nh)
        scales = inter(mlp.c_fc1.scales, mlp.c_fc2.scales).contiguous()
        zeros = inter(mlp.c_fc1.zeros, mlp.c_fc2.zeros).contiguous()
        lib = L.lib()
        if kind == "i8":
            tiled = torch.empty(lib.b2l_q4_tiled_i8_bytes(2 * nh, K), dtype=torch.uint8, device=qw.device)
            L.check(lib.b2l_q4_tile_i8(qw.data_ptr(), tiled.data_ptr(), 2 * nh, K, L.stream_ptr()), "b2l_q4_tile_i8")
        elif kind == "mma":
            tiled = torch.empty(lib.b2l_q4_tiled_mma_bytes(2 * nh, K), dtype=torch.uint8, device=qw.device)
            L.check(lib.b2l_q4_tile_mma(qw.data_ptr(), tiled.data_ptr(), 2 * nh, K, L.stream_ptr()), "b2l_q4_tile_mma")
        else:
            tiled = torch.empty(lib.b2l_q4_tiled_bytes(2 * nh, K), dtype=torch.uint8, device=qw.device)
            L.check(lib.b2l_q4_tile(qw.data_ptr(), tiled.data_ptr(), 2 * nh, K, L.stream_ptr()), "b2l_q4_tile")
        val = (tiled, scales, zeros)
        self._fc12_cache[(i, kind)] = (key, val)
        return val

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        # the interleaved fc1|fc2 copies are plain tensors of this module: they move with it (a compacted model has no other)
        self._fc12_cache = {k: (key, tuple(fn(t) for t in val)) for k, (key, val) in self._fc12_cache.items()}
        self._decode, self._module_graph, self._fast_ok = None, None, None
        return out

    def _fc_from_fc12(self, i: int, which: int) -> torch.Tensor:
        """c_fc1 (which = 0) or c_fc2 (1) of layer i in the reference layout, rebuilt from the interleaved batch-1
        tiling (compacted models keep only that copy): untile (a nibble permutation) and take every other 8 rows."""
        tiled, _, _ = self._fc12_cache[(i, "i8")][1]
        mlp = self.transformer.h[i].mlp
        nh, K = mlp.c_fc1.out_features, mlp.c_fc1.in_features
        both = torch.empty((K // 2, 2 * nh), dtype=torch.uint8, device=tiled.device).t()
        L.check(L.lib().b2l_q4_untile_i8(tiled.data_ptr(), both.data_ptr(), 2 * nh, K, L.stream_ptr()), "b2l_q4_untile_i8")
        return both.contiguous().reshape(nh // 8, 2, 8, K // 2)[:, which].reshape(nh, K // 2).t().contiguous().t()

    def compact(self) -> "LLaMA":
        """Keep ONE resident copy of every gptq.int4 weight: the batch-1 decode tiling (c_fc1 / c_fc2: the interleaved
        fc1|fc2 tiling).  The reference-layout buffers and the per-kernel duplicates are freed; `state_dict()`, prefill
        and batched decode rebuild what they need transiently from that copy (bit-exact permutations).  7B: 3.3 GB of
        weights + 0.26 GB embedding + KV cache instead of 2-3 copies (the reference's gptq.int4 figure is "~5 GB",
        howto/inference.md:37).  Returns self."""
        import functools

        if self._fast_ok is None:
            self._fast_ok = self._fast_decode_ok()
        if not self._fast_ok:
            raise RuntimeError("compact() needs a gptq.int4 model the fused batch-1 decode step can run")
        for i, blk in enumerate(self.transformer.h):
            self._fc12(i, "i8")
            for kind in ("mma", "tc"):
                self._fc12_cache.pop((i, kind), None)
            for lin in (blk.attn.c_attn, blk.attn.c_proj, blk.mlp.c_proj):
                lin.release_reference_layout()
            blk.mlp.c_fc1.release_reference_layout(source=functools.partial(self._fc_from_fc12, i, 0))
            blk.mlp.c_fc2.release_reference_layout(source=functools.partial(self._fc_from_fc12, i, 1))
        self.lm_head.release_reference_layout()
        self._decode, self._module_graph = None, None   # rebuilt on the next step (B > 1 states hold their transient tilings)
        torch.cuda.empty_cache()
        return self

    def _fast_decode_ok(self) -> bool:
        from .quantization import ColBlockQuantizedLinear

        def ok(m):
            return isinstance(m, ColBlockQuantizedLinear) and m.tc_capable and m.gemv_capable

        if not ok(self.lm_head) or self.config.n_embd % 8 != 0:
            return False
        dt = self.lm_head.scales.dtype
        for blk in self.transformer.h:
            lins = (blk.attn.c_attn, blk.attn.c_proj, blk.mlp.c_fc1, blk.mlp.c_fc2, blk.mlp.c_proj)
            if not all(ok(m) and m.scales.dtype == dt for m in lins):
                return False
            if blk.mlp.c_fc1.out_features % 64 != 0:
                return False
        return True

    def logical_kv_caches(self) -> List[KVCache]:
        """kv_caches in the reference's slot order.  Identical to `kv_caches` until the
        roll branch (model.py:214-218) has triggered; afterwards the physical tensors are
        a ring and this returns the un-rotated copies the reference would hold."""
        out = []
        lib = L.lib()
        for k, v in self.kv_caches:
            B, nh, S, hs = k.shape
            ko, vo = torch.empty_like(k), torch.empty_like(v)
            L.check(lib.b2l_kv_unroll(k.data_ptr(), self._ring.data_ptr(), ko.data_ptr(), B, nh, S, hs, L.stream_ptr()), "b2l_kv_unroll")
            L.check(lib.b2l_kv_unroll(v.data_ptr(), self._ring.data_ptr(), vo.data_ptr(), B, nh, S, hs, L.stream_ptr()), "b2l_kv_unroll")
            out.append((ko, vo))
        return out

    # ------------------------------------------------------------------ forward
    def forward(
        self, idx: torch.Tensor, max_seq_length: Optional[int] = None, input_pos: Optional[torch.Tensor] = None
    ) -> Union[torch.Tensor, Tuple[torch.Tensor, List[KVCache]]]:
        B, T = idx.size()
        if not idx.is_cuda:
            raise RuntimeError(f"LLaMA.forward: idx is on {idx.device}; lit_llama_b200 runs on CUDA only (no CPU fallback)")

        block_size = self.config.block_size
        if max_seq_length is None:
            max_seq_length = block_size
        assert T <= max_seq_length, f"Cannot forward sequence of length {T}, max seq length is only {max_seq_length}"
        assert max_seq_length <= block_size, f"Cannot attend to {max_seq_length}, block size is only {block_size}"
        assert T <= block_size, f"Cannot forward sequence of length {T}, block size is only {block_size}"

        if self.rope_cache is None or self.rope_cache.device != idx.device:
            self.rope_cache = self.build_rope_cache(idx).float().contiguous()
        if self._ring is None or self._ring.device != idx.device:
            self._ring = torch.zeros(1, dtype=torch.int32, device=idx.device)
            for blk in self.transformer.h:
                blk.attn._ring, blk.attn._ring_shared = self._ring, True

        if input_pos is not None and not self.kv_caches:
            cfg = self.config
            hs = cfg.n_embd // cfg.n_head
            self._kv_store = torch.zeros((cfg.n_layer, 2, B, cfg.n_head, max_seq_length, hs), device=idx.device, dtype=torch.bfloat16)
            self.kv_caches = [(self._kv_store[i, 0], self._kv_store[i, 1]) for i in range(cfg.n_layer)]
            self._decode = None
            self._module_graph = None

        # ---- decode: one C call per token, replayed as a CUDA graph
        st = None
        if input_pos is not None and T == 1 and B <= 16 and idx.dtype in (torch.int32, torch.int64):
            st = self._decode
            if st is not None and st.generation != WEIGHTS_GENERATION[0]:
                # a linear was reloaded, repacked or moved since the argument block / graph was built: everything that
                # bakes weight pointers is stale (fc1|fc2 interleave, eligibility, module graph included)
                st = self._decode = None
                self._module_graph, self._fast_ok = None, None
                self._fc12_cache.clear()
            if st is None or st.B != B or st.S != max_seq_length or st.idx.dtype != idx.dtype or st.idx.device != idx.device:
                if self._fast_ok is None:
                    self._fast_ok = self._fast_decode_ok()
                st = self._decode = _DecodeState(self, B, max_seq_length, idx.device, idx.dtype) if self._fast_ok else None
        if st is not None:
            st.idx.copy_(idx.reshape(-1))
            st.pos.copy_(input_pos.reshape(-1)[-1:])
            if st.graph is not None:
                st.graph.replay()
            elif self.graph_after and st.calls >= self.graph_after:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    st.enqueue()
                st.graph = g
                g.replay()
            else:
                st.enqueue()
            st.calls += 1
            return st.logits.clone() if self.copy_logits else st.logits

        # ---- single-token decode with any other Linear kind (llm.int8, gptq.int8, grouped scales, dense):
        #      the module-by-module launch sequence, replayed as a CUDA graph once warm
        if input_pos is not None and T == 1 and self.graph_after and idx.dtype in (torch.int32, torch.int64):
            key = (B, max_seq_length, idx.dtype, idx.device, WEIGHTS_GENERATION[0])   # the graph bakes weight pointers too
            mg = self._module_graph
            if mg is None or mg["key"] != key:
                mg = self._module_graph = dict(key=key, calls=0, graph=None, idx=torch.zeros((B, 1), dtype=idx.dtype, device=idx.device),
                                               pos=torch.zeros(1, dtype=torch.int64, device=idx.device), out=None)
            mg["idx"].copy_(idx)
            mg["pos"].copy_(input_pos.reshape(-1)[-1:])
            if mg["graph"] is not None:
                mg["graph"].replay()
                return mg["out"].clone() if self.copy_logits else mg["out"]
            mg["calls"] += 1
            if mg["calls"] > self.graph_after:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    mg["out"] = self._forward_modules(mg["idx"], max_seq_length, mg["pos"])
                mg["graph"] = g
                g.replay()
                return mg["out"].clone() if self.copy_logits else mg["out"]
        return self._forward_modules(idx, max_seq_length, input_pos)

    def _forward_modules(self, idx: torch.Tensor, max_seq_length: int, input_pos: Optional[torch.Tensor]) -> torch.Tensor:
        """Prefill, no-cache forward and non-fused decode: one kernel (or two) per reference module."""
        B, T = idx.size()
        x = torch.empty((B, T, self.config.n_embd), device=idx.device, dtype=torch.bfloat16)
        wte = self.transformer.wte.weight
        if wte.dtype != torch.bfloat16:
            raise RuntimeError(f"wte dtype {wte.dtype} unsupported; the model must be bf16 (model.to(torch.bfloat16))")
        idx_c = idx.contiguous()
        if idx_c.dtype not in (torch.int32, torch.int64):
            idx_c = idx_c.to(torch.int64)
        rc = L.lib().b2l_embedding(idx_c.data_ptr(), 1 if idx_c.dtype == torch.int64 else 0, wte.data_ptr(), x.data_ptr(),
                                   B * T, self.config.n_embd, wte.shape[0], L.stream_ptr())
        L.check(rc, "b2l_embedding")

        if input_pos is None:  # proxy for use_cache=False (model.py:104-106)
            for block in self.transformer.h:
                x, _ = block(x, self.rope_cache, None, max_seq_length, _rope_is_table=True)
        else:
            pos = input_pos.reshape(-1).to(torch.int64)
            L.check(L.lib().b2l_ring_advance(pos.data_ptr(), T, self._ring.data_ptr(), max_seq_length, L.stream_ptr()), "b2l_ring_advance")
            for i, block in enumerate(self.transformer.h):
                x, self.kv_caches[i] = block(x, self.rope_cache, None, max_seq_length, pos, self.kv_caches[i], _rope_is_table=True)

        x = self.transformer.ln_f(x)
        logits = self.lm_head(x)  # (b, t, vocab_size)
        return logits
