"""Generates tests/golden/*.pt by running the UNMODIFIED reference on the CPU.

Run in the build container only (needs /root/reference):

    python oracle/make_golden.py

The reference is imported from /root/reference with oracle/_shim on sys.path (a
stand-in for the absent `lightning` package, which the decode path never calls).
The fixtures pin oracle/llama_oracle.py (tests/test_oracle_golden.py) and are the
vectors the GPU parity tests compare the CUDA path against.  TEST INFRASTRUCTURE.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("B2L_REFERENCE", "/root/reference")
sys.path.insert(0, os.path.join(HERE, "_shim"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import generate as ref_generate  # noqa: E402  (reference generate.py)
from lit_llama.model import LLaMA, LLaMAConfig, RMSNorm, apply_rope, build_rope_cache  # noqa: E402
from lit_llama.quantization import ColBlockQuantizedLinear, GPTQQuantizer  # noqa: E402
from lit_llama.utils import find_multiple, quantization  # noqa: E402

from oracle import llama_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def ref_quantized_linear(w, bits, groupsize):
    """Round-to-nearest through the reference's own GPTQQuantizer helpers and
    ColBlockQuantizedLinear.pack_weight (the tail of GPTQQuantizer.quantize)."""
    out_f, in_f = w.shape
    lin = torch.nn.Linear(in_f, out_f, bias=False)
    lin.weight.data.copy_(w)
    gq = GPTQQuantizer(lin, bits=bits, groupsize=groupsize)
    tc = in_f if groupsize == -1 else groupsize
    rec = torch.empty_like(w)
    for g in range(gq.scales.shape[1]):
        sl = slice(g * tc, (g + 1) * tc)
        scale, zero = gq.find_params_weight(w[:, sl])
        gq.scales[:, g : g + 1] = scale
        gq.zeros[:, g : g + 1] = zero
        rec[:, sl] = gq.quantize_weight(w[:, sl], scale, zero, gq.maxq)
    q = ColBlockQuantizedLinear(in_f, out_f, False, bits=bits, tile_cols=groupsize)
    q.scales = gq.scales
    q.zeros = gq.zeros
    q.pack_weight(rec)
    return q


def golden_quant():
    g = torch.Generator().manual_seed(7)
    cases = []
    for bits, groupsize, out_f, in_f in [(4, -1, 24, 64), (4, 32, 24, 128), (8, -1, 16, 64), (8, 32, 8, 96), (4, -1, 130, 256)]:
        w = torch.randn(out_f, in_f, generator=g) * 0.05
        x = torch.randn(3, in_f, generator=g)
        q = ref_quantized_linear(w, bits, groupsize)
        case = dict(bits=bits, groupsize=groupsize, w=w, x=x,
                    quant_weight=q.quant_weight.clone(), qw_stride=tuple(q.quant_weight.stride()),
                    scales=q.scales.clone(), zeros=q.zeros.clone(),
                    deq_f32=q.get_weight(torch.float32), deq_bf16=q.get_weight(torch.bfloat16),
                    y_f32=q(x))
        qb = ColBlockQuantizedLinear(in_f, out_f, False, bits=bits, tile_cols=groupsize)
        qb.quant_weight.copy_(q.quant_weight)
        qb.scales = q.scales.bfloat16()
        qb.zeros = q.zeros.bfloat16()
        case["y_bf16"] = qb(x.bfloat16())
        case["state_dict_keys"] = sorted(q.state_dict().keys())
        cases.append(case)
    return cases


def golden_ops():
    g = torch.Generator().manual_seed(11)
    out = {}
    x = torch.randn(2, 5, 128, generator=g)
    n = RMSNorm(128)
    n.scale.data = 1.0 + 0.1 * torch.randn(128, generator=g)
    out["rms_x"] = x
    out["rms_scale"] = n.scale.data.clone()
    out["rms_y_f32"] = n(x).detach()
    nb = RMSNorm(128).bfloat16()
    nb.scale.data = n.scale.data.bfloat16()
    out["rms_y_bf16"] = nb(x.bfloat16()).detach()
    idx = torch.zeros(1, 1, dtype=torch.long)
    table = build_rope_cache(seq_len=64, n_elem=32, dtype=idx.dtype, device=idx.device)
    out["rope_table_64x32"] = table
    out["rope_table_2048x128_rows"] = build_rope_cache(seq_len=2048, n_elem=128, dtype=idx.dtype, device=idx.device)[[0, 1, 777, 2047]]
    xr = torch.randn(2, 9, 4, 32, generator=g)
    out["rope_x"] = xr
    out["rope_y_f32"] = apply_rope(xr, table)
    out["rope_y_bf16"] = apply_rope(xr.bfloat16(), table)
    out["find_multiple"] = [(n_, k_, find_multiple(n_, k_)) for n_, k_ in [(10, 5), (11, 5), (32000, 64), (11008, 256), (1, 256), (50, 64)]]
    return out


def build_ref_model(cfg, sd, mode, dtype):
    with quantization(mode):
        m = LLaMA(LLaMAConfig(**cfg))
    m = m.to(dtype)
    missing = m.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return m.eval()


@torch.no_grad()
def golden_model(dtype, tag):
    cfg = dict(block_size=64, vocab_size=96, n_layer=2, n_head=4, n_embd=128)
    sd = O.synth_state_dict(cfg["n_layer"], cfg["n_head"], cfg["n_embd"], cfg["vocab_size"], "gptq.int4", dtype=dtype, seed=1234)
    m = build_ref_model(cfg, sd, "gptq.int4", dtype)
    g = torch.Generator().manual_seed(5)
    prompt = torch.randint(0, 96, (7,), generator=g)
    out = dict(cfg=cfg, seed=1234, prompt=prompt)
    # prefill + 3 decode steps, S = 16
    S = 16
    logits = [m(prompt.view(1, -1), S, torch.arange(7))]
    nxt = [11, 5, 90]
    for i, t in enumerate(nxt):
        logits.append(m(torch.tensor([[t]]), S, torch.tensor([7 + i])))
    out["steps_tokens"] = nxt
    out["steps_logits"] = [l.clone() for l in logits]
    out["kv0_k"] = m.kv_caches[0][0].clone()
    out["kv0_v"] = m.kv_caches[0][1].clone()
    m.reset_cache()
    # no-cache forward (model.py:104-106)
    out["nocache_logits"] = m(prompt.view(1, -1)).clone()
    # roll-when-full branch (model.py:214-218): S = 8, 7-token prompt, 6 more steps
    m.kv_caches.clear()
    S2 = 8
    roll_logits = [m(prompt.view(1, -1), S2, torch.arange(7))[:, -1].clone()]
    toks = [3, 17, 40, 41, 2, 77]
    for i, t in enumerate(toks):
        roll_logits.append(m(torch.tensor([[t]]), S2, torch.tensor([7 + i]))[:, -1].clone())
    out["roll_tokens"] = toks
    out["roll_logits"] = roll_logits
    out["roll_kv1_k"] = m.kv_caches[1][0].clone()
    m.reset_cache()
    # generate(): greedy and sampled
    m.kv_caches.clear()
    out["gen_greedy"] = ref_generate.generate(m, prompt.to(torch.int32), 12, top_k=1).clone()
    m.reset_cache(); m.kv_caches.clear()
    torch.manual_seed(1234)
    out["gen_sampled"] = ref_generate.generate(m, prompt.to(torch.int32), 12, temperature=0.8, top_k=20).clone()
    m.reset_cache(); m.kv_caches.clear()
    torch.manual_seed(99)
    out["gen_roll"] = ref_generate.generate(m, prompt.to(torch.int32), 12, max_seq_length=10, top_k=4).clone()
    torch.save(out, os.path.join(OUT, f"tiny_int4_{tag}.pt"))


@torch.no_grad()
def golden_dense_model():
    """Unquantized fp32 tiny model like tests/test_generate.py:26-54 (head_size 2)."""
    cfg = dict(block_size=128, vocab_size=16, n_layer=1, n_head=4, n_embd=8)
    sd = O.synth_state_dict(1, 4, 8, 16, None, dtype=torch.float32, seed=3)
    m = build_ref_model(cfg, sd, None, torch.float32)
    prompt = torch.tensor([1, 5, 9, 2, 7])
    torch.manual_seed(4)
    y = ref_generate.generate(m, prompt, 20, max_seq_length=10, top_k=4)
    torch.save(dict(cfg=cfg, seed=3, prompt=prompt, gen=y), os.path.join(OUT, "tiny_dense_f32.pt"))


def golden_reference_layout():
    """The public classes and functions of the reference modules lit_llama.patch_reference() rewires, with the module
    each is defined in: tests/test_modules_cpu.py rebuilds a package of placeholders laid out the same way."""
    import importlib
    import json

    layout = {}
    for name in ("lit_llama", "lit_llama.model", "lit_llama.utils", "lit_llama.quantization", "generate"):
        mod = importlib.import_module(name)
        layout[name] = {k: v.__module__ for k, v in sorted(vars(mod).items())
                        if not k.startswith("_") and callable(v)
                        and str(getattr(v, "__module__", "")).split(".")[0] in ("lit_llama", "generate")}
    with open(os.path.join(OUT, "reference_layout.json"), "w") as f:
        json.dump(layout, f, indent=1, sort_keys=True)
        f.write("\n")


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.save(golden_quant(), os.path.join(OUT, "quant_cases.pt"))
    torch.save(golden_ops(), os.path.join(OUT, "ops.pt"))
    golden_model(torch.float32, "f32")
    golden_model(torch.bfloat16, "bf16")
    golden_dense_model()
    golden_reference_layout()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
