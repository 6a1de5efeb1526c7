"""CPU: the drop-in modules keep the reference's construction-time contract (names,
shapes, dtypes, strides, state_dict keys), the quantization() swap behaves like
lit_llama/utils.py:141-162, and nothing silently runs on the CPU."""
import os
import sys

import pytest
import torch

from conftest import GOLDEN, load_golden

import lit_llama_b200 as P
from lit_llama_b200.utils import quantization
from oracle import llama_oracle as O


def test_find_multiple_and_lookup():
    for n, k, want in load_golden("ops.pt")["find_multiple"]:
        assert P.find_multiple(n, k) == want
    assert P.llama_model_lookup({"transformer.wte.weight": torch.empty(8, 5120)}) == "13B"
    with pytest.raises(KeyError):
        P.llama_model_lookup({"transformer.wte.weight": torch.empty(8, 100)})


def test_quantization_context_swaps_and_restores():
    orig = torch.nn.Linear
    with quantization("gptq.int4"):
        lin = torch.nn.Linear(64, 32, bias=False)
        assert isinstance(lin, P.ColBlockQuantizedLinear) and lin.bits == 4 and lin.tile_cols == 64
    assert torch.nn.Linear is orig
    with quantization("gptq.int8"):
        assert torch.nn.Linear(64, 32, bias=False).bits == 8
    with quantization(None):
        assert torch.nn.Linear is orig
    with pytest.raises(ValueError):
        with quantization("gptq.int3"):
            pass
    with pytest.raises(RuntimeError):
        with quantization("gptq.int4"):
            raise RuntimeError("boom")
    assert torch.nn.Linear is orig  # restored even when the body raises


def test_colblock_buffers_match_reference_contract():
    for c in load_golden("quant_cases.pt"):
        out_f, in_f = c["w"].shape
        lin = P.ColBlockQuantizedLinear(in_f, out_f, False, bits=c["bits"], tile_cols=c["groupsize"])
        assert sorted(lin.state_dict().keys()) == c["state_dict_keys"]
        assert lin.quant_weight.dtype == torch.uint8 and lin.quant_weight.shape == c["quant_weight"].shape
        assert tuple(lin.quant_weight.stride()) == c["qw_stride"]
        assert lin.scales.shape == c["scales"].shape and lin.zeros.shape == c["zeros"].shape
        assert lin.bias is None and lin.entries_per_byte == 8 // c["bits"]
        # pack_weight is load-time host logic and follows the reference bit for bit
        lin.scales, lin.zeros = c["scales"].clone(), c["zeros"].clone()
        lin.pack_weight(c["deq_f32"].clone())
        ref = O.pack_weight(c["deq_f32"], c["scales"], c["zeros"], c["bits"], in_f if c["groupsize"] == -1 else c["groupsize"])
        assert torch.equal(lin.quant_weight, ref)
    b = P.ColBlockQuantizedLinear(64, 8, True, bits=8, tile_cols=-1)
    assert b.bias.shape == (8,)


def test_model_structure_and_state_dict_roundtrip():
    cfg = dict(block_size=64, vocab_size=96, n_layer=2, n_head=4, n_embd=128)
    sd = O.synth_state_dict(2, 4, 128, 96, "gptq.int4", dtype=torch.bfloat16)
    with quantization("gptq.int4"):
        m = P.LLaMA(P.LLaMAConfig(**cfg))
    assert sorted(m.state_dict().keys()) == sorted(sd.keys())
    res = m.load_state_dict(sd)
    assert not res.missing_keys and not res.unexpected_keys
    assert m.config.padded_vocab_size == 128
    assert m.transformer.h[0].mlp.c_fc1.out_features == O.n_hidden_for(128)
    out = m.state_dict()
    for k, v in sd.items():
        assert torch.equal(out[k].to(v.dtype), v), k
    assert P.LLaMAConfig.from_name("7B").n_embd == 4096 and P.LLaMAConfig.from_name("65B").n_layer == 80
    m.reset_cache()
    assert m.kv_caches == []


def test_no_cpu_fallback_anywhere():
    with quantization("gptq.int4"):
        m = P.LLaMA(P.LLaMAConfig(block_size=16, vocab_size=64, n_layer=1, n_head=2, n_embd=64)).bfloat16()
    with pytest.raises(RuntimeError, match="CUDA only"):
        m(torch.zeros(1, 3, dtype=torch.long))
    x = torch.zeros(1, 3, 64, dtype=torch.bfloat16)
    for mod in (m.lm_head, m.transformer.ln_f, m.transformer.h[0].mlp):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            mod(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        P.apply_rope(torch.zeros(1, 3, 2, 32, dtype=torch.bfloat16), torch.zeros(3, 16, 2))
    for fn in (P.sample_probs, P.sample_token):   # the sampling tail of generate() has no CPU path either
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(torch.zeros(64, dtype=torch.bfloat16), 0.8, 4)


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lit-llama_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src, f"{f} references oracle/"


def _write_reference_standin(root, layout):
    """A package laid out like the reference (tests/golden/reference_layout.json, recorded from it by
    oracle/make_golden.py): every public class and function is a placeholder class in the module that defines it and
    is imported by name into the modules that import it."""
    defs, imports = {}, {}
    for mod, names in layout.items():
        for name, home in names.items():
            defs.setdefault(home, set()).add(name)
            if home != mod:
                imports.setdefault(mod, []).append((home, name))
    mods = set(defs) | set(imports)
    pkgs = {m.rsplit(".", 1)[0] for m in mods if "." in m}
    for mod in mods:
        path = root.joinpath(*mod.split("."))
        path = path / "__init__.py" if mod in pkgs else path.with_suffix(".py")
        path.parent.mkdir(parents=True, exist_ok=True)
        src = [f"from {home} import {name}" for home, name in sorted(imports.get(mod, []))]
        src += [f"class {name}:\n    pass" for name in sorted(defs.get(mod, ()))]
        path.write_text("\n".join(src) + "\n")


def _reference_modules():
    return [m for m in sys.modules if m in ("generate", "lit_llama") or m.startswith("lit_llama.")]


def test_patch_reference_plugs_into_unmodified_reference(tmp_path, monkeypatch):
    """patch_reference() on a package with the reference's module layout: the B200 classes replace the reference's
    names everywhere a caller reaches them, including the names generate.py imported before the patch."""
    import json

    with open(os.path.join(GOLDEN, "reference_layout.json")) as f:
        _write_reference_standin(tmp_path, json.load(f))
    monkeypatch.syspath_prepend(str(tmp_path))
    for name in _reference_modules():
        monkeypatch.delitem(sys.modules, name)
    import lit_llama
    import lit_llama.quantization  # noqa: F401
    import generate as ref_generate

    saved = P.patch_reference(lit_llama)
    try:
        from lit_llama.utils import quantization as ref_q
        from lit_llama.model import LLaMA as RefLLaMA, LLaMAConfig as RefCfg

        assert RefLLaMA is P.LLaMA and ref_generate.LLaMA is P.LLaMA and ref_generate.quantization is quantization
        with ref_q("gptq.int4"):
            m = RefLLaMA(RefCfg(block_size=16, vocab_size=64, n_layer=1, n_head=2, n_embd=64))
        assert isinstance(m, P.LLaMA) and isinstance(m.lm_head, P.ColBlockQuantizedLinear)
        assert isinstance(m.transformer.h[0], P.Block)
    finally:
        import lit_llama.model as rm, lit_llama.utils as ru, lit_llama.quantization as rq

        for (where, name), val in saved.items():
            tgt = {"model": rm, "pkg": lit_llama, "quant": rq, "utils": ru}[where]
            if val is not None:
                setattr(tgt, name, val)
        ref_generate.LLaMA = saved[("model", "LLaMA")]
        ref_generate.quantization = saved[("utils", "quantization")]
        for name in _reference_modules():
            del sys.modules[name]


def test_linear8bitlt_contract_on_cpu():
    """quantization.py:38-77: quantised at construction and again when a float weight is loaded;
    state_dict key is `weight` (+ `bias`); statistics live on the parameter (CB, SCB)."""
    with quantization("llm.int8"):
        lin = torch.nn.Linear(256, 24, bias=False)
    assert isinstance(lin, P.Linear8bitLt) and lin.threshold == 6.0
    assert lin.weight.dtype == torch.int8 and lin.weight.SCB.shape == (24,) and lin.weight.CB is not None
    assert list(lin.state_dict().keys()) == ["weight"]
    w = torch.randn(24, 256) * 0.1
    lin.load_state_dict({"weight": w})
    cb, scb = O.int8_quantize_weight(w)
    assert torch.equal(lin.weight.data, cb) and torch.equal(lin.weight.SCB, scb)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        lin(torch.zeros(1, 256, dtype=torch.bfloat16))


def test_empty_init_on_device_and_lazy_load(tmp_path):
    """utils.py:73-138 and :332-344: construction context and lazy checkpoint loading (host-side, CPU)."""
    from lit_llama_b200.utils import EmptyInitOnDevice, lazy_load

    before = (torch.nn.Linear, torch.get_default_dtype(), torch.nn.init.normal_)
    with EmptyInitOnDevice(device=torch.device("cpu"), dtype=torch.bfloat16, quantization_mode="gptq.int4"):
        m = P.LLaMA(P.LLaMAConfig(block_size=16, vocab_size=64, n_layer=1, n_head=2, n_embd=64))
        lin = torch.nn.Linear(8, 4, bias=False)
    assert (torch.nn.Linear, torch.get_default_dtype(), torch.nn.init.normal_) == before   # everything restored
    assert isinstance(m.lm_head, P.ColBlockQuantizedLinear) and isinstance(lin, P.ColBlockQuantizedLinear)
    assert m.transformer.wte.weight.dtype == torch.bfloat16
    with pytest.raises(ValueError, match="only supported on the GPU"):
        EmptyInitOnDevice(device=torch.device("cpu"), quantization_mode="llm.int8")
    with pytest.raises(RuntimeError, match="unknown quantization mode"):
        EmptyInitOnDevice(quantization_mode="int3")

    sd = {k: v.clone() for k, v in m.state_dict().items()}
    for v in sd.values():
        if v.dtype == torch.uint8:
            v.random_(0, 256)
        else:
            v.copy_(torch.randn(v.shape))
    path = tmp_path / "ckpt.pth"
    torch.save(sd, path)
    with lazy_load(path) as ck:
        assert set(ck) == set(sd)
        assert P.llama_model_lookup({"transformer.wte.weight": torch.empty(1, 4096)}) == "7B"
        m.load_state_dict(ck)
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]) and v.stride() == sd[k].stride(), k


def test_weight_changes_bump_the_generation_and_compact_refuses_what_it_cannot_serve():
    """Host logic behind two round-2 features, no kernels involved: (1) load_state_dict / pack_weight / .to() bump the
    generation counter that invalidates baked decode states (lit_llama_b200/model.py); (2) compact() /
    release_reference_layout() refuse models and layers the batch-1 decode tiling cannot represent instead of
    freeing their only copy."""
    from lit_llama_b200.quantization import WEIGHTS_GENERATION

    cfg = dict(block_size=16, vocab_size=32, n_layer=1, n_head=2, n_embd=64)
    with quantization("gptq.int4"):
        m = P.LLaMA(P.LLaMAConfig(**cfg))
    g0 = WEIGHTS_GENERATION[0]
    m.load_state_dict(m.state_dict())
    g1 = WEIGHTS_GENERATION[0]
    assert g1 > g0
    lin = m.transformer.h[0].attn.c_proj
    lin.scales.fill_(1.0); lin.zeros.fill_(8.0)
    lin.pack_weight(torch.zeros(64, 64))
    assert WEIGHTS_GENERATION[0] > g1
    g2 = WEIGHTS_GENERATION[0]
    m.to(torch.bfloat16)
    assert WEIGHTS_GENERATION[0] > g2
    # a dense model has nothing to compact
    dense = P.LLaMA(P.LLaMAConfig(**cfg))
    with pytest.raises(RuntimeError):
        dense.compact()
    # grouped scales (gptq with groupsize) and int8 levels are outside the batch-1 tiling: the buffer stays
    grouped = P.ColBlockQuantizedLinear(128, 32, bias=False, bits=4, tile_cols=64)
    with pytest.raises(RuntimeError):
        grouped.release_reference_layout()
    assert grouped.quant_weight.numel() == 32 * 64 and not grouped._released
    q8 = P.ColBlockQuantizedLinear(128, 32, bias=False, bits=8, tile_cols=-1)
    with pytest.raises(RuntimeError):
        q8.release_reference_layout()
    # state_dict of an untouched module is the registered buffer itself (reference strides)
    sd = grouped.state_dict()
    assert sd["quant_weight"].stride() == (1, 32)
