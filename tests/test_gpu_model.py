"""-m gpu: model.py pieces, the whole tiny model, generate() and the 7B-shaped Block
against the oracle and the golden vectors produced by the unmodified reference."""
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

from oracle import llama_oracle as O  # noqa: E402

CFG = dict(block_size=64, vocab_size=96, n_layer=2, n_head=4, n_embd=128)
RTOL, ATOL = 1e-3, 5e-3  # the reference's bf16 tolerance, tests/test_model.py:133


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def test_rmsnorm_and_rope_match_reference(dev):
    import lit_llama_b200 as P

    g = load_golden("ops.pt")
    n = P.RMSNorm(128).to(dev).bfloat16()
    n.scale.data = g["rms_scale"].bfloat16().to(dev)
    xg = g["rms_x"].bfloat16().to(dev)
    y = n(xg).cpu()
    # vs the reference run on the CPU: two bf16 ulps (torch's CPU mean rounds the sum to bf16 before
    # dividing, its CUDA mean does not - the reference itself differs between devices here)
    torch.testing.assert_close(y.float(), g["rms_y_bf16"].float(), rtol=2 ** -6, atol=1e-6)  # two bf16 ulps
    # vs the reference formula (model.py:270-277) evaluated by torch on THIS device in bf16: same rounding points
    ms = torch.mean(xg * xg, dim=-1, keepdim=True)
    yt = (n.scale.data * (xg * torch.rsqrt(ms + 1e-5))).cpu()
    assert float((y == yt).float().mean()) > 0.995
    yr = P.apply_rope(g["rope_x"].bfloat16().to(dev), g["rope_table_64x32"].to(dev)).cpu()
    assert torch.equal(yr, g["rope_y_bf16"])  # fp32 products and sums in the reference's order: bit-exact
    tab = P.build_rope_cache(64, 32, torch.int64, dev)
    torch.testing.assert_close(tab.cpu(), g["rope_table_64x32"], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("graph_after", [0, 2])
def test_tiny_model_matches_reference(dev, graph_after):
    from gpu_util import build_tiny

    gd = load_golden("tiny_int4_bf16.pt")
    model, _, _ = build_tiny(dev, CFG)
    model.graph_after = graph_after
    S = 16
    with torch.no_grad():
        got = [model(gd["prompt"].view(1, -1).to(dev), S, torch.arange(7, device=dev))]
        for i, t in enumerate(gd["steps_tokens"]):
            got.append(model(torch.tensor([[t]], device=dev), S, torch.tensor([7 + i], device=dev)))
    for a, b in zip(got, gd["steps_logits"]):
        torch.testing.assert_close(a.float().cpu(), b.float(), rtol=RTOL, atol=ATOL)
    k, v = model.kv_caches[0]
    torch.testing.assert_close(k.float().cpu(), gd["kv0_k"].float(), rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(v.float().cpu(), gd["kv0_v"].float(), rtol=RTOL, atol=ATOL)
    model.reset_cache()
    with torch.no_grad():
        lg = model(gd["prompt"].view(1, -1).to(dev))
    torch.testing.assert_close(lg.float().cpu(), gd["nocache_logits"].float(), rtol=RTOL, atol=ATOL)


def test_roll_branch_matches_reference(dev):
    from gpu_util import build_tiny

    gd = load_golden("tiny_int4_bf16.pt")
    model, _, _ = build_tiny(dev, CFG)
    S2 = 8
    with torch.no_grad():
        got = [model(gd["prompt"].view(1, -1).to(dev), S2, torch.arange(7, device=dev))[:, -1]]
        for i, t in enumerate(gd["roll_tokens"]):
            got.append(model(torch.tensor([[t]], device=dev), S2, torch.tensor([7 + i], device=dev))[:, -1])
    for a, b in zip(got, gd["roll_logits"]):
        torch.testing.assert_close(a.float().cpu(), b.float(), rtol=RTOL, atol=ATOL)
    kl = model.logical_kv_caches()[1][0]
    torch.testing.assert_close(kl.float().cpu(), gd["roll_kv1_k"].float(), rtol=RTOL, atol=ATOL)


def test_generate_matches_reference_tokens(dev):
    import lit_llama_b200 as P
    from gpu_util import build_tiny

    gd = load_golden("tiny_int4_bf16.pt")
    model, oracle, _ = build_tiny(dev, CFG)
    prompt = gd["prompt"].to(torch.int32).to(dev)
    y = P.generate(model, prompt, 12, top_k=1)
    assert y.shape == gd["gen_greedy"].shape and y.dtype == torch.int32
    assert torch.equal(y[:7].cpu(), gd["prompt"].to(torch.int32))
    # greedy tokens: equal to the reference's unless two logits tie within bf16 noise
    same = (y.cpu() == gd["gen_greedy"]).float().mean()
    assert same >= 0.9, (y.cpu().tolist(), gd["gen_greedy"].tolist())
    # loop semantics of tests/test_generate.py:26-54: length, order of the sampled tokens, roll branch
    model.reset_cache()
    from unittest import mock

    draws = []
    orig = torch.multinomial

    def spy(*a, **k):
        out = orig(*a, **k)
        draws.append(out)
        return out

    with mock.patch("torch.multinomial", spy):
        out = P.generate(model, prompt, 20, max_seq_length=10, top_k=4)
    assert out.size(0) == 7 + 20
    assert torch.equal(out.cpu(), torch.cat((prompt.cpu(), torch.hstack(draws).cpu().to(torch.int32))))
    # eos stops and includes the eos token (generate.py:88-89)
    model.reset_cache()
    first = int(P.generate(model, prompt, 1, top_k=1)[-1])
    model.reset_cache()
    out = P.generate(model, prompt, 5, top_k=1, eos_id=first)
    # generate.py:88-89 returns idx[:input_pos] with input_pos == position of the eos token, i.e. the
    # prompt only (the reference's comment says "include the EOS token"; its slice does not) - mirrored
    assert out.tolist() == prompt.tolist()
    assert torch.equal(out.cpu(), O.generate(oracle, prompt.cpu(), 5, top_k=1, eos_id=first))


def test_fast_path_equals_module_path(dev):
    """b2l_decode_step (fused, graph) vs the module-by-module path on the same step."""
    from gpu_util import build_tiny

    model, _, _ = build_tiny(dev, CFG)
    prompt = torch.tensor([[3, 17, 40, 41, 2, 77, 5]], device=dev)
    with torch.no_grad():
        model(prompt, 16, torch.arange(7, device=dev))
        fast = model(torch.tensor([[9]], device=dev), 16, torch.tensor([7], device=dev)).clone()
        model.reset_cache()
        model._fast_ok = False
        model(prompt, 16, torch.arange(7, device=dev))
        slow = model(torch.tensor([[9]], device=dev), 16, torch.tensor([7], device=dev))
    torch.testing.assert_close(fast.float(), slow.float(), rtol=RTOL, atol=ATOL)


def test_reloading_weights_invalidates_the_baked_decode_state(dev):
    """load_state_dict after decode steps (argument block and CUDA graph already built on the old tilings): the next
    step must use the new weights -- the decode state is rebuilt, not replayed on stale pointers."""
    from gpu_util import build_tiny

    model, _, _ = build_tiny(dev, CFG, seed=1234)
    fresh, _, sd2 = build_tiny(dev, CFG, seed=4321)
    prompt = torch.tensor([[3, 17, 40, 41, 2, 77, 5]], device=dev)

    def run(m):
        m.reset_cache()
        out = [m(prompt, 16, torch.arange(7, device=dev))]
        for i, t in enumerate([9, 11, 60, 2]):   # graph replay from the third step
            out.append(m(torch.tensor([[t]], device=dev), 16, torch.tensor([7 + i], device=dev)).clone())
        return out

    with torch.no_grad():
        old = run(model)
        model.load_state_dict(sd2)
        new, want = run(model), run(fresh)
    assert not torch.equal(old[-1], new[-1])
    for a, b in zip(new, want):
        assert torch.equal(a, b)


def test_compact_keeps_one_copy_and_changes_nothing(dev):
    """LLaMA.compact(): the reference-layout buffers and duplicate tilings are freed (one resident copy = the batch-1
    decode tiling), prefill / batch-1 / batch-2 decode results stay bit-identical, state_dict() still yields the
    reference's tensors bit for bit (rebuilt from the tiling), and load_state_dict() brings the buffers back."""
    from gpu_util import build_tiny

    model, _, sd = build_tiny(dev, CFG, seed=77)
    twin, _, _ = build_tiny(dev, CFG, seed=77)
    prompt = torch.tensor([[3, 17, 40, 41, 2, 77, 5]], device=dev)

    def run(m, B=1):
        m.reset_cache()
        out = [m(prompt.repeat(B, 1), 16, torch.arange(7, device=dev))]
        for i, t in enumerate([9, 11, 60, 2]):
            out.append(m(torch.full((B, 1), t, device=dev), 16, torch.tensor([7 + i], device=dev)).clone())
        return out

    with torch.no_grad():
        before = run(model)
        before_sd = {k: v.clone() for k, v in model.state_dict().items()}
        torch.cuda.synchronize()
        model.reset_cache()
        m0 = torch.cuda.memory_allocated()
        model.compact()
        torch.cuda.synchronize()
        m1 = torch.cuda.memory_allocated()
        after = run(model)
        after2, want2 = run(model, B=2), run(twin, B=2)
    assert m1 < m0, (m0, m1)
    for a, b in zip(before, after):
        assert torch.equal(a, b)
    for a, b in zip(after2, want2):
        assert torch.equal(a, b)
    lin = model.transformer.h[0].attn.c_attn
    assert lin.quant_weight.numel() == 0 and model.transformer.h[1].mlp.c_fc1._tiled_i8 is None
    got_sd = model.state_dict()
    assert got_sd.keys() == before_sd.keys()
    for k, v in before_sd.items():
        assert torch.equal(got_sd[k], v), k
        if k.endswith("quant_weight"):
            assert got_sd[k].stride() == v.stride(), k
    # a new checkpoint after compaction: buffers come back, results follow the new weights
    other, _, sd2 = build_tiny(dev, CFG, seed=78)
    with torch.no_grad():
        model.load_state_dict(sd2)
        for a, b in zip(run(model), run(other)):
            assert torch.equal(a, b)
    assert lin.quant_weight.numel() > 0


def test_7b_shaped_block_vs_oracle(dev):
    """One Block + lm_head at the BASELINE 7B widths (n_embd 4096, 32 heads of 128, n_hidden
    11008, vocab 32000): prefill 5 tokens (tcgen05 kernel, prefill attention) then 3 decode
    steps (batch-1 kernel, fused attention), against the oracle in both of the reference's
    arithmetics: its GPU branch (fp32 dequant) tightly, its dense CPU branch (bf16-rounded
    weights, ~1e-3 noise per linear) loosely."""
    from gpu_util import build_tiny

    cfg = dict(block_size=32, vocab_size=32000, n_layer=1, n_head=32, n_embd=4096)
    model, exact, sd = build_tiny(dev, cfg, seed=11, exact_linears=True)
    dense = O.OracleLLaMA.from_state_dict(sd, 1, 32, 32, "gptq.int4")
    prompt = torch.tensor([[5, 100, 31999, 7, 2048]])
    S = 8
    with torch.no_grad():
        got = [model(prompt.to(dev), S, torch.arange(5, device=dev))]
        want = [exact.forward(prompt, S, torch.arange(5))]
        loose = [dense.forward(prompt, S, torch.arange(5))]
        for i, t in enumerate([77, 12345, 9]):
            got.append(model(torch.tensor([[t]], device=dev), S, torch.tensor([5 + i], device=dev)))
            want.append(exact.forward(torch.tensor([[t]]), S, torch.tensor([5 + i])))
            loose.append(dense.forward(torch.tensor([[t]]), S, torch.tensor([5 + i])))
    for a, b, c in zip(got, want, loose):
        a, b, c = a.float().cpu(), b.float(), c.float()
        scale = b.abs().max()
        # every module output is rounded to bf16 (2^-9 normwise each) on 4096..11008-wide vectors and
        # single-ulp flips propagate through the next RMSNorm/linear: a percent normwise end to end
        ours = float((a - b).norm() / b.norm())
        # the measured anchor of that bound: the REFERENCE's own bf16 CPU arithmetic (dense branch, bf16-rounded
        # weights) sits this far from the same exact-arithmetic result; ours must not be farther than it is
        # (plus the bf16 rounding of the logits themselves)
        ref = float((c - b).norm() / b.norm())
        assert ours < 2e-2, (ours, ref)
        assert ours <= 1.25 * ref + 2.0 ** -8, (ours, ref)
        assert (a - b).abs().max() < 0.05 * scale
        assert (a - c).norm() / c.norm() < 3e-2
    k, v = model.kv_caches[0]
    torch.testing.assert_close(k[:, :, :8].float().cpu(), exact.kv[0][0].float(), rtol=2 ** -6, atol=2e-2)
    torch.testing.assert_close(v[:, :, :8].float().cpu(), exact.kv[0][1].float(), rtol=2 ** -6, atol=2e-2)


def test_13b_width_batch8_prefill_and_decode_vs_oracle(dev):
    """BASELINE.json configs[3] in small: two Blocks at the LLaMA-13B widths (n_embd 5120, 40 heads of 128, n_hidden
    13824), batch 8: prefill 32 tokens per sequence (tcgen05 GEMM at M = 256, tensor-core prefill attention), then 4
    decode steps (2..8-row mma.sync kernel, fused attention, CUDA graph from the third step), every logits tensor and
    the KV cache against the oracle in exact arithmetic."""
    from gpu_util import build_tiny

    cfg = dict(block_size=64, vocab_size=512, n_layer=2, n_head=40, n_embd=5120)
    model, exact, _ = build_tiny(dev, cfg, seed=3, exact_linears=True)
    g = torch.Generator().manual_seed(0)
    B, T, S = 8, 32, 40
    prompt = torch.randint(0, 512, (B, T), generator=g)
    steps = [torch.randint(0, 512, (B, 1), generator=g) for _ in range(4)]
    with torch.no_grad():
        got = [model(prompt.to(dev), S, torch.arange(T, device=dev))]
        want = [exact.forward(prompt, S, torch.arange(T))]
        for i, t in enumerate(steps):
            got.append(model(t.to(dev), S, torch.tensor([T + i], device=dev)))
            want.append(exact.forward(t, S, torch.tensor([T + i])))
    for a, b in zip(got, want):
        a, b = a.float().cpu(), b.float()
        assert a.shape == b.shape
        assert (a - b).norm() / b.norm() < 2e-2, float((a - b).norm() / b.norm())
        for r in range(B):   # every sequence on its own: a row mix-up cannot hide in the batch norm
            assert (a[r] - b[r]).norm() / b[r].norm() < 3e-2, (r, float((a[r] - b[r]).norm() / b[r].norm()))
    for li in range(2):
        k, v = model.kv_caches[li]
        # cache rows are bf16 outputs of a 5120-wide linear whose input already carries the first Block's rounding noise:
        # normwise like the logits, elementwise within two bf16 ulps of values this size (measured on B200: 2 of 1.5 M
        # elements differ by 0.039 at |x| ~ 0.5..8, everything else within one ulp)
        for got_c, want_c in ((k, exact.kv[li][0]), (v, exact.kv[li][1])):
            g_, w_ = got_c[:, :, :T + 4].float().cpu(), want_c[:, :, :T + 4].float()
            assert (g_ - w_).norm() / w_.norm() < 2e-2
            torch.testing.assert_close(g_, w_, rtol=2 ** -5, atol=8e-2)


@pytest.mark.parametrize("S,cases", [
    (300, [(0, 0), (5, 0), (127, 0), (128, 0), (299, 0), (300, 0), (333, 7)]),          # 3 splits
    (128, [(0, 0), (127, 0), (130, 3)]),                                                 # single split
    (256, [(100, 0), (128, 0), (255, 0), (256, 5)]),                                     # 2 splits
    (2048, [(3, 0), (129, 0), (1023, 0), (1024, 0), (1500, 0), (2047, 0), (2050, 11)]),  # 16 splits
])
def test_fused_attention_equals_unfused(dev, S, cases):
    """head_size 128 single-token attention: the fused kernel (rope + append + split-S + ticketed
    merge) against the three-kernel path on identical inputs, at several positions including a full
    cache and the roll branch."""
    from lit_llama_b200 import _lib as L

    B, nh, hs, blk = 2, 8, 128, max(512, S)
    C = nh * hs
    lib = L.lib()
    g = torch.Generator(device=dev).manual_seed(3)
    rope = O.rope_table(blk, hs).to(dev)
    kc = (torch.randn(B, nh, S, hs, device=dev, generator=g) * 0.5).bfloat16()
    vc = (torch.randn(B, nh, S, hs, device=dev, generator=g) * 0.5).bfloat16()
    for pos, ring0 in cases:
        qkv = torch.randn(B, 1, 3 * C, device=dev, generator=g).bfloat16()
        outs = []
        for flags in (0, 8):
            k1, v1, q1 = kc.clone(), vc.clone(), qkv.clone()
            ring = torch.tensor([ring0], dtype=torch.int32, device=dev)
            p = torch.tensor([pos], dtype=torch.int64, device=dev)
            L.check(lib.b2l_ring_advance(p.data_ptr(), 1, ring.data_ptr(), S, L.stream_ptr()), "ring")
            work = torch.zeros(lib.b2l_attn_workspace_bytes(B, nh, hs, 1, S) // 4 + 1, device=dev, dtype=torch.float32)
            y = torch.empty(B, 1, C, device=dev, dtype=torch.bfloat16)
            for rep in range(2 if flags == 0 else 1):  # fused path twice: its ticket counters must re-arm themselves
                rc = lib.b2l_attention(q1.data_ptr(), k1.data_ptr(), v1.data_ptr(), rope.data_ptr(), p.data_ptr(), ring.data_ptr(),
                                       y.data_ptr(), work.data_ptr(), B, 1, nh, hs, S, blk, flags, L.stream_ptr())
                assert rc == 0, lib.b2l_last_error()
            torch.cuda.synchronize()
            outs.append((y, k1, v1))
        (yf, kf, vf), (yu, ku, vu) = outs
        assert torch.equal(kf, ku) and torch.equal(vf, vu), pos      # appended rows bit-identical
        torch.testing.assert_close(yf.float(), yu.float(), rtol=2 ** -7, atol=2e-3)


@pytest.mark.parametrize("B", [1, 8])
def test_fused_attention_vs_oracle_hs128(dev, B):
    """The kernel on the benched path (fused rope + KV append + split-S attention + merge, head_size 128) directly
    against the oracle's restatement of model.py:197-230 (O.rope_apply + index_copy / roll + O.sdpa): positions 0,
    127, 128 (sub-tile boundary of this kernel), 255, 256 (split boundary of this kernel), 1023, 2047 (full
    cache, 8 splits), and two roll states (model.py:214-218: position >= S with different ring offsets)."""
    from lit_llama_b200 import _lib as L

    nh, hs, S, blk = 4, 128, 2048, 4096
    C = nh * hs
    lib = L.lib()
    g = torch.Generator(device=dev).manual_seed(17 + B)
    rope = O.rope_table(blk, hs)
    rope_d = rope.to(dev)
    kc = (torch.randn(B, nh, S, hs, device=dev, generator=g) * 0.5).bfloat16()
    vc = (torch.randn(B, nh, S, hs, device=dev, generator=g) * 0.5).bfloat16()
    for pos, ring0 in [(0, 0), (127, 0), (128, 0), (255, 0), (256, 0), (1023, 0), (2047, 0), (2048, 0), (3000, 777)]:
        qkv = torch.randn(B, 1, 3 * C, device=dev, generator=g).bfloat16()
        k1, v1 = kc.clone(), vc.clone()
        ring = torch.tensor([ring0], dtype=torch.int32, device=dev)
        p = torch.tensor([pos], dtype=torch.int64, device=dev)
        L.check(lib.b2l_ring_advance(p.data_ptr(), 1, ring.data_ptr(), S, L.stream_ptr()), "ring")
        work = torch.zeros(lib.b2l_attn_workspace_bytes(B, nh, hs, 1, S) // 4 + 1, device=dev, dtype=torch.float32)
        y = torch.empty(B, 1, C, device=dev, dtype=torch.bfloat16)
        rc = lib.b2l_attention(qkv.clone().data_ptr(), k1.data_ptr(), v1.data_ptr(), rope_d.data_ptr(), p.data_ptr(), ring.data_ptr(),
                               y.data_ptr(), work.data_ptr(), B, 1, nh, hs, S, blk, 0, L.stream_ptr())
        assert rc == 0, lib.b2l_last_error()
        torch.cuda.synchronize()
        # ---- oracle on the logical cache
        kl = torch.roll(kc.cpu(), -ring0, dims=2)   # logical slot j = physical (j + ring0) % S
        vl = torch.roll(vc.cpu(), -ring0, dims=2)
        q, k, v = qkv.cpu().split(C, dim=2)
        rows = rope[pos : pos + 1]
        q = O.rope_apply(q.view(B, 1, nh, hs), rows).transpose(1, 2)
        k = O.rope_apply(k.view(B, 1, nh, hs), rows).transpose(1, 2)
        v = v.view(B, 1, nh, hs).transpose(1, 2)
        slot = pos
        if pos >= S:   # model.py:214-218
            slot = S - 1
            kl, vl = torch.roll(kl, -1, dims=2), torch.roll(vl, -1, dims=2)
        kl = kl.index_copy(2, torch.tensor([slot]), k)
        vl = vl.index_copy(2, torch.tensor([slot]), v)
        mask = (torch.arange(S) <= slot).view(1, 1, 1, S)
        want = O.sdpa(q, kl, vl, mask).transpose(1, 2).reshape(B, 1, C)
        got = y.cpu()
        err = (got.float() - want.float()).norm() / want.float().norm()
        assert err < 4e-3, (pos, ring0, float(err))   # fp32 softmax in a different summation order + one bf16 rounding (2^-9)
        torch.testing.assert_close(got.float(), want.float(), rtol=2 ** -7, atol=2e-3)
        # the appended row sits in the physical slot the ring assigns, bit-identical to the reference arithmetic
        ring_now = int(ring)
        assert ring_now == (ring0 + (1 if pos >= S else 0)) % S
        phys = (slot + ring_now) % S
        assert torch.equal(k1[:, :, phys].cpu(), k[:, :, 0]) and torch.equal(v1[:, :, phys].cpu(), v[:, :, 0]), (pos, ring0)


@pytest.mark.parametrize("ring0", [0, 37])
def test_prefill_attention_hs128_vs_oracle(dev, ring0):
    """T > 1 at head_size 128 (the tiled tensor-core prefill kernel): a 150-token chunk appended at positions 40..189
    of a partly filled (and possibly rotated) cache, and a 130-token no-cache forward, against the oracle's
    rope_apply + index_copy + masked fp32 sdpa (model.py:200-230)."""
    from lit_llama_b200 import _lib as L

    B, nh, hs, S, blk = 2, 3, 128, 256, 512
    C = nh * hs
    lib = L.lib()
    g = torch.Generator(device=dev).manual_seed(5 + ring0)
    rope = O.rope_table(blk, hs)
    rope_d = rope.to(dev)
    kc = (torch.randn(B, nh, S, hs, device=dev, generator=g) * 0.5).bfloat16()
    vc = (torch.randn(B, nh, S, hs, device=dev, generator=g) * 0.5).bfloat16()
    p0, T = 40, 150
    qkv = torch.randn(B, T, 3 * C, device=dev, generator=g).bfloat16()
    k1, v1, q1 = kc.clone(), vc.clone(), qkv.clone()
    ring = torch.tensor([ring0], dtype=torch.int32, device=dev)
    pos = torch.arange(p0, p0 + T, dtype=torch.int64, device=dev)
    work = torch.zeros(lib.b2l_attn_workspace_bytes(B, nh, hs, T, S) // 4 + 1, device=dev, dtype=torch.float32)
    y = torch.empty(B, T, C, device=dev, dtype=torch.bfloat16)
    rc = lib.b2l_attention(q1.data_ptr(), k1.data_ptr(), v1.data_ptr(), rope_d.data_ptr(), pos.data_ptr(), ring.data_ptr(), y.data_ptr(),
                           work.data_ptr(), B, T, nh, hs, S, blk, 0, L.stream_ptr())
    assert rc == 0, lib.b2l_last_error()
    torch.cuda.synchronize()
    kl, vl = torch.roll(kc.cpu(), -ring0, dims=2), torch.roll(vc.cpu(), -ring0, dims=2)
    q, k, v = qkv.cpu().split(C, dim=2)
    rows = rope[p0 : p0 + T]
    q = O.rope_apply(q.view(B, T, nh, hs), rows).transpose(1, 2)
    k = O.rope_apply(k.view(B, T, nh, hs), rows).transpose(1, 2)
    v = v.view(B, T, nh, hs).transpose(1, 2)
    kl = kl.index_copy(2, pos.cpu(), k)
    vl = vl.index_copy(2, pos.cpu(), v)
    mask = (torch.arange(S).view(1, S) <= pos.cpu().view(T, 1)).view(1, 1, T, S)
    want = O.sdpa(q, kl, vl, mask).transpose(1, 2).reshape(B, T, C)
    torch.testing.assert_close(y.float().cpu(), want.float(), rtol=2 ** -7, atol=2e-3)
    assert (y.float().cpu() - want.float()).norm() / want.float().norm() < 4e-3
    # ---- no cache (input_pos is None, model.py:104-106)
    T2 = 130
    qkv2 = torch.randn(B, T2, 3 * C, device=dev, generator=g).bfloat16()
    q2 = qkv2.clone()
    y2 = torch.empty(B, T2, C, device=dev, dtype=torch.bfloat16)
    work2 = torch.zeros(lib.b2l_attn_workspace_bytes(B, nh, hs, T2, T2) // 4 + 1, device=dev, dtype=torch.float32)
    rc = lib.b2l_attention_nocache(q2.data_ptr(), rope_d.data_ptr(), y2.data_ptr(), work2.data_ptr(), B, T2, nh, hs, blk, L.stream_ptr())
    assert rc == 0, lib.b2l_last_error()
    torch.cuda.synchronize()
    q, k, v = qkv2.cpu().split(C, dim=2)
    q = O.rope_apply(q.view(B, T2, nh, hs), rope[:T2]).transpose(1, 2)
    k = O.rope_apply(k.view(B, T2, nh, hs), rope[:T2]).transpose(1, 2)
    v = v.view(B, T2, nh, hs).transpose(1, 2)
    mask = torch.tril(torch.ones(T2, T2, dtype=torch.bool)).view(1, 1, T2, T2)
    want2 = O.sdpa(q, k, v, mask).transpose(1, 2).reshape(B, T2, C)
    torch.testing.assert_close(y2.float().cpu(), want2.float(), rtol=2 ** -7, atol=2e-3)


def test_batched_decode_rows_are_independent(dev):
    from gpu_util import build_tiny

    model, _, _ = build_tiny(dev, CFG)
    idx = torch.tensor([[3, 17, 40], [9, 9, 1]], device=dev)
    with torch.no_grad():
        model(idx, 16, torch.arange(3, device=dev))
        both = model(torch.tensor([[5], [60]], device=dev), 16, torch.tensor([3], device=dev)).clone()
        model.reset_cache()
        model(idx[1:], 16, torch.arange(3, device=dev))
        one = model(torch.tensor([[60]], device=dev), 16, torch.tensor([3], device=dev))
    torch.testing.assert_close(both[1:].float(), one.float(), rtol=RTOL, atol=ATOL)


def test_fused_sampling_head_matches_torch_ops(dev):
    """b2l_topk_softmax vs the reference's op sequence (generate.py:68-75) run by torch on the
    same device: same kept set (incl. ties at the threshold), probabilities within one bf16 ulp."""
    import lit_llama_b200 as P

    g = torch.Generator(device=dev).manual_seed(0)
    for V, k, temp in [(32000, 200, 0.8), (32000, 1, 1.0), (32000, None, 0.7), (128, 4, 2.0), (1000, 1000, 1.3), (50257, 50, 0.9)]:
        logits = (torch.randn(V, device=dev, generator=g) * 3).bfloat16()
        if V == 128:
            logits[5] = logits[9]  # a tie
        got = P.sample_probs(logits, temp, k)
        ref = logits / temp
        if k is not None:
            v, _ = torch.topk(ref, min(k, V))
            ref = torch.where(ref < v[[-1]], -float("Inf"), ref)
        want = torch.nn.functional.softmax(ref, dim=-1)
        assert torch.equal(got == 0, want == 0), (V, k)
        torch.testing.assert_close(got.float(), want.float(), rtol=2 ** -7, atol=1e-8)
        assert abs(float(got.float().sum()) - 1.0) < 2e-2


def test_fused_draw_equals_torch_multinomial(dev):
    """b2l_topk_softmax_sample: for the same generator state the token is the one `torch.multinomial(probs, 1)`
    draws from the kernel's own probabilities (generate.py:76) -- multinomial is argmax(probs / Exp(1) noise)."""
    import lit_llama_b200 as P

    for V, k, temp in [(32000, 200, 0.8), (32000, None, 1.0), (32003, 50, 0.7), (130, 4, 2.0), (1000, 1000, 1.3)]:
        for trial in range(12):
            logits = (torch.randn(V, device=dev) * (1 + trial % 4)).bfloat16()
            torch.manual_seed(1000 + trial)
            want = torch.multinomial(P.sample_probs(logits, temp, k), num_samples=1)
            torch.manual_seed(1000 + trial)
            got = P.sample_token(logits, temp, k)
            assert got.shape == (1,) and got.dtype == torch.int64
            assert int(got) == int(want), (V, k, trial)
    # the same RNG consumption as multinomial: the generator is in the same state afterwards
    logits = torch.randn(32000, device=dev).bfloat16()
    torch.manual_seed(5); torch.multinomial(P.sample_probs(logits, 0.8, 200), 1); a = torch.rand(4, device=dev)
    torch.manual_seed(5); P.sample_token(logits, 0.8, 200); b = torch.rand(4, device=dev)
    assert torch.equal(a, b)


def test_llm_int8_model_vs_oracle(dev):
    """--quantize llm.int8: tiny model, prefill + decode, against the oracle restatement."""
    from gpu_util import build_tiny

    cfg = dict(block_size=32, vocab_size=96, n_layer=2, n_head=4, n_embd=128)
    model, oracle, _ = build_tiny(dev, cfg, mode="llm.int8", seed=7)
    prompt = torch.tensor([[3, 17, 40, 41, 2]])
    with torch.no_grad():
        got = [model(prompt.to(dev), 16, torch.arange(5, device=dev))]
        want = [oracle.forward(prompt, 16, torch.arange(5))]
        for i, t in enumerate([9, 60, 3, 77, 12, 45]):  # > graph_after steps: the later ones are CUDA-graph replays
            got.append(model(torch.tensor([[t]], device=dev), 16, torch.tensor([5 + i], device=dev)))
            want.append(oracle.forward(torch.tensor([[t]]), 16, torch.tensor([5 + i])))
    assert model._module_graph is not None and model._module_graph["graph"] is not None
    for a, b in zip(got, want):
        a, b = a.float().cpu(), b.float()
        assert (a - b).norm() / b.norm() < 2e-2, float((a - b).norm() / b.norm())
