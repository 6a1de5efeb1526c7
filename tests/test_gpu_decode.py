"""-m gpu: the fused decode step (b2l_decode_step, one kernel per op) against the CPU oracle on head_size-128 models
small enough for the oracle: short and deep positions (both sides of the attention kernel's 256-key split
boundary), a full cache, the roll branch (model.py:214-218), graph replay, greedy generation, PDL vs plain stream
order and tensor parallelism."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import llama_oracle as O  # noqa: E402

# head_size 128 (the fused single-token attention kernel's shape), K = 256 / 768: every linear a multiple of 64 wide
CFG = dict(block_size=512, vocab_size=320, n_layer=3, n_head=2, n_embd=256)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _normwise(a, b):
    a, b = a.float().cpu().flatten(), b.float().cpu().flatten()
    return float((a - b).norm() / b.norm())


def _decode(model, oracle, dev, prompt, S, steps, seed=0):
    """Prefill `prompt`, then `steps` single-token steps; returns ([model logits], [oracle logits])."""
    g = torch.Generator().manual_seed(seed)
    T = prompt.shape[1]
    got, want = [], []
    with torch.no_grad():
        got.append(model(prompt.to(dev), S, torch.arange(T, device=dev))[:, -1])
        if oracle is not None:
            want.append(oracle.forward(prompt, S, torch.arange(T))[:, -1])
        for i in range(steps):
            t = int(torch.randint(0, CFG["vocab_size"], (1,), generator=g))
            got.append(model(torch.tensor([[t]], device=dev), S, torch.tensor([T + i], device=dev))[:, -1])
            if oracle is not None:
                want.append(oracle.forward(torch.tensor([[t]]), S, torch.tensor([T + i]))[:, -1])
    return got, want


@pytest.mark.parametrize("S,T0,steps", [(300, 120, 20), (300, 250, 70), (128, 120, 20)])
def test_deep_context_and_roll_vs_oracle(dev, S, T0, steps):
    """Positions crossing the attention kernel's 128-key sub-tile and 256-key split boundaries, a full cache and the
    roll branch: every step's logits vs the exact-arithmetic oracle (normwise), the ring start and the logical cache
    order vs the oracle's."""
    from gpu_util import build_tiny

    torch.manual_seed(S + T0)
    prompt = torch.randint(0, CFG["vocab_size"], (1, T0))
    model, oracle, _ = build_tiny(dev, CFG, seed=5, exact_linears=True)
    got, want = _decode(model, oracle, dev, prompt, S, steps, seed=1)
    assert model._decode is not None and model._decode.graph is not None   # fused step, replayed as a graph
    for i, (a, b) in enumerate(zip(got, want)):
        assert _normwise(a, b) < 1.5e-2, (i, _normwise(a, b))
    assert int(model._ring) == max(0, T0 + steps - S)
    # logical order == the oracle's rolled cache
    kl = model.logical_kv_caches()[0][0]
    torch.testing.assert_close(kl.float().cpu(), oracle.kv[0][0].float(), rtol=2 ** -6, atol=3e-2)


def test_greedy_generate_equals_oracle_tokens(dev):
    import lit_llama_b200 as P
    from gpu_util import build_tiny

    model, oracle, _ = build_tiny(dev, CFG, seed=9)
    prompt = torch.tensor([5, 100, 319, 7, 48, 1, 250], dtype=torch.int32)
    y = P.generate(model, prompt.to(dev), 40, top_k=1)
    want = O.generate(oracle, prompt, 40, top_k=1)
    same = float((y.cpu() == want).float().mean())
    assert same >= 0.9, (y.cpu().tolist(), want.tolist())


def test_per_op_path_pdl_equals_plain_order(dev):
    """Programmatic dependent launch must not change a single bit: 24 decode steps of the one-kernel-per-op path
    with PDL (every activation read after griddepcontrol.wait is a coherent load) vs plain stream order."""
    from gpu_util import build_tiny

    outs = []
    for flags in (1, 0):
        model, _, _ = build_tiny(dev, CFG, seed=13)
        model.decode_flags = flags
        got, _ = _decode(model, None, dev, torch.tensor([[3, 17, 40, 41, 2, 77, 5, 9]]), 160, 24, seed=2)
        outs.append(torch.stack(got))
    assert torch.equal(outs[0], outs[1])
    # and for a batch of 4 (two-launch batch kernel, PDL between its launches)
    outs = []
    for flags in (1, 0):
        model, _, _ = build_tiny(dev, CFG, seed=13)
        model.decode_flags = flags
        idx = torch.tensor([[3, 17, 40], [9, 9, 1], [100, 2, 7], [64, 65, 66]], device=dev)
        with torch.no_grad():
            model(idx, 64, torch.arange(3, device=dev))
            step = [model(torch.full((4, 1), 5 + i, device=dev), 64, torch.tensor([3 + i], device=dev)).clone() for i in range(12)]
        outs.append(torch.stack(step))
    assert torch.equal(outs[0], outs[1])


def test_tensor_parallel_matches_single_gpu(dev):
    """TPLLaMA on 2 GPUs (module path and the fused graph-replayed rank step) vs the single-GPU model: tests/tp_check.py
    under torch.distributed.run.  Skipped on a one-GPU box."""
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29517", os.path.join(root, "tests", "tp_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("OK") >= 2, r.stdout[-2000:]
