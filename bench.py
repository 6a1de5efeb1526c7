"""bench.py - LLaMA-7B gptq.int4 batch-1 decode throughput on B200 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A step = one decoded token (one pass of generate()'s loop body, generate.py:63-89: model forward + top-k / softmax /
multinomial sampling) on random-init 7B gptq.int4 weights, KV cache S = 2048.  Each decode step of the warm-up and timed
loops reads its input token from a fixed seeded sequence instead of the previous step's sample (the sampling still runs
on every step), so no step's input depends on how the build under test rounds.  The K timed steps are spread EVENLY over
positions 16..2047 whatever K is (a stride, not consecutive positions), so `value` is a true ctx-2048 mean;
`config.points` adds tokens/s at fixed positions 128, 1024 and 2047.  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes what the last timed step returned on rank 0, as float32 arrays: DIR/logits.npy (the model's
(1, 1, 32000) logits) and DIR/token.npy (the sampled token).  Weights, prompt, input tokens and sampling noise are drawn
from fixed seeds, so the same arguments give the same inputs on every run, and two builds that round differently give
logits that differ by their rounding only (the token can differ only where that rounding decides a near-tie).

  value     tokens/s, device-timed (CUDA events), inputs resident in HBM, no host sync
  e2e       same loop driven from HOST buffers: per step a pinned H2D copy of the token and position, and a D2H read
            of the sampled token
  roofline  the dominant kernel, q4_gemv_kernel (exact int8-digit MMA): algorithmic bytes of all its launches in one
            token / their summed duration, against MEASURED_PEAKS.json hbm_gbs; whole_token_* = the same for the full
            step (weights + KV bytes of the timed positions) from `value`
  cpu_baseline / --impl reference: the UNMODIFIED reference model (lit_llama.model.LLaMA under
            quantization("gptq.int4"), installed from the reference checkout into oracle/_ref by
            __graft_entry__.build()) on the host cores, same synthetic weights as the GPU arm, whole tokens through
            all 32 Blocks; the token loop is the golden-pinned restatement of generate.py (oracle/llama_oracle.py).
            Fallback when oracle/_ref is absent: the oracle port (kind "port").
N > 1: `value` = independent replicas, one process per GPU (the reference has no multi-GPU inference, SURVEY.md section
2.1; 7B fits one GPU): weak scaling, no data-path collective.  The same run then measures the TENSOR-PARALLEL path on
the same ranks and reports it under "tp": LLaMA-7B split N ways, and LLaMA-65B gptq.int4 TP = 8 (BASELINE.json
configs[4]) when N = 8 -- fused per-rank step, two one-shot all-reduces per Block over peer memory (tools/tp_bench.py).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "7B"
S_CTX = 2048
PROMPT_T = 16
TOP_K, TEMPERATURE = 200, 0.8  # generate.py:99-100 defaults


LLAMA_SHAPES = {"7B": (32, 32, 4096), "13B": (40, 40, 5120), "30B": (60, 52, 6656), "65B": (80, 64, 8192)}  # model.py:43-48


def n_hidden_for(n_embd: int) -> int:
    """model.py:243-245: find_multiple(int(2 * 4 * n_embd / 3), 256)."""
    h = int(2 * 4 * n_embd / 3)
    return h if h % 256 == 0 else h + 256 - h % 256


def model_bytes(cfg_name: str):
    """Algorithmic bytes of SURVEY.md section 8d for batch 1: W (packed int4 linears incl. lm_head, bf16 scales and
    zeros, RMSNorm scales, one wte row) and KV bytes per position."""
    L, _, C = LLAMA_SHAPES[cfg_name]
    nh, V = n_hidden_for(C), 32000
    lin_params = L * (3 * C * C + C * C + 3 * C * nh) + V * C
    lin_rows = L * (3 * C + C + 2 * nh + C) + V
    W = lin_params // 2 + lin_rows * 2 * 2 + (2 * L + 1) * C * 2 + C * 2
    kv_per_pos = 2 * L * C * 2
    return W, kv_per_pos


def synth_state(name, seed=1234, dev=None):
    """Random-init gptq.int4 weights of the named size: the direct synthesis of SURVEY.md section 8d (uniform levels,
    zero 8, per-row scales).  Drawn with the generator of `dev` (default: cuda:0 when there is one, so that the GPU
    arm and the CPU reference arm -- which moves the tensors to the host -- hold IDENTICAL weights)."""
    import torch

    if dev is None:
        dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    L, _, C = LLAMA_SHAPES[name]
    nh, V = n_hidden_for(C), 32000
    g = torch.Generator(device=dev).manual_seed(seed)
    std = 0.02 / (2 * L) ** 0.5
    sd = {}

    def lin(prefix, out_f, in_f):
        sd[prefix + ".quant_weight"] = torch.empty((in_f // 2, out_f), dtype=torch.uint8, device=dev).random_(0, 256, generator=g).t()  # strides (1, out)
        sd[prefix + ".scales"] = ((0.75 + 0.5 * torch.rand((out_f, 1), generator=g, device=dev)) * (std / 4.61)).to(torch.bfloat16)
        sd[prefix + ".zeros"] = torch.full((out_f, 1), 8.0, dtype=torch.bfloat16, device=dev)

    sd["transformer.wte.weight"] = (torch.randn((V, C), generator=g, device=dev) * 0.02).to(torch.bfloat16)
    for i in range(L):
        p = f"transformer.h.{i}."
        sd[p + "rms_1.scale"] = torch.ones(C, dtype=torch.bfloat16, device=dev)
        sd[p + "rms_2.scale"] = torch.ones(C, dtype=torch.bfloat16, device=dev)
        lin(p + "attn.c_attn", 3 * C, C)
        lin(p + "attn.c_proj", C, C)
        lin(p + "mlp.c_fc1", nh, C)
        lin(p + "mlp.c_fc2", nh, C)
        lin(p + "mlp.c_proj", C, nh)
    sd["transformer.ln_f.scale"] = torch.ones(C, dtype=torch.bfloat16, device=dev)
    lin("lm_head", V, C)
    return sd


def build_synthetic_model(name, dev, seed=1234, state=None):
    """The B200 model of the named size holding synth_state(name, seed) (same tensors as the CPU reference arm)."""
    import torch

    import lit_llama_b200 as P
    from lit_llama_b200.utils import quantization

    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device(dev), quantization("gptq.int4"):
            model = P.LLaMA.from_name(name)
    finally:
        torch.set_default_dtype(prev)
    sd = state if state is not None else synth_state(name, seed, dev)
    with torch.no_grad():
        own = model.state_dict()
        for k, v in sd.items():
            own[k].copy_(v)     # in place: keeps the reference strides of quant_weight
    return model.eval()


class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.samples:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7 or not (t0 - 0.15 <= t <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def sample_next(logits, top_k=TOP_K, temperature=TEMPERATURE):
    """generate.py:68-76 as lit_llama_b200.generate() runs it on the GPU (fused temperature /
    top-k / softmax / draw kernel on torch's Exp(1) noise = torch.multinomial's sample); the CPU baseline keeps the reference's torch ops."""
    import torch

    if logits.is_cuda:
        from lit_llama_b200 import sample_token

        return sample_token(logits[0, -1], temperature, top_k)
    logits = logits[0, -1] / temperature
    v, _ = torch.topk(logits, min(top_k, logits.size(-1)))
    logits = torch.where(logits < v[[-1]], -float("Inf"), logits)
    probs = torch.nn.functional.softmax(logits, dim=-1)
    return torch.multinomial(probs, num_samples=1)


def host_threads():
    """Threads for the CPU arm: every core this process may use (torchrun exports OMP_NUM_THREADS=1, which would
    silently turn the baseline into a single-core run), capped at 32 -- the reference's CPU path is a chain of small
    torch ops per Linear and runs SLOWER beyond that on a 100+-thread host (measured in round 1: 7.4x swings)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, int(os.environ.get("B2L_CPU_THREADS", "32"))))


def reference_model(state):
    """The UNMODIFIED reference model on the CPU: lit_llama.model.LLaMA built under lit_llama.utils.quantization
    ("gptq.int4") from oracle/_ref (pip-installed from the reference checkout by __graft_entry__.build(); the three
    file `lightning` stand-in oracle/_shim satisfies lit_llama/utils.py:15).  None when oracle/_ref is absent."""
    import torch

    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "lit_llama")):
        return None
    for pth in (os.path.join(ROOT, "oracle", "_shim"), ref_dir):
        if pth not in sys.path:
            sys.path.insert(0, pth)
    from lit_llama.model import LLaMA  # noqa: E402  (the reference's own class)
    from lit_llama.utils import quantization  # noqa: E402

    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with quantization("gptq.int4"):
            model = LLaMA.from_name(MODEL)
    finally:
        torch.set_default_dtype(prev)
    own = model.state_dict()
    with torch.no_grad():
        for k, v in state.items():
            own[k].copy_(v.cpu())
    return model.eval()


def cpu_reference_tokens(n_tokens, budget_s, prompt_t=8):
    """Decode on the host with the reference's own model code: prefill `prompt_t` tokens (untimed), then whole decoded
    tokens (all 32 Blocks + lm_head + the reference's sampling ops) until `n_tokens` are done or `budget_s` is spent
    (always at least one).  Returns the cpu_baseline dict; value = 1 / median seconds per token."""
    import torch

    from oracle import llama_oracle as O

    threads = host_threads()
    torch.set_num_threads(threads)
    state = synth_state(MODEL, 1234)
    model = reference_model(state)
    kind = "reference"
    if model is None:   # oracle/_ref missing (the reference checkout was not available at build time): the pinned port
        kind = "port"
        cpu = {k: v.cpu() for k, v in state.items()}
        L, nh, _ = LLAMA_SHAPES[MODEL]
        model = O.OracleLLaMA.from_state_dict(cpu, L, nh, S_CTX, "gptq.int4")
        fwd = model.forward
    else:
        fwd = model.__call__
    del state
    g = torch.Generator().manual_seed(7)
    prompt = torch.randint(0, 32000, (1, prompt_t), generator=g)
    times = []
    with torch.no_grad():
        logits = fwd(prompt, S_CTX, torch.arange(prompt_t))
        tok = sample_next(logits)
        t_start = time.perf_counter()
        for i in range(max(1, n_tokens)):
            t0 = time.perf_counter()
            logits = fwd(tok.view(1, 1), S_CTX, torch.tensor([prompt_t + i]))
            tok = sample_next(logits)
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_start > budget_s:
                break
    times.sort()
    med = times[len(times) // 2]
    what = ("unmodified reference model (lit_llama.model.LLaMA under quantization('gptq.int4'), oracle/_ref) " if kind == "reference"
            else "oracle port of the reference CPU path (oracle/_ref absent) ")
    return {"value": 1.0 / med, "unit": "tokens/s", "cores": threads, "kind": kind,
            "sample": f"{len(times)} whole decoded token(s) after a {prompt_t}-token prefill, all {LLAMA_SHAPES[MODEL][0]} Blocks + lm_head + sampling, "
                      f"median {med:.2f} s (min {times[0]:.2f}, max {times[-1]:.2f}); " + what +
                      "on the same synthetic weights as the GPU arm; token loop = generate.py:63-89 restated",
            "s_per_token": med, "tokens": len(times)}


def run_reference(args, rank, world):
    if rank != 0:
        return
    cb = cpu_reference_tokens(n_tokens=max(3, min(args.steps, 4)), budget_s=150.0)
    line = {"impl": "reference", "metric": "LLaMA-7B gptq.int4 decode tokens/sec", "value": cb["value"], "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": cb["tokens"], "warmup": 1, "ms_per_step": cb["s_per_token"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "LLaMA-7B gptq.int4 decode batch=1 ctx=2048 (random-init weights)", "where": "host CPU",
                       "positions": "8.. (the CPU path costs the same at every position: it attends over all 2048 slots)"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def time_q4_launches(model, dev):
    """Every launch of the batch-1 int4 linear kernel (q4_gemv_kernel) of one token, back to back (all
    layers' distinct weights: 3.3 GB, far beyond L2), timed with CUDA events."""
    import ctypes as C

    import torch

    from lit_llama_b200 import _lib as L

    st = model._decode
    a = st.args
    calls = []

    gemv = bool(a.lm_head.qw_mma)

    def mk(w, x, ldx, y, ldy, pro, ns, epi, res):
        return L.Q4LinearArgs(x=x, ldx=ldx, qw_tiled=w.qw_mma if gemv else w.qw_tiled, scales=w.scales, zeros=w.zeros, sz_dtype=a.sz_dtype, y=y, ldy=ldy,
                              M=1, N=w.N, K=w.K, prologue=pro, norm_scale=ns, eps=a.eps, epilogue=epi, res=res, ldres=ldy,
                              split_k=0, flags=1)  # PDL, as b2l_decode_step launches them

    Cd = a.n_embd
    for i in range(a.n_layer):
        ly = st.layers[i]
        calls.append(mk(ly.c_attn, a.x, Cd, a.qkv, 3 * Cd, 1, ly.rms_1, 0, None))
        calls.append(mk(ly.c_proj, a.att, Cd, a.x, Cd, 0, None, 1, a.x))
        calls.append(mk(ly.c_fc12, a.x, Cd, a.hid, a.n_hidden, 1, ly.rms_2, 2, None))
        calls.append(mk(ly.mlp_proj, a.hid, a.n_hidden, a.x, Cd, 0, None, 1, a.x))
    calls.append(mk(a.lm_head, a.x, Cd, a.logits, a.vocab, 1, a.ln_f, 0, None))
    lib, sp = L.lib(), L.stream_ptr()

    fn = lib.b2l_q4_gemv if gemv else lib.b2l_q4_linear_tc

    def run():
        for c in calls:
            rc = fn(C.byref(c), sp)
            if rc:
                raise RuntimeError(lib.b2l_last_error().decode())

    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3, len(calls), ("q4_gemv_kernel" if gemv else "q4_linear_tc_kernel")


def build_line(args, world, K, warm, t_dev, t_e2e, Ke, timed_pos, points, clk, t_q4, n_q4, q4_name, launches, lo):
    """The JSON line of the `ours` arm (rank 0)."""
    W, kv = model_bytes(MODEL)
    mean_p = sum(timed_pos) / K
    bytes_per_token = W + kv * (mean_p + 1) + kv
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    which = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    ach = W / t_q4 / 1e9
    traffic = None
    try:  # dram bytes of the kernel's launches of one token, from the committed ncu capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["bytes_per_token"]
    except (OSError, KeyError, ValueError):
        pass
    return {
        "metric": "LLaMA-7B gptq.int4 decode tokens/sec", "value": aggregate_throughput(world, K, t_dev), "unit": "tokens/s", "n_gpus": world,
        "steps": K, "warmup": warm, "ms_per_step": t_dev / K * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "LLaMA-7B gptq.int4 decode batch=1 ctx=2048 (random-init weights)", "prompt_tokens": PROMPT_T,
                   "positions": f"{K} positions spread evenly over {lo}..{S_CTX - 1} (mean {mean_p:.0f})",
                   "points": {**points, "unit": "tokens/s at fixed position"}, "sampling": f"top_k={TOP_K} temperature={TEMPERATURE}",
                   "parallelism": f"replicas x{world}" if world > 1 else "single GPU",
                   "l2": "weights 3.31 GB per token >> 126 MB L2 (inputs larger than L2)"},
        "clocks": clk,
        "e2e": {"value": aggregate_throughput(world, Ke, t_e2e), "unit": "tokens/s", "h2d_bytes_per_step": 12, "d2h_bytes_per_step": 8, "steps": Ke},
        "gpu_launches": (launches + 1) * K,  # b2l_decode_step's kernels + the fused sampling kernel, per token
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                     "kernel": q4_name, "launches_per_token": n_q4, "bytes_per_token_launches": W,
                     "peak_source": which,
                     "whole_token_bytes": bytes_per_token, "whole_token_achieved": bytes_per_token * K / t_dev / 1e9,
                     "whole_token_frac": bytes_per_token * K / t_dev / 1e9 / peak},
    }


def reduce_max(times, device):
    """Max over ranks of per-rank times (the N > 1 rule of the bench contract).  Replicas
    share nothing else: there is no data-path collective."""
    import torch
    import torch.distributed as dist

    t = torch.tensor(times, device=device, dtype=torch.float64)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def aggregate_throughput(world, steps, t_max):
    """Whole-job tokens/s of `world` replicas that each decoded `steps` tokens."""
    return world * steps / t_max


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tp", action="store_true", help="N > 1: skip the tensor-parallel block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's logits and token as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warm = max(3, args.warmup)
    K = args.steps
    torch.manual_seed(1234 + rank)   # sampling noise (and any other default-generator draw): same arguments, same run

    model = build_synthetic_model(MODEL, dev, seed=1234)   # every replica holds the same weights, decodes its own stream
    compacted = False
    if os.environ.get("B2L_COMPACT", "1") != "0":
        model.compact()     # one resident copy of the weights, as generate.py runs the model (lit_llama_b200/model.py)
        compacted = True
    gen = torch.Generator(device=dev).manual_seed(7 + rank)
    prompt = torch.randint(0, 32000, (PROMPT_T,), device=dev, dtype=torch.int32, generator=gen)
    feed = torch.randint(0, 32000, (warm + K, 1, 1), device=dev, dtype=torch.int32, generator=gen)   # decode inputs
    lo, span = PROMPT_T, S_CTX - PROMPT_T
    # the K timed positions are spread evenly over [16, 2047] whatever K is (slots in between stay zero rows: the
    # attention kernel reads them exactly like written ones); warm-up walks the first positions
    timed_pos = [lo + (i * span) // K for i in range(K)]
    pos_all = [torch.tensor([lo + (i % span)], device=dev) for i in range(warm)] + [torch.tensor([q], device=dev) for q in timed_pos]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        # ---- setup: prefill + graph capture (untimed)
        logits = model(prompt.view(1, -1), S_CTX, torch.arange(PROMPT_T, device=dev))
        tok = sample_next(logits).to(torch.int32)

        # ---- value: device-resident loop, no host sync inside
        for i in range(warm):
            tok = sample_next(model(feed[i], S_CTX, pos_all[i])).to(torch.int32)
        barrier()
        clocks = ClockSampler(local)
        clocks.start()
        time.sleep(0.25)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.time()
        e0.record()
        for i in range(warm, warm + K):
            logits = model(feed[i], S_CTX, pos_all[i])
            tok = sample_next(logits).to(torch.int32)
        e1.record()
        barrier()
        tw1 = time.time()
        t_dev = e0.elapsed_time(e1) * 1e-3
        clk = clocks.stop(tw0, tw1)
        if args.dump_outputs and rank == 0:   # nothing has run since the last timed step
            dump_outputs(args.dump_outputs, {"logits": logits.float().cpu().numpy(), "token": tok.float().cpu().numpy()})

        # ---- e2e: host buffers; per step H2D (token, position) from pinned memory, D2H sampled token
        h_tok = torch.empty(1, dtype=torch.int32).pin_memory()
        h_pos = torch.empty(1, dtype=torch.int64).pin_memory()
        h_out = torch.empty(1, dtype=torch.int64).pin_memory()
        d_tok = torch.empty(1, dtype=torch.int32, device=dev)
        d_pos = torch.empty(1, dtype=torch.int64, device=dev)
        h_tok[0] = int(tok)
        Ke = min(K, 512)
        for phase in ("warm", "timed"):
            n = 8 if phase == "warm" else Ke
            barrier()
            t0 = time.perf_counter()
            for i in range(n):
                h_pos[0] = lo + ((i * span) // n if phase == "timed" else i)
                d_tok.copy_(h_tok, non_blocking=True)
                d_pos.copy_(h_pos, non_blocking=True)
                nxt = sample_next(model(d_tok.view(1, 1), S_CTX, d_pos))
                h_out.copy_(nxt, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                h_tok[0] = int(h_out[0])
            barrier()
            t_e2e = time.perf_counter() - t0

        # ---- tokens/s at fixed positions (SURVEY 8d): 24 steps each at p = 128, 1024, 2047
        points = {}
        for q in (128, 1024, 2047):
            pq = torch.tensor([q], device=dev)
            for _ in range(4):
                tok = sample_next(model(tok.view(1, 1), S_CTX, pq)).to(torch.int32)
            torch.cuda.synchronize()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            for _ in range(24):
                tok = sample_next(model(tok.view(1, 1), S_CTX, pq)).to(torch.int32)
            p1.record()
            torch.cuda.synchronize()
            points[f"p{q}"] = round(24 / (p0.elapsed_time(p1) * 1e-3), 1)

        t_q4, n_q4, q4_name = time_q4_launches(model, dev)
        resident = {"allocated_gb": round(torch.cuda.memory_allocated(dev) / 1e9, 3), "compacted": compacted,
                    "what": "torch.cuda.memory_allocated after the timed loops: weights (one copy when compacted), embedding, KV cache S=2048, activations"}

    t_dev, t_e2e = reduce_max([t_dev, t_e2e], dev)

    from lit_llama_b200 import _lib as L
    import ctypes as C
    launches = L.lib().b2l_decode_step_launches(C.byref(model._decode.args))

    # ---- N > 1: the tensor-parallel path on the same ranks (SURVEY.md section 8e; `value` stays the replicas metric).
    # 7B split N ways, and LLaMA-65B gptq.int4 TP = 8 (BASELINE.json configs[4]) when N = 8.  A watchdog ends the run with
    # the headline line intact should a collective ever hang.
    tp = None
    if world > 1 and not args.no_tp:
        del model
        torch.cuda.empty_cache()
        box = {"line": None}

        def bail():
            if rank == 0 and box["line"] is not None:
                box["line"]["tp"] = {"error": "tensor-parallel block did not finish within its time limit"}
                print(json.dumps(box["line"]), flush=True)
            os._exit(0)

        watchdog = threading.Timer(float(os.environ.get("B2L_TP_BENCH_LIMIT_S", "420")), bail)
        watchdog.daemon = True
        if rank == 0:
            box["line"] = build_line(args, world, K, warm, t_dev, t_e2e, Ke, timed_pos, points, clk, t_q4, n_q4, q4_name, launches, lo)
        watchdog.start()
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import tp_bench

        tp = {}
        # the model that NEEDS the split first (BASELINE.json configs[4]); every model in its own try: shapes are the same
        # on every rank, so a failure is symmetric and the next model still runs
        for name, steps in ([("65B", 64)] if world == 8 else []) + [("7B", 96)]:
            try:
                tp[name] = tp_bench.run_tp(name, steps, 8, dev, rank, world)
            except Exception as e:  # noqa: BLE001 -- reported in the line, the replicas numbers stand
                tp[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
                torch.cuda.empty_cache()
        watchdog.cancel()

    if rank == 0:
        line = build_line(args, world, K, warm, t_dev, t_e2e, Ke, timed_pos, points, clk, t_q4, n_q4, q4_name, launches, lo)
        line["config"]["resident_memory"] = resident
        if tp is not None:
            line["tp"] = tp
        if not args.no_cpu_baseline and world == 1:
            model = None
            torch.cuda.empty_cache()
            cb = cpu_reference_tokens(n_tokens=1, budget_s=30.0, prompt_t=1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
    if world > 1:
        # No orderly teardown: with peer-mapped (symmetric-memory) buffers alive, destroy_process_group / interpreter
        # exit was measured to block on a 2-GPU box AFTER every rank had finished; the result line is out, nothing is
        # left to flush, and a failed collective may have left peers waiting anyway.
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
