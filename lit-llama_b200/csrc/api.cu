// Error state, device facts and the whole-token entry point of libb200llama.
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <utility>
#include <vector>

#include "b2l_common.cuh"

namespace b2l {

extern void* g_attn_timeline;

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  (void)cudaGetLastError();  // clear the sticky-less error so the next call starts clean
  return (int)e;
}

int sm_count() {
  static int n[B2L_MAX_DEVICES] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= B2L_MAX_DEVICES) return 148;
  if (n[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    n[dev] = v;
  }
  return n[dev];
}

}  // namespace b2l

using namespace b2l;

extern "C" int b2l_version(void) { return 100; }

extern "C" const char* b2l_last_error(void) { return g_err; }

extern "C" int b2l_device_info(int* sm, int* cc_major, int* cc_minor) {
  int dev = 0;
  B2L_CUDA(cudaGetDevice(&dev));
  int a = 0, b = 0, c = 0;
  B2L_CUDA(cudaDeviceGetAttribute(&a, cudaDevAttrMultiProcessorCount, dev));
  B2L_CUDA(cudaDeviceGetAttribute(&b, cudaDevAttrComputeCapabilityMajor, dev));
  B2L_CUDA(cudaDeviceGetAttribute(&c, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm) *sm = a;
  if (cc_major) *cc_major = b;
  if (cc_minor) *cc_minor = c;
  return 0;
}

// ---------------------------------------------------------------------------------
// LLaMA.forward for one new token per sequence (model.py:76-122 with T == 1):
//   wte -> n_layer x Block (model.py:156-168) -> ln_f -> lm_head
// Per Block: [rms_1 + c_attn] -> rope/append/attention -> [c_proj + residual]
//            -> [rms_2 + c_fc1|c_fc2 + silu*mul] -> [mlp.c_proj + residual]
// ---------------------------------------------------------------------------------
// ---- L2 prefetch windows of the batch-1 step (b2l_q4_linear_args::pf_ptr).
// The packed weights of a token are read in a fixed order: per Block c_attn, c_proj, fc1|fc2, mlp.c_proj, then lm_head,
// then the next token's Block 0 again.  Seen as one byte stream, launch j (bytes [S_j, E_j)) asks the L2 for
// [max(S_j + D, E_j), E_j + D): after every launch everything up to D bytes beyond its own end has been requested, so
// HBM always has a backlog to work on while a launch waits for its activations (prologue), reduces and stores
// (epilogue) or the attention kernel runs.  D = B2L_PF_MB (MB, read once; 0 switches the hint off).
struct PfWindow { const void* ptr[B2L_PF_SEGMENTS]; unsigned long long bytes[B2L_PF_SEGMENTS]; };

static size_t prefetch_distance() {
  static const long mb = [] { const char* e = getenv("B2L_PF_MB"); return e ? atol(e) : 0L; }();
  return mb > 0 ? (size_t)mb << 20 : 0;
}

static std::vector<PfWindow> prefetch_windows(const b2l_decode_args* d) {
  std::vector<std::pair<const uint8_t*, size_t>> ops;
  auto add = [&](const b2l_q4_weight& w) { ops.push_back({(const uint8_t*)w.qw_mma, b2l_q4_tiled_i8_bytes(w.N, w.K)}); };
  for (int l = 0; l < d->n_layer; ++l) {
    add(d->layers[l].c_attn); add(d->layers[l].c_proj); add(d->layers[l].c_fc12); add(d->layers[l].mlp_proj);
  }
  add(d->lm_head);
  const size_t n = ops.size(), D = prefetch_distance();
  std::vector<PfWindow> out(n, PfWindow{});
  if (D == 0) return out;
  std::vector<size_t> start(n + 1, 0);
  for (size_t j = 0; j < n; ++j) start[j + 1] = start[j] + ops[j].second;
  for (size_t j = 0; j < n; ++j) {
    size_t lo = std::max(start[j] + D, start[j + 1]), hi = start[j + 1] + D;   // may run past `total`: wraps to the next token
    int sg = 0;
    size_t k = j + 1;      // first op at or after `lo` (positions counted from this token's start; op k lives at k % n)
    size_t base = start[j + 1];
    while (lo < hi && sg < B2L_PF_SEGMENTS && k < j + 1 + n) {
      const auto& op = ops[k % n];
      const size_t op_lo = base, op_hi = base + op.second;
      if (lo < op_hi) {
        const size_t a = (lo - op_lo) & ~(size_t)127, b = std::min(hi, op_hi) - op_lo;
        if (b > a && op.first != nullptr) {
          out[j].ptr[sg] = op.first + a;
          out[j].bytes[sg] = (b - a + 15) & ~(size_t)15;
          ++sg;
        }
        lo = std::min(hi, op_hi);
      }
      base = op_hi;
      ++k;
    }
  }
  return out;
}

static int q4_call(const b2l_q4_weight& w, const void* x, int ldx, void* y, int ldy, int M, int sz_dtype, int prologue,
                   const void* norm_scale, float eps, int epilogue, const void* res, int ldres, int flags,
                   b2l_stream_t stream, void* trace = nullptr, void* batch_work = nullptr, const PfWindow* pf = nullptr,
                   const b2l_decode_args* kv_of = nullptr, int kv_layer = 0) {
  b2l_q4_linear_args a{};
  if (kv_of != nullptr) {   // this linear also asks the L2 for the KV-cache rows of layer `kv_layer`'s attention
    const int hs = kv_of->n_embd / kv_of->n_head;
    a.pf_kv[0] = kv_of->layers[kv_layer].k_cache; a.pf_kv[1] = kv_of->layers[kv_layer].v_cache;
    a.pf_rows = (const long long*)kv_of->input_pos;
    a.pf_rows_max = kv_of->S; a.pf_nseg = kv_of->B * kv_of->n_head; a.pf_row_bytes = hs * 2;
    a.pf_seg_stride = (unsigned long long)kv_of->S * hs * 2;
  }
  if (pf != nullptr)
    for (int i = 0; i < B2L_PF_SEGMENTS; ++i) { a.pf_ptr[i] = pf->ptr[i]; a.pf_bytes[i] = pf->bytes[i]; }
  a.x = x; a.ldx = ldx;
  const bool gemv = (M == 1 && w.qw_mma != nullptr);
  const bool batch = (!gemv && M <= 8 && w.qw_mma != nullptr && batch_work != nullptr);
  a.qw_tiled = (gemv || batch) ? w.qw_mma : w.qw_tiled; a.scales = w.scales; a.zeros = w.zeros; a.sz_dtype = sz_dtype;
  a.y = y; a.ldy = ldy;
  a.M = M; a.N = w.N; a.K = w.K;
  a.prologue = prologue; a.norm_scale = norm_scale; a.eps = eps;
  a.epilogue = epilogue; a.res = res; a.ldres = ldres;
  a.split_k = 0;
  a.flags = flags;
  a.trace = gemv ? trace : nullptr;
  if (gemv) return b2l_q4_gemv(&a, stream);
  if (batch) {
    a.workspace = batch_work;
    return b2l_q4_gemv_batch(&a, stream);
  }
  if (a.qw_tiled == nullptr) {
    set_error("b2l_decode_step: weight has no tiling for batch %d", M);
    return B2L_E_STATE;
  }
  return b2l_q4_linear_tc(&a, stream);
}

extern "C" int b2l_decode_step_launches(const b2l_decode_args* d) {
  if (!d) return 0;
  const int attn = (d->n_embd / d->n_head == 128) ? 1 : 3;  // fused single-token attention for head_size 128
  const int lin = (d->B > 1 && d->B <= 8 && d->batch_work) ? 2 : 1;  // the batch kernel is two launches per linear
  return 2 + d->n_layer * (4 * lin + attn) + lin;  // ring advance + embedding, per Block 4 linears + attention, ln_f+lm_head
}

extern "C" int b2l_decode_step(const b2l_decode_args* d, b2l_stream_t stream) {
  B2L_CHECK_ARG(d != nullptr && d->layers != nullptr, "b2l_decode_step: null args");
  B2L_CHECK_ARG(d->n_layer > 0 && d->n_head > 0 && d->n_embd % d->n_head == 0 && d->B >= 1 && d->S >= 1,
                "b2l_decode_step: bad model shape");
  B2L_CHECK_SUPPORTED(d->B <= 16, "b2l_decode_step: batch %d > 16", d->B);
  B2L_CHECK_ARG(d->wte && d->ln_f && d->rope && d->idx && d->input_pos && d->ring_start && d->x && d->qkv && d->att &&
                    d->hid && d->attn_work && d->logits,
                "b2l_decode_step: null pointer");
  const int C = d->n_embd, hs = C / d->n_head, B = d->B;
  const int fl = d->flags;
  int rc;
  // debug timeline: launch i of the step writes uint64[64] at timeline + 512*i (order: per Block c_attn,
  // attention, c_proj, fc12, mlp_proj; then lm_head)
  char* tlb = (char*)d->timeline;
  int li = 0;
  auto tl = [&]() -> void* { void* r = tlb ? (void*)(tlb + 512 * li) : nullptr; ++li; return r; };
  // batch 1 on the int8-MMA kernel: every linear carries the L2 prefetch window of the weights that follow it
  std::vector<PfWindow> pfw;
  if (B == 1 && d->lm_head.qw_mma != nullptr) pfw = prefetch_windows(d);
  // B2L_KV_PREFETCH (read once): 0 off, 1 the previous Block's mlp.c_proj asks for a Block's KV rows, 2 its own c_attn does
  static const int kv_prefetch = [] { const char* e = getenv("B2L_KV_PREFETCH"); return e ? atoi(e) : 0; }();
  const bool kv_ok = B == 1 && hs == 128 && d->lm_head.qw_mma != nullptr;
  int oi = 0;
  auto pf = [&]() -> const PfWindow* { const PfWindow* r = pfw.empty() ? nullptr : &pfw[oi]; ++oi; return r; };
  if ((rc = b2l_ring_advance(d->input_pos, 1, d->ring_start, d->S, stream))) return rc;
  if ((rc = b2l_embedding(d->idx, d->idx_is_i64, d->wte, d->x, B, C, d->vocab, stream))) return rc;
  for (int l = 0; l < d->n_layer; ++l) {
    const b2l_layer& L = d->layers[l];
    if ((rc = q4_call(L.c_attn, d->x, C, d->qkv, 3 * C, B, d->sz_dtype, B2L_PRO_RMSNORM, L.rms_1, d->eps, B2L_EPI_STORE,
                      nullptr, 0, fl, stream, tl(), d->batch_work, pf(), (kv_ok && kv_prefetch == 2) ? d : nullptr, l)))
      return rc;
    g_attn_timeline = tl();
    if ((rc = b2l_attention(d->qkv, L.k_cache, L.v_cache, d->rope, d->input_pos, d->ring_start, d->att, d->attn_work, B,
                            1, d->n_head, hs, d->S, d->block_size, fl, stream))) {
      g_attn_timeline = nullptr;
      return rc;
    }
    g_attn_timeline = nullptr;
    if ((rc = q4_call(L.c_proj, d->att, C, d->x, C, B, d->sz_dtype, B2L_PRO_NONE, nullptr, 0.f, B2L_EPI_RESIDUAL, d->x, C,
                      fl, stream, tl(), d->batch_work, pf())))
      return rc;
    if ((rc = q4_call(L.c_fc12, d->x, C, d->hid, d->n_hidden, B, d->sz_dtype, B2L_PRO_RMSNORM, L.rms_2, d->eps,
                      B2L_EPI_SWIGLU, nullptr, 0, fl, stream, tl(), d->batch_work, pf())))
      return rc;
    // mlp.c_proj fits the weight ring entirely, so HBM idles while it converts its activations: it asks the L2 for
    // the NEXT Block's KV-cache rows (B2L_KV_PREFETCH=0 switches that off)
    const bool kvpf = kv_prefetch == 1 && kv_ok && l + 1 < d->n_layer;
    if ((rc = q4_call(L.mlp_proj, d->hid, d->n_hidden, d->x, C, B, d->sz_dtype, B2L_PRO_NONE, nullptr, 0.f,
                      B2L_EPI_RESIDUAL, d->x, C, fl, stream, tl(), d->batch_work, pf(), kvpf ? d : nullptr, l + 1)))
      return rc;
  }
  return q4_call(d->lm_head, d->x, C, d->logits, d->vocab, B, d->sz_dtype, B2L_PRO_RMSNORM, d->ln_f, d->eps,
                 B2L_EPI_STORE, nullptr, 0, fl, stream, tl(), d->batch_work, pf());
}
