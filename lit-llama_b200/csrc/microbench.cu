// Debug-only microbenchmarks (tools/diag.py): tcgen05 issue/completion costs, legacy tensor-pipe issue rates,
// grid-wide flag latency.  Built into libb200diag.so (include/b2l_diag.h), NOT into the product library.
#include "b2l_common.cuh"
#include "../../include/b2l_diag.h"

namespace b2l {
// the diagnostic library carries its own copy of the error state (the product's lives in api.cu)
static thread_local char g_diag_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_diag_err, sizeof(g_diag_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  (void)cudaGetLastError();
  return (int)e;
}
int sm_count() {
  int dev = 0, v = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
  return v;
}
}  // namespace b2l

extern "C" const char* b2l_diag_last_error(void) { return b2l::g_diag_err; }

namespace b2l {
namespace q4tc {
// PTX wrappers shared with q4_tc.cu (kept in sync by inclusion order: this file re-declares the few it needs)
__device__ __forceinline__ uint32_t mb_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
}  // namespace q4tc

__global__ void __launch_bounds__(128) mma_rate_kernel(unsigned long long* out, int n_mma, int n_acc, int a_from_smem, int rounds) {
  __shared__ __align__(128) uint8_t bsm[16 * 1024];
  __shared__ __align__(8) unsigned long long bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar_a = q4tc::mb_smem_u32(&bar);
  for (int i = tid; i < 16 * 1024 / 4; i += 128) reinterpret_cast<uint32_t*>(bsm)[i] = 0x3f803f80u;  // bf16 1.0
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(q4tc::mb_smem_u32(&tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_slot;
  // A operand in TMEM: 128 lanes x 8 columns of bf16 pairs (1.0, 1.0)
  {
    uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
    uint32_t v = 0x3f803f80u;
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(v) : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (tid == 0) {
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((16u >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t sb = q4tc::mb_smem_u32(bsm);
    // B: K-major no-swizzle, LBO = 256 (next 8-k column), SBO = 128 (next 8 rows of N)
    uint64_t bdesc = (uint64_t)((sb & 0x3FFFFu) >> 4) | ((uint64_t)(256 >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
    // A from smem (SS): 128 rows K-major: LBO = 2048 (next 8-k column), SBO = 128 (next 8 rows)
    uint64_t adesc = (uint64_t)((sb & 0x3FFFFu) >> 4) | ((uint64_t)(2048 >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
    uint32_t parity = 0;
    for (int r = 0; r < rounds; ++r) {
      long long t0 = clock64();
      // fully unrolled, compile-time addresses: n_mma in {1,4,16}, n_acc in {1,4}
#define B2L_MMA(I, NACC)                                                                                                     \
  do {                                                                                                                       \
    const uint32_t d_ = tmem + 64 + (uint32_t)(((I) % (NACC)) * 16);                                                          \
    if (a_from_smem)                                                                                                         \
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_), \
                   "l"(adesc), "l"(bdesc), "r"(idesc), "r"((I) >= (NACC) ? 1u : 0u) : "memory");                               \
    else                                                                                                                     \
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_), \
                   "r"(tmem), "l"(bdesc), "r"(idesc), "r"((I) >= (NACC) ? 1u : 0u) : "memory");                                \
  } while (0)
#define B2L_MMA4(I, NACC) B2L_MMA(I, NACC); B2L_MMA(I + 1, NACC); B2L_MMA(I + 2, NACC); B2L_MMA(I + 3, NACC)
      if (n_acc == 1) {
        if (n_mma >= 1) B2L_MMA(0, 1);
        if (n_mma >= 4) { B2L_MMA(1, 1); B2L_MMA(2, 1); B2L_MMA(3, 1); }
        if (n_mma >= 16) { B2L_MMA4(4, 1); B2L_MMA4(8, 1); B2L_MMA4(12, 1); }
      } else {
        if (n_mma >= 1) B2L_MMA(0, 4);
        if (n_mma >= 4) { B2L_MMA(1, 4); B2L_MMA(2, 4); B2L_MMA(3, 4); }
        if (n_mma >= 16) { B2L_MMA4(4, 4); B2L_MMA4(8, 4); B2L_MMA4(12, 4); }
      }
      long long t1 = clock64();
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_a) : "memory");
      long long t2 = clock64();
      uint32_t ok;
      do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar_a), "r"(parity) : "memory");
      } while (!ok);
      long long t3 = clock64();
      parity ^= 1;
      out[r * 3 + 0] = (unsigned long long)(t1 - t0);
      out[r * 3 + 1] = (unsigned long long)(t2 - t1);
      out[r * 3 + 2] = (unsigned long long)(t3 - t0);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}


// ---- can several threads of one CTA keep the tensor pipe fed better than one?  `n_issuers` warps (1..4) each
// elect lane 0 to issue 16 back-to-back 128x16x16 tcgen05.mma (A in TMEM, shared; own 16-column accumulator) and
// one commit on their own mbarrier.  out[r * 8 + w] = cycles from the common start until warp w's commit arrived,
// out[r * 8 + 4 + w] = cycles warp w spent issuing.  If the per-warp time does not grow with n_issuers, MMA issue
// is a per-thread limit and a multi-issuer kernel scales; if it grows linearly it is a per-SM limit.
__global__ void __launch_bounds__(128) mma_multi_issuer_kernel(unsigned long long* out, int n_issuers, int rounds) {
  __shared__ __align__(128) uint8_t bsm[16 * 1024];
  __shared__ __align__(8) unsigned long long bars[4];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < 16 * 1024 / 4; i += 128) reinterpret_cast<uint32_t*>(bsm)[i] = 0x3f803f80u;  // bf16 1.0
  if (tid == 0) {
    for (int i = 0; i < 4; ++i)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(q4tc::mb_smem_u32(&bars[i])) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(q4tc::mb_smem_u32(&tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_slot;
  {
    uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
    uint32_t v = 0x3f803f80u;
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(v) : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((16u >> 3) << 17) | ((128u >> 4) << 24);
  const uint32_t sb = q4tc::mb_smem_u32(bsm);
  const uint64_t bdesc = (uint64_t)((sb & 0x3FFFFu) >> 4) | ((uint64_t)(256 >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
  const uint32_t bar_a = q4tc::mb_smem_u32(&bars[warp]);
  const uint32_t d = tmem + 64 + (uint32_t)(warp * 16);
  uint32_t parity = 0;
  for (int r = 0; r < rounds; ++r) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (warp < n_issuers && lane == 0) {
      const long long t0 = clock64();
#pragma unroll
      for (int i = 0; i < 16; ++i)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d),
                     "r"(tmem), "l"(bdesc), "r"(idesc), "r"(i > 0 ? 1u : 0u) : "memory");
      const long long t1 = clock64();
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_a) : "memory");
      uint32_t ok;
      do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar_a), "r"(parity) : "memory");
      } while (!ok);
      const long long t2 = clock64();
      out[r * 8 + warp] = (unsigned long long)(t2 - t0);
      out[r * 8 + 4 + warp] = (unsigned long long)(t1 - t0);
    }
    parity ^= 1;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}

}  // namespace b2l

// out: uint64[rounds * 3] = {issue cycles of n_mma MMAs, commit issue cycles, total cycles until the commit arrives}
// ---- legacy tensor pipe: how often can one SM sub-partition issue mma.sync.m16n8k16 (HMMA.16816.F32)?
// One CTA, `warps` warps, each with CH independent accumulator chains; optionally the 5 ALU ops per MMA
// of the int4 unpack (1 shift + 4 LOP3 per word) in front of every MMA.
template <int CH>
__global__ void __launch_bounds__(1024) hmma_rate_kernel(unsigned long long* out, int iters, int with_unpack, uint32_t seed) {
  float acc[CH][4];
#pragma unroll
  for (int c = 0; c < CH; ++c)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[c][i] = 0.f;
  uint32_t w = seed + threadIdx.x;
  uint32_t a0 = 0x3c003c00u, a1 = 0x3c003c00u, a2 = 0x3c003c00u, a3 = 0x3c003c00u;
  const uint32_t b0 = 0x3c003c00u, b1 = 0x3c003c00u;
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (with_unpack) {
        const uint32_t w8 = w >> 8;
        asm volatile("lop3.b32 %0, %1, 0x000f000f, 0x64006400, 0xEA;" : "=r"(a0) : "r"(w));
        asm volatile("lop3.b32 %0, %1, 0x000f000f, 0x64006400, 0xEA;" : "=r"(a1) : "r"(w8));
        asm volatile("lop3.b32 %0, %1, 0x00f000f0, 0x64006400, 0xEA;" : "=r"(a2) : "r"(w));
        asm volatile("lop3.b32 %0, %1, 0x00f000f0, 0x64006400, 0xEA;" : "=r"(a3) : "r"(w8));
        w += 0x01010101u;
      }
      asm volatile(
          "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
          : "+f"(acc[j % CH][0]), "+f"(acc[j % CH][1]), "+f"(acc[j % CH][2]), "+f"(acc[j % CH][3])
          : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    }
  }
  const long long t1 = clock64();
  __syncthreads();
  float sink = 0.f;
#pragma unroll
  for (int c = 0; c < CH; ++c) sink += acc[c][0] + acc[c][1] + acc[c][2] + acc[c][3];
  if (threadIdx.x == 0) { out[0] = (unsigned long long)(t1 - t0); out[1] = (unsigned long long)__float_as_uint(sink); }
}

extern "C" int b2l_debug_hmma_rate(void* out, int warps, int chains, int iters, int with_unpack, b2l_stream_t stream) {
  B2L_CHECK_ARG(out && warps > 0 && warps <= 32 && iters > 0 && (chains == 1 || chains == 2 || chains == 4 || chains == 8),
                "b2l_debug_hmma_rate: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* o = (unsigned long long*)out;
  if (chains == 1) hmma_rate_kernel<1><<<1, warps * 32, 0, st>>>(o, iters, with_unpack, 0x12345678u);
  else if (chains == 2) hmma_rate_kernel<2><<<1, warps * 32, 0, st>>>(o, iters, with_unpack, 0x12345678u);
  else if (chains == 4) hmma_rate_kernel<4><<<1, warps * 32, 0, st>>>(o, iters, with_unpack, 0x12345678u);
  else hmma_rate_kernel<8><<<1, warps * 32, 0, st>>>(o, iters, with_unpack, 0x12345678u);
  B2L_LAUNCH_CHECK("hmma_rate_kernel");
  return 0;
}

// ---- legacy integer tensor pipe: how often can one SM sub-partition issue mma.sync.m16n8k32 u8 x s8 (IMMA.16832.U8.S8)?
// Round-2 question: an int8 contraction consumes 512 weight nibbles per MMA (two packed words per lane) with at most
// two LOP3 in front of it, against 256 nibbles and five ALU ops for the fp16 form.  n_alu = ALU ops issued per MMA.
template <int CH>
__global__ void __launch_bounds__(1024) imma_rate_kernel(unsigned long long* out, int iters, int n_alu, uint32_t seed) {
  int acc[CH][4];
#pragma unroll
  for (int c = 0; c < CH; ++c)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[c][i] = 0;
  uint32_t w0 = seed + threadIdx.x, w1 = seed * 3 + threadIdx.x;
  uint32_t a1 = w0 & 0xf0f0f0f0u, a3 = w1 & 0xf0f0f0f0u;
  const uint32_t b0 = 0x01020304u, b1 = 0x7f80fe02u;
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (n_alu >= 2) {
        asm volatile("lop3.b32 %0, %1, 0xf0f0f0f0, 0, 0xC0;" : "=r"(a1) : "r"(w0));
        asm volatile("lop3.b32 %0, %1, 0xf0f0f0f0, 0, 0xC0;" : "=r"(a3) : "r"(w1));
      }
      if (n_alu >= 4) {
        asm volatile("add.u32 %0, %0, 0x01010101;" : "+r"(w0));
        asm volatile("add.u32 %0, %0, 0x03010101;" : "+r"(w1));
      }
      asm volatile(
          "mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
          : "+r"(acc[j % CH][0]), "+r"(acc[j % CH][1]), "+r"(acc[j % CH][2]), "+r"(acc[j % CH][3])
          : "r"(w0), "r"(a1), "r"(w1), "r"(a3), "r"(b0), "r"(b1));
    }
  }
  const long long t1 = clock64();
  __syncthreads();
  int sink = 0;
#pragma unroll
  for (int c = 0; c < CH; ++c) sink += acc[c][0] + acc[c][1] + acc[c][2] + acc[c][3];
  if (threadIdx.x == 0) { out[0] = (unsigned long long)(t1 - t0); out[1] = (unsigned long long)(uint32_t)sink; }
}

extern "C" int b2l_debug_imma_rate(void* out, int warps, int chains, int iters, int n_alu, b2l_stream_t stream) {
  B2L_CHECK_ARG(out && warps > 0 && warps <= 32 && iters > 0 && (chains == 1 || chains == 2 || chains == 4 || chains == 8),
                "b2l_debug_imma_rate: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* o = (unsigned long long*)out;
  if (chains == 1) imma_rate_kernel<1><<<1, warps * 32, 0, st>>>(o, iters, n_alu, 0x12345678u);
  else if (chains == 2) imma_rate_kernel<2><<<1, warps * 32, 0, st>>>(o, iters, n_alu, 0x12345678u);
  else if (chains == 4) imma_rate_kernel<4><<<1, warps * 32, 0, st>>>(o, iters, n_alu, 0x12345678u);
  else imma_rate_kernel<8><<<1, warps * 32, 0, st>>>(o, iters, n_alu, 0x12345678u);
  B2L_LAUNCH_CHECK("imma_rate_kernel");
  return 0;
}

// ---- the decode kernels' consumer loop in isolation: `warps` warps sweep 16 KB stages that already sit in shared
// memory (no TMA, no barriers): per stage a warp loads its two 512-byte tiles (LDS.128 each), its activation-digit
// fragments (LDS.128, lanes 16..31 read a zero block or are predicated off) and issues 4 IMMA.16832.U8.S8.
// mode bits: 1 = weight loads, 2 = digit loads, 4 = IMMAs, 8 = predicate the digit load of lanes 16..31 off,
// 16 = 8 warps x 4 tiles instead of 16 x 2.  out[0] = cycles for `iters` sweeps over 8 stages.
__global__ void __launch_bounds__(512) consumer_rate_kernel(unsigned long long* out, int iters, int mode) {
  extern __shared__ __align__(128) uint8_t csm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  constexpr int NST = 8, STAGE = 16384, PS = 4096 + 64;
  uint8_t* ring = csm;
  uint8_t* xf = csm + NST * STAGE;
  uint8_t* zero = xf + 4 * PS;
  for (int i = tid; i < (NST * STAGE + 4 * PS + 16) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(csm)[i] = 0x01030507u * (i + 1);
  if (tid < 4) reinterpret_cast<uint32_t*>(zero)[tid] = 0u;
  __syncthreads();
  const int ncol = lane >> 2, t4 = lane & 3;
  const bool pred_off = (mode & 8) != 0;
  const uint8_t* xf_lane = (ncol < 4) ? xf + ncol * PS + t4 * 16 : zero;
  const int xf_step = (ncol < 4) ? 64 : 0;
  const int tiles = 32 / nw;   // tiles per warp per stage
  int acc[4][4];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[c][i] = 0;
  uint4 wv = make_uint4(lane, lane * 3, lane * 5, lane * 7), xb = make_uint4(1, 2, 3, 4);
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
#pragma unroll 1
    for (int st = 0; st < NST; ++st) {
      const uint8_t* base = ring + st * STAGE + lane * 16;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (i < tiles) {
          const int tile = i * nw + warp;
          if (mode & 1) wv = *reinterpret_cast<const uint4*>(base + tile * 512);
          if (mode & 2) {
            if (!pred_off || ncol < 4) xb = *reinterpret_cast<const uint4*>(xf_lane + ((st * 16 + tile) & 63) * xf_step);
            else xb = make_uint4(0, 0, 0, 0);
          }
          if (mode & 4) {
            asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                         : "+r"(acc[i][0]), "+r"(acc[i][1]), "+r"(acc[i][2]), "+r"(acc[i][3])
                         : "r"(wv.x), "r"(wv.x & 0xf0f0f0f0u), "r"(wv.y), "r"(wv.y & 0xf0f0f0f0u), "r"(xb.x), "r"(xb.y));
            asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                         : "+r"(acc[(i + 2) & 3][0]), "+r"(acc[(i + 2) & 3][1]), "+r"(acc[(i + 2) & 3][2]), "+r"(acc[(i + 2) & 3][3])
                         : "r"(wv.z), "r"(wv.z & 0xf0f0f0f0u), "r"(wv.w), "r"(wv.w & 0xf0f0f0f0u), "r"(xb.z), "r"(xb.w));
          } else {
            acc[i][0] += (int)(wv.x ^ wv.y ^ wv.z ^ wv.w ^ xb.x ^ xb.y ^ xb.z ^ xb.w);
          }
        }
      }
    }
  }
  const long long t1 = clock64();
  __syncthreads();
  int sink = 0;
#pragma unroll
  for (int c = 0; c < 4; ++c) sink += acc[c][0] + acc[c][1] + acc[c][2] + acc[c][3];
  if (tid == 0) { out[0] = (unsigned long long)(t1 - t0); out[1] = (unsigned long long)(uint32_t)sink; }
}

extern "C" int b2l_debug_consumer_rate(void* out, int warps, int iters, int mode, int n_ctas, b2l_stream_t stream) {
  B2L_CHECK_ARG(out && (warps == 8 || warps == 16) && iters > 0 && n_ctas > 0, "b2l_debug_consumer_rate: bad argument");
  const int smem = 8 * 16384 + 4 * (4096 + 64) + 16;
  B2L_CUDA(cudaFuncSetAttribute(consumer_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  consumer_rate_kernel<<<n_ctas, warps * 32, smem, (cudaStream_t)stream>>>((unsigned long long*)out, iters, mode);
  B2L_LAUNCH_CHECK("consumer_rate_kernel");
  return 0;
}

// ---- what does a grid-wide dependency cost without a kernel boundary?  Every CTA (all co-resident) arrives on a
// global counter with red.release and polls it with ld.acquire until all have arrived; out[r] = max over CTAs of
// the nanoseconds between its arrival and its release, out[rounds + r] = min.  A kernel that fuses several ops
// pays one of these for every kernel boundary it removes (DESIGN.md section 3 compares the two costs).
__global__ void __launch_bounds__(128) grid_flag_kernel(unsigned long long* out, unsigned int* counter, int rounds) {
  if (threadIdx.x != 0) return;
  for (int r = 0; r < rounds; ++r) {
    const unsigned int target = (unsigned int)(r + 1) * gridDim.x;
    const unsigned long long t0 = b2l::globaltimer_ns();
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
    } while (seen < target);
    const unsigned long long dt = b2l::globaltimer_ns() - t0;
    atomicMax(out + r, dt);
    atomicMin(out + rounds + r, dt);
  }
}

extern "C" int b2l_debug_grid_flag(void* out, void* counter, int ctas_per_sm, int rounds, b2l_stream_t stream) {
  B2L_CHECK_ARG(out && counter && ctas_per_sm >= 1 && ctas_per_sm <= 4 && rounds > 0 && rounds <= 64, "b2l_debug_grid_flag: bad argument");
  // the caller zero-fills `counter` (uint32) and out[0 .. rounds) and fills out[rounds .. 2 rounds) with ~0
  grid_flag_kernel<<<ctas_per_sm * b2l::sm_count(), 128, 0, (cudaStream_t)stream>>>((unsigned long long*)out, (unsigned int*)counter, rounds);
  B2L_LAUNCH_CHECK("grid_flag_kernel");
  return 0;
}

extern "C" int b2l_debug_mma_issuers(void* out, int n_issuers, int rounds, b2l_stream_t stream) {
  B2L_CHECK_ARG(out && n_issuers >= 1 && n_issuers <= 4 && rounds > 0, "b2l_debug_mma_issuers: bad argument");
  b2l::mma_multi_issuer_kernel<<<1, 128, 0, (cudaStream_t)stream>>>((unsigned long long*)out, n_issuers, rounds);
  B2L_LAUNCH_CHECK("mma_multi_issuer_kernel");
  return 0;
}

extern "C" int b2l_debug_mma_rate(void* out, int n_mma, int n_acc, int a_from_smem, int rounds, b2l_stream_t stream) {
  B2L_CHECK_ARG(out && n_mma > 0 && n_acc > 0 && n_acc <= 8 && rounds > 0, "b2l_debug_mma_rate: bad argument");
  b2l::mma_rate_kernel<<<1, 128, 0, (cudaStream_t)stream>>>((unsigned long long*)out, n_mma, n_acc, a_from_smem, rounds);
  B2L_LAUNCH_CHECK("mma_rate_kernel");
  return 0;
}
