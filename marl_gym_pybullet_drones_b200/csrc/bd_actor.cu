// Fused actor forward on 5th-gen tensor cores (tcgen05 + TMEM), sm_100a.
//
// Replaces the batched branch of `MAPPOActorCritic.step` (reference
// gym_pybullet_drones/mappo/agent.py:389-415): for every drone row
//     mean = W3 tanh(W2 tanh(W1 obs + b1) + b2) + b3        (MLP, neural_networks.py:18-53)
//     act  = mean + exp(logstd) * eps,  eps ~ N(0, I)        (dist.sample, agent.py:399-400)
//     logp = sum_k [-eps_k^2/2 - logstd_k - log(2 pi)/2]     (Normal.log_prob summed, distributions.py:12-21)
// in ONE kernel: observations are read once (fp32 -> bf16 in registers), the three GEMMs run
// as tcgen05.mma (bf16 x bf16 -> fp32 in TMEM, M = 128 rows per CTA, N = hidden, K = 16 per
// instruction, issued by one thread), activations never leave the SM: TMEM -> registers
// (tcgen05.ld) -> +bias, tanh.approx -> bf16 -> shared memory in the canonical K-major UMMA
// layout -> next layer's A operand.
//
// Shared memory (hidden = 256, obs_dim = 72 -> K1 = 80): region A 64 KB holds {X tile 20 KB,
// W1 40 KB} during layer 1 and the 128 x 256 bf16 activation tile afterwards; W2 (128 KB) and W3
// (8 KB, N padded to 16) stay resident for the CTA's lifetime (persistent grid, one CTA per SM);
// W1 is re-read from L2 per tile (40 KB).  TMEM: 256 columns (128 lanes x 256 fp32) reused by the
// three layers.  Operand layout: 8 x 8 bf16 core matrices (128 B), LBO = 128 B between the two
// K-halves of an instruction, SBO = (K/8) * 128 B between 8-row groups, no swizzle.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <new>

#include "../../include/batch_drones.h"

namespace {

constexpr int kRows = 128;   // UMMA M
constexpr int kNOut = 16;    // layer-3 N (act_dim padded; UMMA needs N % 16 == 0 at M = 128)

thread_local char g_actor_err[256] = "";
int afail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_actor_err, sizeof(g_actor_err), fmt, ap);
  va_end(ap);
  return code;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor, K-major, no swizzle (cute/arch/mma_sm100_desc.hpp SmemDescriptor)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version 1 (Blackwell)
  return d;
}

// instruction descriptor: D fp32, A/B bf16, both K-major, M = 128 (InstrDescriptor bit layout)
__host__ __device__ constexpr uint32_t umma_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kRows >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc),
      "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t v[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

// element (r, k) of a [rows x K] K-major operand tile, in bf16 elements
__host__ __device__ __forceinline__ size_t canon_off(int r, int k, int K) {
  return (size_t)(r >> 3) * (K >> 3) * 64 + (size_t)(k >> 3) * 64 + (size_t)(r & 7) * 8 + (k & 7);
}

struct ActorDev {
  const __nv_bfloat16 *w1, *w2, *w3;   // canonical layouts: [HID x K1], [HID x HID], [16 x HID]
  const float *b1, *b2, *b3, *logstd;  // b3 / logstd padded to 16
  int obs_dim, K1, act_dim;
  const float *nmean, *nrstd;   // optional input normalisation (bd_actor_set_input_norm), period rows
  int nperiod;
  float nclip;
  long long* trace;   // optional: [tiles of CTA 0][16] SM-clock stamps of the pipeline phases (bd_actor_set_trace)
};

__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t v[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

constexpr int CW = 16;   // columns per TMEM load / published chunk of a hidden epilogue

template <int HID>
__device__ __forceinline__ void hidden_chunk(const uint32_t* v, int c0, const float* __restrict__ bias, __nv_bfloat16* sH, int row) {
#pragma unroll
  for (int q = 0; q < CW / 8; ++q) {
    float h[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) h[j] = tanh_fast(__uint_as_float(v[q * 8 + j]) + bias[c0 + q * 8 + j]);
    uint4 pk;
    pk.x = pack_bf16(h[0], h[1]); pk.y = pack_bf16(h[2], h[3]); pk.z = pack_bf16(h[4], h[5]); pk.w = pack_bf16(h[6], h[7]);
    *reinterpret_cast<uint4*>(sH + canon_off(row, c0 + q * 8, HID)) = pk;
  }
}

// mbarrier helpers.  A wait that does not complete within ~2 s of SM clocks traps (a protocol bug
// must fail the launch, not hang the GPU).
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_guarded(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    // try_wait suspends the thread in hardware for up to the hinted time: no issue slots are
    // taken from the other warps of the SM sub-partition while waiting
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
    if (done) break;
    if ((it & 255u) == 255u) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) __trap();
    }
  }
}

// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t sdst, const void* gsrc, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sdst), "l"(gsrc),
               "r"(bytes), "r"(bar)
               : "memory");
}

// TMEM accumulator row -> +bias, tanh -> bf16 activation tile (next layer's A operand), 16 columns
// at a time.  After each chunk the thread publishes it (generic -> async proxy fence, mbarrier
// arrive): the MMA warp starts the next layer's K-steps over those columns while the remaining
// chunks are still going through the SFU, so tensor pipe and epilogue overlap inside one tile.
// The TMEM read of the next 16 columns is in flight while the current 16 are processed.
template <int HID>
__device__ __forceinline__ void epilogue_hidden(uint32_t tmem_row, const float* __restrict__ bias, __nv_bfloat16* sH, int row,
                                                int cbeg, int n_chunks, uint32_t chunk_bar0) {
  uint32_t va[CW], vb[CW];
  tmem_ld16_nowait(tmem_row + (uint32_t)cbeg, va);
  tmem_wait_ld();
#pragma unroll 1
  for (int j = 0; j < n_chunks; j += 2) {
    const int c0 = cbeg + j * CW;
    const bool more1 = j + 1 < n_chunks;
    if (more1) tmem_ld16_nowait(tmem_row + (uint32_t)(c0 + CW), vb);
    hidden_chunk<HID>(va, c0, bias, sH, row);
    proxy_fence();
    mbar_arrive(chunk_bar0 + 8u * (uint32_t)j);
    tmem_wait_ld();
    if (!more1) break;
    const bool more2 = j + 2 < n_chunks;
    if (more2) tmem_ld16_nowait(tmem_row + (uint32_t)(c0 + 2 * CW), va);
    hidden_chunk<HID>(vb, c0 + CW, bias, sH, row);
    proxy_fence();
    mbar_arrive(chunk_bar0 + 8u * (uint32_t)(j + 1));
    tmem_wait_ld();
  }
}

constexpr int kMaxChunks = 4;                 // column chunks per thread and layer
// barrier indices (one phase per tile each)
enum { BAR_STAGE = 0, BAR_L1, BAR_L2, BAR_L3, BAR_W1, BAR_W23, BAR_H1, BAR_H2 = BAR_H1 + kMaxChunks,
       BAR_COUNT = BAR_H2 + kMaxChunks };

// G = 4 threads per row (column groups): warps 0..4G-1 stage and run the epilogues (warp w owns TMEM
// lanes 32*(w%4).. and column group w/4), warp 4G issues every tcgen05.mma and TMA copy.
// 16 epilogue warps (4 per SM sub-partition) hide the TMEM-load / MUFU latencies of the tanh
// epilogue twice as well as G = 2 did; the register file then allows 96 registers per thread.
struct ActorShape {
  static constexpr int G = 4;
  static constexpr int kEpiThreads = kRows * G;
  static constexpr int kThreads = kEpiThreads + 32;
};

template <int HID>
__global__ void __launch_bounds__(ActorShape::kThreads, 1)
actor_forward_kernel(ActorDev W, const float* __restrict__ obs, long long rows, const float* __restrict__ noise,
                     unsigned long long seed, unsigned long long offset, float* __restrict__ act, float* __restrict__ logp,
                     float* __restrict__ mean_out) {
  constexpr int G = ActorShape::G, kEpiThreads = ActorShape::kEpiThreads, kThreads = ActorShape::kThreads;
  extern __shared__ __align__(128) unsigned char smem[];
  const int K1 = W.K1;
  const size_t actb = (size_t)kRows * HID * 2, l1b = (size_t)(kRows + HID) * K1 * 2;
  const size_t regA = ((actb > l1b ? actb : l1b) + 127) & ~(size_t)127;   // same formula on the host
  __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem);               // X tile, later activations
  __nv_bfloat16* sW1 = sA + (size_t)kRows * K1;                             // inside region A
  __nv_bfloat16* sW2 = reinterpret_cast<__nv_bfloat16*>(smem + regA);
  __nv_bfloat16* sW3 = sW2 + (size_t)HID * HID;
  float* sB1 = reinterpret_cast<float*>(sW3 + (size_t)kNOut * HID);
  float* sB2 = sB1 + HID;
  float* sB3 = sB2 + HID;        // [16]
  float* sLs = sB3 + kNOut;      // [16]
  __shared__ __align__(8) uint64_t mbar[BAR_COUNT];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5;
  const bool is_mma_warp = warp == kEpiThreads / 32;
  const int row = tid & (kRows - 1);      // my row of the tile = my TMEM lane
  const int grp = (tid >> 7) & (G - 1);   // which group of columns I handle in the epilogues
  constexpr int kGrpCols = HID / G;       // columns per thread and layer
  constexpr int kChunks = kGrpCols / CW;
  static_assert(kChunks >= 1 && kChunks <= kMaxChunks, "unsupported HID / G");
  constexpr uint32_t kTmemCols = HID == 256 ? 512u : (HID == 128 ? 256u : 128u);   // two accumulators
  const int cbeg = grp * kGrpCols;
  // ---- one-time: resident weights, barriers, tensor memory ------------------------------------
  // (W2 / W3 / W1 arrive by TMA bulk copies issued by the MMA thread)
  for (int i = tid; i < HID; i += kThreads) { sB1[i] = W.b1[i]; sB2[i] = W.b2[i]; }
  if (tid < kNOut) { sB3[tid] = W.b3[tid]; sLs[tid] = W.logstd[tid]; }
  if (tid == 0) {
    mbar_init(smem_u32(&mbar[BAR_STAGE]), kEpiThreads);
    mbar_init(smem_u32(&mbar[BAR_L1]), 1);
    mbar_init(smem_u32(&mbar[BAR_L2]), 1);
    mbar_init(smem_u32(&mbar[BAR_L3]), 1);
    mbar_init(smem_u32(&mbar[BAR_W1]), 1);
    mbar_init(smem_u32(&mbar[BAR_W23]), 1);
    for (int j = 0; j < kMaxChunks; ++j) {
      mbar_init(smem_u32(&mbar[BAR_H1 + j]), kEpiThreads);
      mbar_init(smem_u32(&mbar[BAR_H2 + j]), kEpiThreads);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  const uint32_t acc0 = tmem_base, acc1 = tmem_base + (uint32_t)HID;            // L1 / L3 and L2 accumulators
  const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;                  // my warp's 32 TMEM lanes
  const uint32_t bar0 = smem_u32(&mbar[0]);
  auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const uint32_t aA = smem_u32(sA), aW1 = smem_u32(sW1), aW2 = smem_u32(sW2), aW3 = smem_u32(sW3);
  const long long n_tiles = (rows + kRows - 1) / kRows;

  if (is_mma_warp) {
    // =============================== MMA issuer (one thread) =====================================
    if ((tid & 31) == 0) {
      uint32_t parity = 0;
      const uint32_t sbo1 = (uint32_t)(K1 / 8) * 128u, sboH = (uint32_t)(HID / 8) * 128u;
      const uint32_t w1_bytes = (uint32_t)(HID * K1 * 2);
      // resident weights: W2, W3 once (they land while the first tile is staged and goes through layer 1)
      mbar_expect_tx(bar(BAR_W23), (uint32_t)((HID + kNOut) * HID * 2));
      bulk_g2s(aW2, W.w2, (uint32_t)(HID * HID * 2), bar(BAR_W23));
      bulk_g2s(aW3, W.w3, (uint32_t)(kNOut * HID * 2), bar(BAR_W23));
      bool first = true;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        // W1 shares region A with the activation tile: re-fetched from L2 (40 KB) once the previous
        // tile's layer-3 MMAs have finished reading H2
        if (!first) mbar_wait_guarded(bar(BAR_L3), parity ^ 1);
        mbar_expect_tx(bar(BAR_W1), w1_bytes);
        bulk_g2s(aW1, W.w1, w1_bytes, bar(BAR_W1));
        // layer 1: acc0[128 x HID] = X W1^T, as soon as the tile is staged
        mbar_wait_guarded(bar(BAR_STAGE), parity);
        mbar_wait_guarded(bar(BAR_W1), parity);
        tc_fence_after();
        long long* tr = (W.trace != nullptr && blockIdx.x == 0) ? W.trace + (tile / gridDim.x) * 16 : nullptr;
        if (tr) tr[8] = clock64();    // MMA thread: tile staged, W1 landed
        for (int s = 0; s < K1 / 16; ++s)
          umma_bf16(acc0, umma_desc(aA + s * 256, 128, sbo1), umma_desc(aW1 + s * 256, 128, sbo1), umma_idesc(HID), s > 0);
        umma_commit(bar(BAR_L1));
        if (tr) tr[9] = clock64();    // layer-1 MMAs issued
        if (first) { mbar_wait_guarded(bar(BAR_W23), 0); first = false; }
        // layer 2: acc1 = H1 W2^T, K-steps follow the layer-1 epilogue chunk by chunk
        for (int j = 0; j < kChunks; ++j) {
          mbar_wait_guarded(bar(BAR_H1 + j), parity);
          tc_fence_after();
#pragma unroll
          for (int h = 0; h < G; ++h) {
#pragma unroll
            for (int q = 0; q < CW / 16; ++q) {
              const int s = (h * kGrpCols + j * CW) / 16 + q;
              umma_bf16(acc1, umma_desc(aA + s * 256, 128, sboH), umma_desc(aW2 + s * 256, 128, sboH), umma_idesc(HID),
                        (j | h | q) != 0);
            }
          }
        }
        umma_commit(bar(BAR_L2));
        if (tr) tr[10] = clock64();   // last layer-2 MMA issued
        // layer 3: acc0[128 x 16] = H2 W3^T, same pipelining against the layer-2 epilogue
        for (int j = 0; j < kChunks; ++j) {
          mbar_wait_guarded(bar(BAR_H2 + j), parity);
          tc_fence_after();
#pragma unroll
          for (int h = 0; h < G; ++h) {
#pragma unroll
            for (int q = 0; q < CW / 16; ++q) {
              const int s = (h * kGrpCols + j * CW) / 16 + q;
              umma_bf16(acc0, umma_desc(aA + s * 256, 128, sboH), umma_desc(aW3 + s * 256, 128, sboH), umma_idesc(kNOut),
                        (j | h | q) != 0);
            }
          }
        }
        umma_commit(bar(BAR_L3));
        if (tr) tr[11] = clock64();   // last layer-3 MMA issued
        parity ^= 1;
      }
    }
  } else {
    // =============================== staging + epilogue warps ====================================
    // The next tile's observation chunks are prefetched into registers while the current tile is in flight.
    constexpr int kMaxX = 16 / G;   // K1 <= 128: 16 chunks of 8 columns, dealt round-robin to the row's G threads
    const bool vec4 = (W.obs_dim & 3) == 0;   // rows are 16-byte aligned: two 128-bit loads per 8 columns
    // raw fp32 chunks stay in registers until the next tile starts: converting right after the load
    // would stall on the global latency that the prefetch is meant to hide
    auto load_x = [&](long long tile, float4 (&xa)[kMaxX], float4 (&xb)[kMaxX]) {
      const long long rg = tile * kRows + row;
      const bool ok = rg < rows;
      const float* src = obs + (size_t)rg * W.obs_dim;
#pragma unroll
      for (int c = 0; c < kMaxX; ++c) {
        const int k0 = (grp + c * G) * 8;      // the G threads of a row take alternate 8-column chunks
        xa[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        xb[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k0 < K1 && ok) {
          if (vec4 && k0 + 8 <= W.obs_dim) {
            xa[c] = __ldg(reinterpret_cast<const float4*>(src + k0));
            xb[c] = __ldg(reinterpret_cast<const float4*>(src + k0 + 4));
          } else {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = (k0 + j < W.obs_dim) ? __ldg(src + k0 + j) : 0.0f;
            xa[c] = make_float4(x[0], x[1], x[2], x[3]);
            xb[c] = make_float4(x[4], x[5], x[6], x[7]);
          }
        }
      }
    };
    // MeanStdNormalizer on load (normalization.py:84-88): statistics are per (agent, column)
    auto normalise_x = [&](long long tile, float4 (&xa)[kMaxX], float4 (&xb)[kMaxX]) {
      const long long rg = tile * kRows + row;
      const size_t base = (size_t)(rg % W.nperiod) * W.obs_dim;
      const float cl = W.nclip;
#pragma unroll
      for (int c = 0; c < kMaxX; ++c) {
        const int k0 = (grp + c * G) * 8;
        if (k0 < W.obs_dim) {
          float x[8] = {xa[c].x, xa[c].y, xa[c].z, xa[c].w, xb[c].x, xb[c].y, xb[c].z, xb[c].w};
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (k0 + j < W.obs_dim) {
              const float v = (x[j] - __ldg(W.nmean + base + k0 + j)) * __ldg(W.nrstd + base + k0 + j);
              x[j] = fminf(fmaxf(v, -cl), cl);
            }
          }
          xa[c] = make_float4(x[0], x[1], x[2], x[3]);
          xb[c] = make_float4(x[4], x[5], x[6], x[7]);
        }
      }
    };

    float4 xa[kMaxX], xb[kMaxX];
    uint32_t parity = 0;
    // Gaussian sample + log-prob of one row from the layer-3 accumulator values (already in registers)
    auto finish_row = [&](long long row_g, const uint32_t (&v)[16]) {
      float eps[4] = {0.f, 0.f, 0.f, 0.f};
      if (noise != nullptr) {
        for (int k = 0; k < W.act_dim; ++k) eps[k] = noise[(size_t)row_g * W.act_dim + k];
      } else {   // Philox4x32-10 keyed by the seed, counter = (row, call offset) -> 4 normals (Box-Muller)
        uint32_t c[4] = {(uint32_t)row_g, (uint32_t)((unsigned long long)row_g >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        const float u0 = ((c[0] >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = (c[1] >> 8) * (1.0f / 16777216.0f);
        const float u2 = ((c[2] >> 8) + 0.5f) * (1.0f / 16777216.0f), u3 = (c[3] >> 8) * (1.0f / 16777216.0f);
        const float r0 = sqrtf(-2.0f * __logf(u0)), r1 = sqrtf(-2.0f * __logf(u2));
        float s0, c0, s1, c1;
        __sincosf(6.28318530718f * u1, &s0, &c0);
        __sincosf(6.28318530718f * u3, &s1, &c1);
        eps[0] = r0 * c0; eps[1] = r0 * s0; eps[2] = r1 * c1; eps[3] = r1 * s1;
      }
      float lp = 0.f;
      for (int k = 0; k < W.act_dim; ++k) {
        const float m = __uint_as_float(v[k]) + sB3[k];
        const float ls = sLs[k];
        act[(size_t)row_g * W.act_dim + k] = fmaf(__expf(ls), eps[k], m);
        if (mean_out != nullptr) mean_out[(size_t)row_g * W.act_dim + k] = m;
        lp += -0.5f * eps[k] * eps[k] - ls - 0.91893853320467f;
      }
      logp[row_g] = lp;
    };
    auto stage_x = [&]() {   // prefetched fp32 chunks -> bf16, canonical K-major layout
#pragma unroll
      for (int c = 0; c < kMaxX; ++c) {
        const int k0 = (grp + c * G) * 8;
        if (k0 < K1)
          *reinterpret_cast<uint4*>(sA + canon_off(row, k0, K1)) =
              make_uint4(pack_bf16(xa[c].x, xa[c].y), pack_bf16(xa[c].z, xa[c].w), pack_bf16(xb[c].x, xb[c].y), pack_bf16(xb[c].z, xb[c].w));
      }
    };
    if ((long long)blockIdx.x < n_tiles) {
      load_x(blockIdx.x, xa, xb);
      if (W.nmean != nullptr) normalise_x(blockIdx.x, xa, xb);
      stage_x();
      proxy_fence();
      mbar_arrive(bar(BAR_STAGE));
      if ((long long)blockIdx.x + gridDim.x < n_tiles) load_x(blockIdx.x + gridDim.x, xa, xb);
    }
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const long long row_g = tile * kRows + row;
      const long long next = tile + gridDim.x;
      // ---- layer-1 epilogue: H1 over X / W1 (layer-1 MMAs are complete), chunks feed layer 2 --------
      long long* tr = (W.trace != nullptr && blockIdx.x == 0 && tid == 0) ? W.trace + (tile / gridDim.x) * 16 : nullptr;
      if (tr) tr[0] = clock64();      // waiting for layer 1
      mbar_wait_guarded(bar(BAR_L1), parity);
      tc_fence_after();
      if (tr) tr[1] = clock64();      // layer-1 accumulator ready
      epilogue_hidden<HID>(acc0 + lane_off, sB1, sA, row, cbeg, kChunks, bar(BAR_H1));
      tc_fence_before();
      if (tr) tr[2] = clock64();      // my layer-1 epilogue done
      // ---- layer-2 epilogue: H2 over H1 (layer-2 MMAs are complete), chunks feed layer 3 -------------
      mbar_wait_guarded(bar(BAR_L2), parity);
      tc_fence_after();
      if (tr) tr[3] = clock64();      // layer-2 accumulator ready
      epilogue_hidden<HID>(acc1 + lane_off, sB2, sA, row, cbeg, kChunks, bar(BAR_H2));
      tc_fence_before();
      if (tr) tr[4] = clock64();      // my layer-2 epilogue done
      // ---- layer 3 done: pull my row's 16 outputs out of TMEM, hand region A and acc0 to the next
      //      tile (its layer-1 MMA runs while this tile's rows are sampled and written) --------------
      mbar_wait_guarded(bar(BAR_L3), parity);
      tc_fence_after();
      if (tr) tr[5] = clock64();      // layer-3 accumulator ready
      parity ^= 1;
      uint32_t v[16];
      if (grp == 0) tmem_ld16(acc0 + lane_off, v);   // warp-uniform: warps 0-3 finish the rows
      if (next < n_tiles) {
        if (W.nmean != nullptr) normalise_x(next, xa, xb);
        stage_x();
        proxy_fence();       // generic-proxy smem writes -> visible to the tensor core (async proxy)
        tc_fence_before();   // my tcgen05.ld of this tile are complete (wait::ld) and ordered
        mbar_arrive(bar(BAR_STAGE));
      }
      if (tr) tr[6] = clock64();      // next tile staged
      if (grp == 0 && row_g < rows) finish_row(row_g, v);
      if (tr) tr[7] = clock64();      // rows sampled and written
      // prefetch the tile after next into registers.  Issued after the fences above and consumed one
      // tile later: a proxy fence waits for the thread's outstanding global loads
      if (next + gridDim.x < n_tiles) load_x(next + gridDim.x, xa, xb);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols));
}

// =================================================================================================
// TMEM-resident variant (hidden = 256): the hidden activations never leave tensor memory.
//
// The epilogue threads turn an accumulator row into the next layer's A operand IN PLACE: 16 fp32
// columns come out with tcgen05.ld, go through +bias / tanh, and are written back as 8 columns of packed
// bf16 pairs (tcgen05.st) at the start of the thread's own 64-column group, where the next layer's
// tcgen05.mma reads them as a TMEM A operand (K-major, column c = elements 2c | 2c+1).  Shared memory
// then holds only operands that never change (W1, W2: 168 KB) plus the staged observation tiles,
// so W1 is no longer re-fetched per tile, and the accumulator of layer 1 is free as soon as layer 2
// has consumed it: the MMA thread runs layer 1 of tile t+1 while the epilogue threads are still in
// tile t's second epilogue.  Loading / converting the observations and sampling / writing the finished
// rows are taken off the epilogue threads' critical path by four auxiliary warps (one thread per row).
//
// Layer 3 (hidden -> act_dim <= 4) does NOT go through the tensor pipe.  With a TMEM A operand an M = 128 instruction
// takes ~128 cycles whatever N is, so sixteen N = 16 MMAs cost as much pipe time as layer 2, and they kept accumulator 1
// occupied until the whole second epilogue had finished: layer 2 of the next tile could not run under that tile's first
// epilogue (tile period 3.9 us, 1.4 us of it epilogue threads waiting for layer 2).  Here the second epilogue keeps its
// tanh outputs in fp32 registers and multiplies them with W3 on the FMA pipe (epilogue_out below): H2 is never rounded
// to bf16 and never written anywhere; accumulator 1 is free as soon as every epilogue thread has loaded its last chunk.
//   per tile:  E (16 warps):    wait L1 | epilogue 1 (acc0 -> H1 in acc0) | wait L2 | epilogue 2 (acc1 -> tanh -> x W3 -> partials)
//              MMA (1 thread):  L2(t) chunk by chunk behind epilogue 1 | L1(t+1)
//              loader (4 warps):  X(t+NX): global fp32 -> (normalised) bf16 -> canonical tile in shared memory
//              sampler (3 warps): noise for tile t | wait partials | sum, + b3, sample, write rows
// TMEM: acc0 = columns [0,256), acc1 = [256,512).  Measured (262 144 rows, obs 72): 69 us (the layer-3-on-MMA version
// of this kernel 70, the shared-memory kernel above 83); tile period 3.6 us against an SFU floor of 2.1 us (2 x 128 x 256
// MUFU.TANH at 16 / clock / SM) — profiles/r2_actor_tmem_ncu.txt, r2_actor_tmem_trace.txt.
// epilogue | MMA | loader warps | sampler warps: 24 warps = 80 registers per thread (ptxas sizes the allocation for
// whole groups of four warps: 25 warps got 72 registers and spilled)
constexpr int kTEpi = 512, kTAux = 128, kTSamp = 96, kTThreads = kTEpi + 32 + kTAux + kTSamp;
// warp roles: the loader warps come first (lowest warp ids)
constexpr int kWLoad0 = 0, kWEpi0 = kTAux / 32, kWMma = kWEpi0 + kTEpi / 32, kWSamp0 = kWMma + 1;
enum { TB_W = 0, TB_L1, TB_L2, TB_OUT, TB_PFREE, TB_ACC1FREE, TB_XFULL, TB_XFREE = TB_XFULL + 2, TB_H1 = TB_XFREE + 2,
       TB_COUNT = TB_H1 + 4 };

__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc),
      "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&p)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(p[0]), "r"(p[1]), "r"(p[2]),
               "r"(p[3]), "r"(p[4]), "r"(p[5]), "r"(p[6]), "r"(p[7])
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 16 accumulator columns -> +bias, tanh -> 8 columns of bf16 pairs, in place
__device__ __forceinline__ void hidden_chunk_tmem(const uint32_t (&v)[16], const float* __restrict__ bias16, uint32_t dst) {
  const float4* b4 = reinterpret_cast<const float4*>(bias16);
  uint32_t p[8];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 b = b4[q];
    p[2 * q] = pack_bf16(tanh_fast(__uint_as_float(v[4 * q]) + b.x), tanh_fast(__uint_as_float(v[4 * q + 1]) + b.y));
    p[2 * q + 1] = pack_bf16(tanh_fast(__uint_as_float(v[4 * q + 2]) + b.z), tanh_fast(__uint_as_float(v[4 * q + 3]) + b.w));
  }
  tmem_st8(dst, p);
}

// one hidden epilogue of a thread: its 64 columns [64 g, 64 g + 64) of the accumulator row, four chunks
// of 16, each published (mbarrier) as soon as it is back in tensor memory
__device__ __forceinline__ void epilogue_tmem(uint32_t grp_base, const float* __restrict__ bias64, uint32_t chunk_bar0) {
  uint32_t va[16], vb[16];
  tmem_ld16_nowait(grp_base, va);
  tmem_wait_ld();
#pragma unroll
  for (int j = 0; j < 4; j += 2) {
    tmem_ld16_nowait(grp_base + 16u * (uint32_t)(j + 1), vb);
    hidden_chunk_tmem(va, bias64 + 16 * j, grp_base + 8u * (uint32_t)j);
    tmem_wait_st();
    tc_fence_before();
    mbar_arrive(chunk_bar0 + 8u * (uint32_t)j);
    tmem_wait_ld();
    if (j + 2 < 4) tmem_ld16_nowait(grp_base + 16u * (uint32_t)(j + 2), va);
    hidden_chunk_tmem(vb, bias64 + 16 * (j + 1), grp_base + 8u * (uint32_t)(j + 1));
    tmem_wait_st();
    tc_fence_before();
    mbar_arrive(chunk_bar0 + 8u * (uint32_t)(j + 1));
    if (j + 2 < 4) tmem_wait_ld();
  }
}

// Second epilogue: accumulator 1 -> +bias, tanh (fp32, never rounded) -> layer 3 on the FMA pipe.
// The accumulator is read with the 16x256b shape (the m16n8 fragment layout: thread t of a warp holds rows t/4 and
// t/4 + 8 of a 16-lane half, columns 8 j + 2 (t % 4) + {0, 1} of every 8-column block), so a thread's 64 elements are
// 4 rows x 16 columns instead of 1 row x 64 columns: one float4 of W3 (column c, outputs 0..3) then serves four rows.
// With one row per thread every tanh needed its own broadcast LDS.128, and a broadcast still returns 16 B to each of
// the 32 lanes — 2.1 us per tile on the 128 B / clock return path, twice the SFU time (measured; the constant bank was
// worse: ptxas turns the operands into LDCU.128, 3.1 us).  The four lanes that share rows exchange partial sums by
// shuffle (12 per tile) and each writes one finished row-partial over the warp group's 64 columns.
// (Packed fp32 pairs — fma.rn.f32x2 / FFMA2 over the two rows of a 16-lane half, W3 stored pre-duplicated — halve the
// FMA instructions but took 2.7 us per tile instead of 1.6: measured, reverted.)
__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}
// 16 columns [c0, c0 + 16) of the warp's 32 lanes: va = lanes 0..15, vb = lanes 16..31; o[r][k]: r = 2 * half + rowsel
__device__ __forceinline__ void out_chunk4(const uint32_t (&va)[8], const uint32_t (&vb)[8], const float* __restrict__ bias_c,
                                           const float4* __restrict__ w_c, float (&o)[4][4]) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {      // 8-column block j: my columns 8 j + {0, 1} (+ 2 (t % 4), folded into the pointers)
    const float2 b = *reinterpret_cast<const float2*>(bias_c + 8 * j);
    const float4 w0 = w_c[8 * j], w1 = w_c[8 * j + 1];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const uint32_t* v = (r < 2) ? va : vb;
      const float h0 = tanh_fast(__uint_as_float(v[4 * j + 2 * (r & 1)]) + b.x);
      const float h1 = tanh_fast(__uint_as_float(v[4 * j + 2 * (r & 1) + 1]) + b.y);
      o[r][0] = fmaf(h0, w0.x, o[r][0]); o[r][1] = fmaf(h0, w0.y, o[r][1]); o[r][2] = fmaf(h0, w0.z, o[r][2]); o[r][3] = fmaf(h0, w0.w, o[r][3]);
      o[r][0] = fmaf(h1, w1.x, o[r][0]); o[r][1] = fmaf(h1, w1.y, o[r][1]); o[r][2] = fmaf(h1, w1.z, o[r][2]); o[r][3] = fmaf(h1, w1.w, o[r][3]);
    }
  }
}
// grp_base: accumulator 1 at the warp's lane quadrant and 64-column group; bias_t / w_t already offset by the group's
// first column + 2 (t % 4).  Returns the partial sums of row 8 m + t / 4 of the quadrant, m = 2 (t & 1) + ((t >> 1) & 1).
__device__ __forceinline__ float4 epilogue_out(uint32_t grp_base, const float* __restrict__ bias_t, const float4* __restrict__ w_t,
                                               uint32_t acc_free, int lane) {
  float o[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int k = 0; k < 4; ++k) o[r][k] = 0.f;
  uint32_t va[8], vb[8], vc[8], vd[8];
  const uint32_t hi = grp_base + (16u << 16);
  tmem_ld_16x256b_x2(grp_base, va);
  tmem_ld_16x256b_x2(hi, vb);
  tmem_wait_ld();
  tmem_ld_16x256b_x2(grp_base + 16u, vc);
  tmem_ld_16x256b_x2(hi + 16u, vd);
  out_chunk4(va, vb, bias_t, w_t, o);
  tmem_wait_ld();
  tmem_ld_16x256b_x2(grp_base + 32u, va);
  tmem_ld_16x256b_x2(hi + 32u, vb);
  out_chunk4(vc, vd, bias_t + 16, w_t + 16, o);
  tmem_wait_ld();
  tmem_ld_16x256b_x2(grp_base + 48u, vc);
  tmem_ld_16x256b_x2(hi + 48u, vd);
  out_chunk4(va, vb, bias_t + 32, w_t + 32, o);
  tmem_wait_ld();
  tc_fence_before();
  mbar_arrive(acc_free);
  out_chunk4(vc, vd, bias_t + 48, w_t + 48, o);
  // rows are shared by the four lanes of a quad: halve the row set twice
  const bool odd = (lane & 1) != 0, up = (lane & 2) != 0;
  float a[2][4], b[4];
#pragma unroll
  for (int rr = 0; rr < 2; ++rr)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float recv = __shfl_xor_sync(0xffffffffu, odd ? o[rr][k] : o[rr + 2][k], 1);
      a[rr][k] = (odd ? o[rr + 2][k] : o[rr][k]) + recv;
    }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float recv = __shfl_xor_sync(0xffffffffu, up ? a[0][k] : a[1][k], 2);
    b[k] = (up ? a[1][k] : a[0][k]) + recv;
  }
  return make_float4(b[0], b[1], b[2], b[3]);
}

template <int NX>
__global__ void __launch_bounds__(kTThreads, 1)
actor_tmem_kernel(ActorDev W, const float* __restrict__ obs, long long rows, const float* __restrict__ noise,
                  unsigned long long seed, unsigned long long offset, float* __restrict__ act, float* __restrict__ logp,
                  float* __restrict__ mean_out) {
  constexpr int HID = 256;
  extern __shared__ __align__(128) unsigned char smem[];
  const int K1 = W.K1;
  __nv_bfloat16* sW1 = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* sW2 = sW1 + (size_t)HID * K1;
  __nv_bfloat16* sX = sW2 + (size_t)HID * HID;                 // NX tiles of [128 x K1]
  float* sB1 = reinterpret_cast<float*>(sX + (size_t)NX * kRows * K1);
  float* sB2 = sB1 + HID;
  float* sB3 = sB2 + HID;
  float* sLs = sB3 + kNOut;
  float4* sW3f = reinterpret_cast<float4*>(sLs + kNOut);       // [HID] columns x 4 outputs, fp32 values of the packed bf16 W3
  float4* sPart = sW3f + HID;                                  // [4 column groups][128 rows] partial layer-3 sums
  __shared__ __align__(8) uint64_t mbar[TB_COUNT];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < HID; i += kTThreads) { sB1[i] = W.b1[i]; sB2[i] = W.b2[i]; }
  if (tid < kNOut) { sB3[tid] = W.b3[tid]; sLs[tid] = W.logstd[tid]; }
  for (int c = tid; c < HID; c += kTThreads)     // rows >= act_dim of the packed W3 are zero
    sW3f[c] = make_float4(__bfloat162float(W.w3[canon_off(0, c, HID)]), __bfloat162float(W.w3[canon_off(1, c, HID)]),
                          __bfloat162float(W.w3[canon_off(2, c, HID)]), __bfloat162float(W.w3[canon_off(3, c, HID)]));
  {   // padded columns [obs_dim, K1) of the observation tiles stay zero for the kernel's lifetime
    uint4* z = reinterpret_cast<uint4*>(sX);
    const int n16 = NX * kRows * K1 / 8;
    for (int i = tid; i < n16; i += kTThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
    proxy_fence();
  }
  if (tid == 0) {
    mbar_init(smem_u32(&mbar[TB_W]), 1);
    mbar_init(smem_u32(&mbar[TB_L1]), 1);
    mbar_init(smem_u32(&mbar[TB_L2]), 1);
    mbar_init(smem_u32(&mbar[TB_OUT]), kTEpi);
    mbar_init(smem_u32(&mbar[TB_PFREE]), kTSamp);
    mbar_init(smem_u32(&mbar[TB_ACC1FREE]), kTEpi);
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&mbar[TB_XFULL + b]), kTAux);
      mbar_init(smem_u32(&mbar[TB_XFREE + b]), 1);
    }
    for (int j = 0; j < 4; ++j) {
      mbar_init(smem_u32(&mbar[TB_H1 + j]), kTEpi);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  const uint32_t acc0 = tmem_base, acc1 = tmem_base + 256u;
  const uint32_t bar0 = smem_u32(&mbar[0]);
  auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const long long n_tiles = (rows + kRows - 1) / kRows;
  const int n_local = (long long)blockIdx.x < n_tiles ? (int)((n_tiles - 1 - blockIdx.x) / gridDim.x) + 1 : 0;
  long long* const trace = (W.trace != nullptr && blockIdx.x == 0) ? W.trace : nullptr;

  if (warp == kWMma) {
    // =============================== MMA issuer (one thread) =====================================
    if (lane == 0 && n_local > 0) {
      const uint32_t sbo1 = (uint32_t)(K1 / 8) * 128u, sboH = (uint32_t)(HID / 8) * 128u;
      mbar_expect_tx(bar(TB_W), (uint32_t)((HID * K1 + HID * HID) * 2));
      bulk_g2s(smem_u32(sW1), W.w1, (uint32_t)(HID * K1 * 2), bar(TB_W));
      bulk_g2s(smem_u32(sW2), W.w2, (uint32_t)(HID * HID * 2), bar(TB_W));
      const uint64_t dW1 = umma_desc(smem_u32(sW1), 128, sbo1), dW2 = umma_desc(smem_u32(sW2), 128, sboH);
      const uint64_t dX0 = umma_desc(smem_u32(sX), 128, sbo1);
      const uint64_t x_stride = (uint64_t)((kRows * K1 * 2) >> 4);   // one observation tile, in descriptor address units
      constexpr uint32_t idH = umma_idesc(HID);
      const int k1_steps = K1 / 16;
      auto layer1 = [&](int i) {   // acc0 = X(i) W1^T; the commit also hands the observation buffer back
        const int b = i % NX;
        mbar_wait_guarded(bar(TB_XFULL + b), (uint32_t)(i / NX) & 1u);
        tc_fence_after();
        const uint64_t dX = dX0 + (uint64_t)b * x_stride;
        for (int s = 0; s < k1_steps; ++s) umma_bf16(acc0, dX + (uint64_t)(s * 16), dW1 + (uint64_t)(s * 16), idH, s > 0);
        umma_commit(bar(TB_L1));
        umma_commit(bar(TB_XFREE + b));
      };
      mbar_wait_guarded(bar(TB_W), 0);
      layer1(0);
      for (int i = 0; i < n_local; ++i) {
        const uint32_t p = (uint32_t)i & 1u;
        long long* tr = trace ? trace + (size_t)i * 16 : nullptr;
        // layer 2: acc1 = H1 W2^T, the K-steps follow the layer-1 epilogue chunk by chunk
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          mbar_wait_guarded(bar(TB_H1 + j), p);
          if (j == 0 && i > 0) mbar_wait_guarded(bar(TB_ACC1FREE), p ^ 1u);   // tile i-1's second epilogue has loaded its last chunk
          tc_fence_after();
#pragma unroll
          for (int g = 0; g < 4; ++g)
            umma_bf16_ts(acc1, acc0 + (uint32_t)(64 * g + 8 * j), dW2 + (uint64_t)((4 * g + j) * 16), idH, (j | g) != 0);
        }
        umma_commit(bar(TB_L2));
        if (tr) tr[10] = clock64();
        // layer 1 of the next tile: acc0 is free (layer 2 above read it in issue order)
        if (i + 1 < n_local) layer1(i + 1);
        if (tr) tr[9] = clock64();
      }
    }
  } else if (warp >= kWEpi0 && warp < kWMma) {
    // =============================== epilogue warps ==============================================
    const int grp = (warp - kWEpi0) >> 2;                                        // my 64-column group
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;                 // my warp's 32 TMEM lanes
    const uint32_t g0 = acc0 + lane_off + 64u * (uint32_t)grp, g1 = acc1 + lane_off + 64u * (uint32_t)grp;
    for (int i = 0; i < n_local; ++i) {
      const uint32_t p = (uint32_t)i & 1u;
      long long* tr = (trace && tid == kWEpi0 * 32) ? trace + (size_t)i * 16 : nullptr;
      if (tr) tr[0] = clock64();
      mbar_wait_guarded(bar(TB_L1), p);
      tc_fence_after();
      if (tr) tr[1] = clock64();
      epilogue_tmem(g0, sB1 + 64 * grp, bar(TB_H1));
      if (tr) tr[2] = clock64();
      mbar_wait_guarded(bar(TB_L2), p);
      tc_fence_after();
      if (tr) tr[3] = clock64();
      const float4 part = epilogue_out(g1, sB2 + 64 * grp + 2 * (lane & 3), sW3f + 64 * grp + 2 * (lane & 3), bar(TB_ACC1FREE), lane);
      if (i > 0) mbar_wait_guarded(bar(TB_PFREE), p ^ 1u);     // tile i-1's partial sums have been consumed (long ago)
      sPart[grp * kRows + (warp & 3) * 32 + 8 * (2 * (lane & 1) + ((lane >> 1) & 1)) + (lane >> 2)] = part;
      mbar_arrive(bar(TB_OUT));
      if (tr) tr[4] = clock64();
    }
  } else if (warp < kWEpi0) {
    // =============================== loader warps: observation tiles in ==========================
    // On their own (nothing else in their loop) so that a tile's global loads are in flight while the previous one is
    // still being converted; the loads of a tile are issued BEFORE the wait for its shared-memory buffer.
    const int q = warp & 3;                       // my warp's 32 rows of the tile
    const int od = W.obs_dim;
    const bool vec4 = (od & 3) == 0;
    // Fast path (obs_dim a multiple of 8, <= 80): lane = row.  A lane reads its row 32 bytes at a time (two LDG.128 at
    // immediate offsets) and writes one 16-byte core-matrix row per 8 columns (STS.128 at immediate offsets; eight
    // consecutive lanes fill one 128-byte core matrix, no bank conflicts): 27 memory instructions per lane and tile and
    // no index arithmetic.  Every LDG / STS / LDL of a loader warp queues behind the epilogue warps' MUFU.TANH in the
    // sub-partition's memory-IO queue (~100 cycles each while the epilogues run), so their NUMBER is what a tile costs
    // the loader: the first version (float4 units, offsets through two divisions, 4-byte-granular stores) took 3.8 us
    // per tile and was the slowest role of the kernel.
    constexpr int kMaxU = 10, kHalfU = 5;
    const int n8 = od >> 3;
    const bool fast = (od & 7) == 0 && n8 <= kMaxU;
    auto stage = [&](long long tile, int b, int wait_parity, long long* ltr) {     // fp32 rows -> (normalised) bf16, canonical K-major tile b
      __nv_bfloat16* dst = sX + (size_t)b * kRows * K1;
      bool waited = wait_parity < 0;
      const long long r0 = tile * kRows + q * 32;                 // the warp's 32 rows are contiguous in memory
      const bool norm = W.nmean != nullptr;
      const float cl = W.nclip;
      if (fast) {
        const long long rg = r0 + lane;
        const bool live = rg < rows;
        const float4* src = reinterpret_cast<const float4*>(obs + (size_t)rg * od);
        const uint32_t dst_l = smem_u32(dst) + (uint32_t)canon_off(q * 32 + lane, 0, K1) * 2u;
        {   // the tile this warp stages next: into L2 now (one 128-byte line per lane and step)
          const long long nt = tile + gridDim.x;
          if ((nt + 1) * kRows <= rows) {
            const char* nx = reinterpret_cast<const char*>(obs + (size_t)(nt * kRows + q * 32) * od);
            for (int o = lane * 128; o < 32 * od * 4; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + o));
          }
        }
        const float4 *nm = nullptr, *ns = nullptr;
        if (norm && live) {
          const size_t sidx = (size_t)(rg % W.nperiod) * od;
          nm = reinterpret_cast<const float4*>(W.nmean + sidx);
          ns = reinterpret_cast<const float4*>(W.nrstd + sidx);
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float4 x[kHalfU][2];
          if (ltr) ltr[12 + 2 * h] = clock64();
#pragma unroll
          for (int u = 0; u < kHalfU; ++u) {
            const int uu = h * kHalfU + u;
            if (uu < n8) {
              x[u][0] = live ? __ldg(src + 2 * uu) : make_float4(0.f, 0.f, 0.f, 0.f);
              x[u][1] = live ? __ldg(src + 2 * uu + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
          if (!waited) { mbar_wait_guarded(bar(TB_XFREE + b), (uint32_t)wait_parity); waited = true; }
          if (ltr) ltr[13 + 2 * h] = clock64() + (__float_as_uint(x[0][0].x) & 1u);   // after the wait and the first load's arrival
#pragma unroll
          for (int u = 0; u < kHalfU; ++u) {
            const int uu = h * kHalfU + u;
            if (uu < n8) {
              float4 v0 = x[u][0], v1 = x[u][1];
              if (nm != nullptr) {
                const float4 m0 = __ldg(nm + 2 * uu), m1 = __ldg(nm + 2 * uu + 1), s0 = __ldg(ns + 2 * uu), s1 = __ldg(ns + 2 * uu + 1);
                v0.x = fminf(fmaxf((v0.x - m0.x) * s0.x, -cl), cl); v0.y = fminf(fmaxf((v0.y - m0.y) * s0.y, -cl), cl);
                v0.z = fminf(fmaxf((v0.z - m0.z) * s0.z, -cl), cl); v0.w = fminf(fmaxf((v0.w - m0.w) * s0.w, -cl), cl);
                v1.x = fminf(fmaxf((v1.x - m1.x) * s1.x, -cl), cl); v1.y = fminf(fmaxf((v1.y - m1.y) * s1.y, -cl), cl);
                v1.z = fminf(fmaxf((v1.z - m1.z) * s1.z, -cl), cl); v1.w = fminf(fmaxf((v1.w - m1.w) * s1.w, -cl), cl);
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst_l + 128u * (uint32_t)uu), "r"(pack_bf16(v0.x, v0.y)),
                           "r"(pack_bf16(v0.z, v0.w)), "r"(pack_bf16(v1.x, v1.y)), "r"(pack_bf16(v1.z, v1.w))
                           : "memory");
            }
          }
        }
      } else if (vec4) {
        if (!waited) { mbar_wait_guarded(bar(TB_XFREE + b), (uint32_t)wait_parity); waited = true; }
        const int q4 = od >> 2, n4 = 32 * q4;
        const float4* src = reinterpret_cast<const float4*>(obs + (size_t)r0 * od);
        constexpr int U = 4;
        for (int f0 = lane; f0 < n4; f0 += 32 * U) {
          float4 x[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int f = f0 + 32 * u;
            const int r = f / q4;
            x[u] = (f < n4 && r0 + r < rows) ? __ldg(src + f) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int f = f0 + 32 * u;
            if (f < n4) {
              const int r = f / q4, c = (f - r * q4) * 4;
              float4 v = x[u];
              if (norm && r0 + r < rows) {
                const size_t sidx = (size_t)((r0 + r) % W.nperiod) * od + c;
                const float4 m = __ldg(reinterpret_cast<const float4*>(W.nmean + sidx));
                const float4 s = __ldg(reinterpret_cast<const float4*>(W.nrstd + sidx));
                v.x = fminf(fmaxf((v.x - m.x) * s.x, -cl), cl); v.y = fminf(fmaxf((v.y - m.y) * s.y, -cl), cl);
                v.z = fminf(fmaxf((v.z - m.z) * s.z, -cl), cl); v.w = fminf(fmaxf((v.w - m.w) * s.w, -cl), cl);
              }
              *reinterpret_cast<uint2*>(dst + canon_off(q * 32 + r, c, K1)) = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
            }
          }
        }
      } else {
        if (!waited) mbar_wait_guarded(bar(TB_XFREE + b), (uint32_t)wait_parity);
        const int n = 32 * od;
        const float* src = obs + (size_t)r0 * od;
        for (int e = lane; e < n; e += 32) {
          const int r = e / od, c = e - r * od;
          float v = 0.f;
          if (r0 + r < rows) {
            v = __ldg(src + e);
            if (norm) {
              const size_t sidx = (size_t)((r0 + r) % W.nperiod) * od + c;
              v = fminf(fmaxf((v - __ldg(W.nmean + sidx)) * __ldg(W.nrstd + sidx), -cl), cl);
            }
          }
          dst[canon_off(q * 32 + r, c, K1)] = __float2bfloat16(v);
        }
      }
      proxy_fence();               // generic-proxy writes -> visible to the tensor core (async proxy)
      mbar_arrive(bar(TB_XFULL + b));
    };
    for (int j = 0; j < n_local; ++j) {     // tile j goes into the buffer of tile j - NX, free once that tile's layer-1 MMAs have completed
      stage((long long)blockIdx.x + (long long)j * gridDim.x, j % NX, j >= NX ? ((j - NX) / NX) & 1 : -1,
            (trace && tid == 0 && j >= NX) ? trace + (size_t)(j - NX) * 16 : nullptr);
      if (trace && tid == 0 && j >= NX) trace[(size_t)(j - NX) * 16 + 6] = clock64();
    }
  } else {
    // =============================== sampler warps: finished rows out =============================
    // 96 threads for 128 rows: the first warp takes rows 96..127 in a second pass
    const int ts = tid - kWSamp0 * 32;
    for (int i = 0; i < n_local; ++i) {
     const long long tile = (long long)blockIdx.x + (long long)i * gridDim.x;
     long long* tr = (trace && ts == 0) ? trace + (size_t)i * 16 : nullptr;
     for (int row = ts; row < kRows; row += kTSamp) {
      // the row's Gaussian noise does not depend on the network: drawn while the tile is still in flight
      const long long row_g = tile * kRows + row;
      const bool live = row_g < rows;
      float eps[4] = {0.f, 0.f, 0.f, 0.f};
      if (live) {
        if (noise != nullptr) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k < W.act_dim) eps[k] = __ldg(noise + (size_t)row_g * W.act_dim + k);
        } else {   // Philox4x32-10 keyed by the seed, counter = (row, call offset) -> 4 normals (Box-Muller)
          uint32_t c[4] = {(uint32_t)row_g, (uint32_t)((unsigned long long)row_g >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
          philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
          const float u0 = ((c[0] >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = (c[1] >> 8) * (1.0f / 16777216.0f);
          const float u2 = ((c[2] >> 8) + 0.5f) * (1.0f / 16777216.0f), u3 = (c[3] >> 8) * (1.0f / 16777216.0f);
          const float ra = sqrtf(-2.0f * __logf(u0)), rb = sqrtf(-2.0f * __logf(u2));
          float s0, c0, s1, c1;
          __sincosf(6.28318530718f * u1, &s0, &c0);
          __sincosf(6.28318530718f * u3, &s1, &c1);
          eps[0] = ra * c0; eps[1] = ra * s0; eps[2] = rb * c1; eps[3] = rb * s1;
        }
      }
      if (row == ts) mbar_wait_guarded(bar(TB_OUT), (uint32_t)i & 1u);
      if (tr && row == ts) tr[5] = clock64();
      float v[4];
      {
        const float4 p0 = sPart[row], p1 = sPart[kRows + row], p2 = sPart[2 * kRows + row], p3 = sPart[3 * kRows + row];
        v[0] = (p0.x + p1.x) + (p2.x + p3.x); v[1] = (p0.y + p1.y) + (p2.y + p3.y);
        v[2] = (p0.z + p1.z) + (p2.z + p3.z); v[3] = (p0.w + p1.w) + (p2.w + p3.w);
      }
      if (row + kTSamp >= kRows) mbar_arrive(bar(TB_PFREE));   // the partial-sum rows may be overwritten by the next tile
      if (live) {
        float lp = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (k < W.act_dim) {
            const float m = v[k] + sB3[k];
            const float ls = sLs[k];
            act[(size_t)row_g * W.act_dim + k] = fmaf(__expf(ls), eps[k], m);
            if (mean_out != nullptr) mean_out[(size_t)row_g * W.act_dim + k] = m;
            lp += -0.5f * eps[k] * eps[k] - ls - 0.91893853320467f;
          }
        }
        logp[row_g] = lp;
      }
     }
     if (tr) tr[7] = clock64();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// fp32 [n x k] row-major (torch nn.Linear weight) -> bf16 canonical K-major [n_pad x k_pad], zero padded
__global__ void pack_weight_kernel(const float* __restrict__ w, int n, int k, int n_pad, int k_pad, __nv_bfloat16* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_pad * k_pad) return;
  const int r = idx / k_pad, c = idx - r * k_pad;
  const float v = (r < n && c < k) ? w[(size_t)r * k + c] : 0.0f;
  out[canon_off(r, c, k_pad)] = __float2bfloat16(v);
}
__global__ void pad_vector_kernel(const float* __restrict__ v, int n, int n_pad, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) out[i] = i < n ? v[i] : 0.0f;
}

}  // namespace

using ActorKernel = void (*)(ActorDev, const float*, long long, const float*, unsigned long long, unsigned long long, float*,
                             float*, float*);
static ActorKernel actor_kernel(int hidden) {
  return hidden == 256 ? actor_forward_kernel<256> : (hidden == 128 ? actor_forward_kernel<128> : actor_forward_kernel<64>);
}

struct bd_actor {
  int device, obs_dim, hidden, act_dim, K1, sm_count;
  __nv_bfloat16 *w1 = nullptr, *w2 = nullptr, *w3 = nullptr;
  float *b1 = nullptr, *b2 = nullptr, *b3 = nullptr, *logstd = nullptr;
  size_t smem = 0;
  int impl = 0;          // 0: activations through shared memory (actor_forward_kernel); 1 / 2: TMEM-resident activations
  size_t smem_t = 0;     //    (actor_tmem_kernel) with that many observation buffers
  int64_t launches = 0;
  long long* trace = nullptr;
  const float *nmean = nullptr, *nrstd = nullptr;
  int nperiod = 1;
  float nclip = 10.0f;
};

extern "C" {

const char* bd_actor_last_error(void) { return g_actor_err; }

int bd_actor_create(int obs_dim, int hidden, int act_dim, int device, bd_actor** out) {
  if (!out) return afail(BD_EINVAL, "bd_actor_create: null out");
  *out = nullptr;
  if (hidden != 256 && hidden != 128 && hidden != 64) return afail(BD_EINVAL, "bd_actor_create: hidden must be 64, 128 or 256");
  if (act_dim < 1 || act_dim > 4) return afail(BD_EINVAL, "bd_actor_create: act_dim must be in [1,4]");
  if (obs_dim < 1) return afail(BD_EINVAL, "bd_actor_create: obs_dim must be positive");
  const int K1 = (obs_dim + 15) & ~15;
  int prev = -1;
  if (cudaGetDevice(&prev) != cudaSuccess || cudaSetDevice(device) != cudaSuccess)
    return afail(BD_ECUDA, "bd_actor_create: cannot select device %d", device);
  bd_actor* a = new (std::nothrow) bd_actor();
  if (!a) return afail(BD_ENOMEM, "bd_actor_create: out of host memory");
  a->device = device; a->obs_dim = obs_dim; a->hidden = hidden; a->act_dim = act_dim; a->K1 = K1;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  a->sm_count = prop.multiProcessorCount;
  const size_t actb = (size_t)kRows * hidden * 2, l1b = (size_t)(kRows + hidden) * K1 * 2;
  const size_t regA = ((actb > l1b ? actb : l1b) + 127) & ~(size_t)127;
  a->smem = regA + (size_t)hidden * hidden * 2 + (size_t)kNOut * hidden * 2 + (size_t)(2 * hidden + 2 * kNOut) * 4;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes); };
  alloc((void**)&a->w1, (size_t)hidden * K1 * 2);
  alloc((void**)&a->w2, (size_t)hidden * hidden * 2);
  alloc((void**)&a->w3, (size_t)kNOut * hidden * 2);
  alloc((void**)&a->b1, hidden * 4); alloc((void**)&a->b2, hidden * 4);
  alloc((void**)&a->b3, kNOut * 4); alloc((void**)&a->logstd, kNOut * 4);
  if (hidden == 256) {   // TMEM-resident variant: W1 / W2 / W3 resident + one or two observation tiles
    const size_t fixed = (size_t)(hidden * K1 + hidden * hidden) * 2 + (size_t)(2 * hidden + 2 * kNOut) * 4 + (size_t)(hidden + 4 * kRows) * 16;
    const size_t xb = (size_t)kRows * K1 * 2, room = prop.sharedMemPerBlockOptin - 1024;   // static shared memory: barriers
    if (fixed + 2 * xb <= room) { a->impl = 2; a->smem_t = fixed + 2 * xb; }
    else if (fixed + xb <= room) { a->impl = 1; a->smem_t = fixed + xb; }
  }
  if (a->impl == 0 && a->smem > prop.sharedMemPerBlockOptin) {
    cudaFree(a->w1); cudaFree(a->w2); cudaFree(a->w3); cudaFree(a->b1); cudaFree(a->b2); cudaFree(a->b3); cudaFree(a->logstd);
    const size_t need = a->smem;
    delete a;
    if (prev >= 0 && prev != device) cudaSetDevice(prev);
    return afail(BD_EINVAL, "bd_actor_create: obs_dim %d with hidden %d needs %zu B of shared memory (> %zu)", obs_dim, hidden,
                 need, (size_t)prop.sharedMemPerBlockOptin);
  }
  if (e == cudaSuccess) {
    if (a->impl == 0)
      e = cudaFuncSetAttribute(actor_kernel(hidden), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)a->smem);
    else
      e = cudaFuncSetAttribute(a->impl == 2 ? actor_tmem_kernel<2> : actor_tmem_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)a->smem_t);
  }
  if (prev >= 0 && prev != device) cudaSetDevice(prev);
  if (e != cudaSuccess) {
    cudaFree(a->w1); cudaFree(a->w2); cudaFree(a->w3); cudaFree(a->b1); cudaFree(a->b2); cudaFree(a->b3); cudaFree(a->logstd);
    delete a;
    return afail(BD_ECUDA, "bd_actor_create: %s", cudaGetErrorString(e));
  }
  *out = a;
  return BD_OK;
}

void bd_actor_destroy(bd_actor* a) {
  if (!a) return;
  cudaFree(a->w1); cudaFree(a->w2); cudaFree(a->w3); cudaFree(a->b1); cudaFree(a->b2); cudaFree(a->b3); cudaFree(a->logstd);
  delete a;
}

int bd_actor_set_weights(bd_actor* a, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                         const float* b3, const float* logstd, void* stream) {
  if (!a || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !logstd) return afail(BD_EINVAL, "bd_actor_set_weights: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = a->hidden;
  auto grid = [](int n) { return (n + 255) / 256; };
  pack_weight_kernel<<<grid(H * a->K1), 256, 0, st>>>(w1, H, a->obs_dim, H, a->K1, a->w1);
  pack_weight_kernel<<<grid(H * H), 256, 0, st>>>(w2, H, H, H, H, a->w2);
  pack_weight_kernel<<<grid(kNOut * H), 256, 0, st>>>(w3, a->act_dim, H, kNOut, H, a->w3);
  pad_vector_kernel<<<grid(H), 256, 0, st>>>(b1, H, H, a->b1);
  pad_vector_kernel<<<grid(H), 256, 0, st>>>(b2, H, H, a->b2);
  pad_vector_kernel<<<1, 32, 0, st>>>(b3, a->act_dim, kNOut, a->b3);
  pad_vector_kernel<<<1, 32, 0, st>>>(logstd, a->act_dim, kNOut, a->logstd);
  a->launches += 7;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return afail(BD_ECUDA, "bd_actor_set_weights: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_actor_forward(bd_actor* a, const float* obs_dev, int64_t rows, const float* noise_dev, uint64_t seed, uint64_t offset,
                     float* act_dev, float* logp_dev, float* mean_dev, void* stream) {
  if (!a || !obs_dev || !act_dev || !logp_dev) return afail(BD_EINVAL, "bd_actor_forward: obs, act and logp are required");
  if (rows <= 0) return BD_OK;
  ActorDev W{a->w1, a->w2, a->w3, a->b1, a->b2, a->b3, a->logstd, a->obs_dim, a->K1, a->act_dim, a->nmean, a->nrstd, a->nperiod,
             a->nclip, a->trace};
  const long long n_tiles = (rows + kRows - 1) / kRows;
  const int grid = (int)(n_tiles < a->sm_count ? n_tiles : a->sm_count);   // persistent: one CTA per SM
  cudaStream_t st = (cudaStream_t)stream;
  if (a->impl != 0) {
    (a->impl == 2 ? actor_tmem_kernel<2> : actor_tmem_kernel<1>)<<<grid, kTThreads, a->smem_t, st>>>(W, obs_dev, rows, noise_dev, seed,
                                                                                                   offset, act_dev, logp_dev, mean_dev);
  } else {
    actor_kernel(a->hidden)<<<grid, ActorShape::kThreads, a->smem, st>>>(W, obs_dev, rows, noise_dev, seed, offset, act_dev, logp_dev,
                                                                        mean_dev);
  }
  a->launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return afail(BD_ECUDA, "bd_actor_forward: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_actor_set_input_norm(bd_actor* a, const float* mean_dev, const float* rstd_dev, int period, float clip) {
  if (!a) return afail(BD_EINVAL, "bd_actor_set_input_norm: null handle");
  if (mean_dev != nullptr && (rstd_dev == nullptr || period < 1 || !(clip > 0.f)))
    return afail(BD_EINVAL, "bd_actor_set_input_norm: rstd, period >= 1 and clip > 0 are required");
  a->nmean = mean_dev; a->nrstd = mean_dev ? rstd_dev : nullptr; a->nperiod = period > 0 ? period : 1; a->nclip = clip;
  return BD_OK;
}

int bd_actor_set_trace(bd_actor* a, long long* trace_dev) {
  if (!a) return afail(BD_EINVAL, "bd_actor_set_trace: null handle");
  a->trace = trace_dev;
  return BD_OK;
}

int64_t bd_actor_launch_count(const bd_actor* a) { return a ? a->launches : 0; }

}  // extern "C"
