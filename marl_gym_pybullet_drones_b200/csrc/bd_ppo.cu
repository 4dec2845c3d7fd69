// Hand-written PPO update for MAPPO on sm_100a (SURVEY.md 8f-1): the reference's `MAPPOAgent.update`
// (gym_pybullet_drones/mappo/agent.py:602-772) and `_compute_single_agent_returns` (mappo/buffer.py:561-614)
// without any library GEMM, autograd graph or elementwise torch kernel.
//
//   gae_kernel        returns / advantages as ONE backwards scan per env + the buffer-wide moments (buffer.py:561-695)
//   mlp_tile_kernel   per 128-row tile: gather rows by minibatch index -> 3-layer tanh MLP forward on tcgen05 (bf16
//                     operands, fp32 TMEM accumulators) -> PPO clipped-ratio loss / value loss and their gradient at the
//                     MLP output -> backward through both hidden layers on tcgen05; activations stay in shared memory,
//                     weights stream from L2 through a TMA slab ring; the tile's X, H1, H2, dZ2, dZ1, dZ3 leave the SM
//                     once, as bf16 UMMA tiles, for the weight-gradient pass
//   dw_kernel         weight gradients dW = dZ^T . input as tall-skinny GEMMs on tcgen05 with MN-major (transposed)
//                     operand descriptors straight over those tiles (TMA bulk loads, 3-stage ring), 256 x N fp32
//                     accumulators resident in TMEM over a CTA's whole row range; bias gradients by the idle warps
//   reduce_kernel     per-CTA partials -> flat gradient in torch parameter order (the unit of the NCCL all-reduce)
//   adam_kernel       torch.optim.Adam's arithmetic with the reference's KL gate decided on the device (agent.py:731)
//   pack_kernel       fp32 master weights -> bf16 K-step slabs for the next minibatch
//
// Why two tensor-core kernels and not one: the weight-gradient accumulators of the 256 x 256 layer are 256 KB of fp32 —
// all of an SM's tensor memory — so they cannot live next to the activation accumulators of the forward / backward
// chain; they get their own kernel, and the activations cross HBM exactly once in bf16 (280 KB per 128 rows).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/batch_drones.h"
#include "bd_umma.cuh"

namespace {
using namespace bdu;
typedef __nv_bfloat16 bf16;

constexpr int kRows = 128;          // rows per tile = UMMA M
constexpr int HID = 256;            // hidden width (both layers)
constexpr int kNOut = 16;           // output layer padded to the smallest UMMA N
constexpr int kSlabBytes = 8192;    // one K = 16 step of a 256-row weight operand
constexpr int kMaxStages = 8;       // weight slab ring: as many 8 KB stages as the tile kernel's other buffers leave room for
constexpr int kEpiThreads = 512;    // 4 threads per row (column groups of 64)
constexpr int kThreads = kEpiThreads + 64;   // + MMA warp + TMA warp
constexpr int kMaxPieces = 3;       // 8-column input pieces per thread and chunk (K1p <= 96)
constexpr int kStatSlots = 16;

thread_local char g_err[384] = "";
int pfail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// ---------------------------------------------------------------------------------------------
//                                   returns / advantages
// ---------------------------------------------------------------------------------------------
// One thread per env: the reward is shared by the env's agents (mappo.py:758-772), so every agent's sequence is the
// same scan.  vals (T+1, N): rollout values (zeros in the reference's rollout, agent.py:413) with the bootstrap value
// in row T.  acc[0..1] += sum adv, sum adv^2 (fp64); acc[2] += count.
__global__ void gae_kernel(const float* __restrict__ rew, const uint8_t* __restrict__ term, const uint8_t* __restrict__ trunc,
                           const float* __restrict__ vals, int T, int N, float gamma, float lam, int use_gae,
                           float* __restrict__ ret, float* __restrict__ adv, double* __restrict__ acc) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  double s1 = 0.0, s2 = 0.0;
  if (n < N) {
    float r_run = vals[(size_t)T * N + n], a_run = 0.f;
    for (int t = T - 1; t >= 0; --t) {
      const size_t i = (size_t)t * N + n;
      const float mask = (term[i] | trunc[i]) ? 0.f : 1.f;
      const float r = rew[i];                       // terminal_v is always 0 (mappo.py:827,845)
      r_run = r + gamma * mask * r_run;             // buffer.py:600
      if (use_gae) {
        const float td = r + gamma * mask * vals[i + N] - vals[i];
        a_run = a_run * lam * gamma * mask + td;    // :606-607
      } else {
        a_run = r_run - vals[i];
      }
      ret[i] = r_run;
      adv[i] = a_run;
      s1 += (double)a_run;
      s2 += (double)a_run * (double)a_run;
    }
  }
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  __shared__ double sh[2][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sh[0][warp] = s1; sh[1][warp] = s2; }
  __syncthreads();
  if (warp == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    s1 = lane < nw ? sh[0][lane] : 0.0;
    s2 = lane < nw ? sh[1][lane] : 0.0;
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if (lane == 0) {
      atomicAdd(acc + 0, s1);
      atomicAdd(acc + 1, s2);
      if (blockIdx.x == 0) atomicAdd(acc + 2, (double)T * (double)N);
    }
  }
}

// (sum, sum of squares, count) -> (mean, scale) with normalize_advantages' rule (buffer.py:666-695, numpy branch):
// population std; (adv - mean) / (std + eps), or adv - mean when std < eps.
__global__ void adv_stats_kernel(const double* __restrict__ acc, float* __restrict__ out2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const double n = acc[2] > 0.0 ? acc[2] : 1.0;
    const double mean = acc[0] / n;
    double var = acc[1] / n - mean * mean;
    var = var > 0.0 ? var : 0.0;
    const double sd = sqrt(var);
    out2[0] = (float)mean;
    out2[1] = (float)(sd < 1e-8 ? 1.0 : 1.0 / (sd + 1e-8));
  }
}

// ---------------------------------------------------------------------------------------------
//                       forward + loss + activation backward, one tile at a time
// ---------------------------------------------------------------------------------------------
struct NetDev {
  const bf16* w1_slabs;    // [C][K1p/16] slabs [256 n x 16 k]
  const bf16* w2f_slabs;   // [16] slabs [256 n x 16 k] in issue order i -> K-step 4*(i&3) + (i>>2)
  const bf16* w2b_slabs;   // [16] slabs [256 i x 16 j] = W2[j][i] (backward), same issue order over j
  const bf16* w3f;         // [16 o x 256 j] canonical, resident
  const bf16* w3b_slab;    // [256 j x 16 o] = W3[o][j]
  const float *b1, *b2, *b3, *logstd;   // b3 / logstd padded to 16
  int C, D, K1p, out_dim;
};


enum { MODE_ACTOR_TRAIN = 0, MODE_CRITIC_TRAIN = 1 };

struct TileArgs {
  NetDev net;
  int mode;
  const float* obs;          // (slots, N, M, D) raw observations
  int N, M;                  // envs per slot, agents per env
  const long long* idx;      // minibatch: sample s -> env-step index (t * N + n); nullptr = identity
  long long rows;            // actor: samples * M, critic: samples
  const float *act, *logp_old, *adv, *adv_stats;   // actor loss inputs (adv per env-step, stats = (mean, scale))
  const float *ret, *v_old;  // critic loss inputs per env-step
  float clip, use_clipped_value;
  const float *nmean, *nrstd;   // optional observation normalisation: per slot (t), per (agent, column)
  float nclip;
  bf16 *Xt, *H1t, *H2t, *dZ2t, *dZ1t, *dZ3t;   // tile scratch for dw_kernel
  double* stats;             // [0] sum loss, [1] sum (logp_old - logp), [2] rows, [3..6] dlogstd sums, [7..10] db3 sums
  int stages;                // ring depth (<= kMaxStages)
  long long* trace;          // diagnostics: CTA 0's epilogue thread 0 writes [tile][16] SM-clock stamps of its phases
};

enum { B_W3 = 0, B_XFULL, B_XEMPTY = B_XFULL + 2, B_L1 = B_XEMPTY + 2, B_L2, B_L3, B_D2, B_D1, B_Z3, B_TDONE, B_H1C,
       B_H2C = B_H1C + 4, B_Z2C = B_H2C + 4, B_FULL = B_Z2C + 4, B_EMPTY = B_FULL + kMaxStages, B_COUNT = B_EMPTY + kMaxStages };

__global__ void __launch_bounds__(kThreads, 1)
mlp_tile_kernel(const __grid_constant__ TileArgs P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const NetDev& W = P.net;
  const int K1p = W.K1p, C = W.C, D = W.D;
  bf16* bufH1 = reinterpret_cast<bf16*>(smem);                        // 64 KB: H1, later dZ1
  bf16* bufH2 = bufH1 + (size_t)kRows * HID;                          // 64 KB: H2, later dZ2
  // input chunks [128 x K1p]: one buffer for the actor (one chunk per tile, long consumed when the next tile is staged),
  // two for the centralised critic (chunk c + 1 is staged while the tensor core reads chunk c)
  const int nxb = C > 1 ? 2 : 1;
  const int kStages = P.stages;
  bf16* bufX = bufH2 + (size_t)kRows * HID;
  bf16* bufZ3 = bufX + (size_t)nxb * kRows * K1p;                     // [128 x 16]
  bf16* sW3 = bufZ3 + (size_t)kRows * kNOut;                          // [16 x 256]
  unsigned char* ring = reinterpret_cast<unsigned char*>(sW3 + (size_t)kNOut * HID);   // stages x 8 KB
  float* sB1 = reinterpret_cast<float*>(ring + (size_t)kStages * kSlabBytes);
  float* sB2 = sB1 + HID;
  float* sB3 = sB2 + HID;      // [16]
  float* sLs = sB3 + kNOut;    // [16]
  __shared__ __align__(8) uint64_t mbar[B_COUNT];
  __shared__ uint32_t tmem_base_s;
  __shared__ float s_red[11];   // CTA-wide sums of the tiles' statistics, flushed to P.stats once at the end

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < HID; i += kThreads) { sB1[i] = W.b1[i]; sB2[i] = W.b2[i]; }
  if (tid < kNOut) { sB3[tid] = W.b3[tid]; sLs[tid] = W.logstd != nullptr ? W.logstd[tid] : 0.f; }
  if (tid < 11) s_red[tid] = 0.f;
  if (tid == 0) {
    mbar_init(smem_u32(&mbar[B_W3]), 1);
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&mbar[B_XFULL + i]), kEpiThreads); mbar_init(smem_u32(&mbar[B_XEMPTY + i]), 1); }
    for (int i = B_L1; i <= B_D1; ++i) mbar_init(smem_u32(&mbar[i]), 1);
    mbar_init(smem_u32(&mbar[B_Z3]), kRows);
    mbar_init(smem_u32(&mbar[B_TDONE]), kEpiThreads);
    for (int i = 0; i < 4; ++i) {
      mbar_init(smem_u32(&mbar[B_H1C + i]), kEpiThreads);
      mbar_init(smem_u32(&mbar[B_H2C + i]), kEpiThreads);
      mbar_init(smem_u32(&mbar[B_Z2C + i]), kEpiThreads);
    }
    for (int i = 0; i < kMaxStages; ++i) { mbar_init(smem_u32(&mbar[B_FULL + i]), 1); mbar_init(smem_u32(&mbar[B_EMPTY + i]), 1); }
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
  const uint32_t acc0 = tmem_base, acc1 = tmem_base + (uint32_t)HID;
  const uint32_t bar0 = smem_u32(&mbar[0]);
  auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const uint32_t aH1 = smem_u32(bufH1), aH2 = smem_u32(bufH2), aX = smem_u32(bufX), aZ3 = smem_u32(bufZ3), aW3 = smem_u32(sW3),
                 aRing = smem_u32(ring);
  const long long n_tiles = (P.rows + kRows - 1) / kRows;
  const int k1_steps = K1p / 16;
  const uint32_t xbuf_bytes = (uint32_t)kRows * (uint32_t)K1p * 2u;

  if (warp == kEpiThreads / 32 + 1) {
    // ===================================== TMA producer ===========================================
    if (lane == 0) {
      mbar_expect_tx(bar(B_W3), (uint32_t)(kNOut * HID * 2));
      bulk_g2s(aW3, W.w3f, (uint32_t)(kNOut * HID * 2), bar(B_W3));
      // (replicating the slabs 8x in global memory, one copy per CTA modulo 8, changed nothing: the slab supply is not
      // an L2 hot-spot problem but the ring's round trip — measured, round 2, scripts/microbench/umma_rate.cu)
      uint32_t st = 0, epar = 1, lap0 = 1;   // first lap: the stages are free
      auto push = [&](const bf16* src) {
        if (!lap0) mbar_wait(bar(B_EMPTY + (int)st), epar);
        mbar_expect_tx(bar(B_FULL + (int)st), kSlabBytes);
        bulk_g2s(aRing + st * kSlabBytes, src, kSlabBytes, bar(B_FULL + (int)st));
        if (++st == (uint32_t)kStages) { st = 0; epar ^= 1; lap0 = 0; }
      };
      const int n1 = C * k1_steps;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int q = 0; q < n1; ++q) push(W.w1_slabs + (size_t)q * (kSlabBytes / 2));
#pragma unroll 4
        for (int q = 0; q < 16; ++q) push(W.w2f_slabs + (size_t)q * (kSlabBytes / 2));
        push(W.w3b_slab);
#pragma unroll 4
        for (int q = 0; q < 16; ++q) push(W.w2b_slabs + (size_t)q * (kSlabBytes / 2));
      }
    }
  } else if (warp == kEpiThreads / 32) {
    // ===================================== MMA issuer =============================================
    // The issuing thread runs alone: every instruction between two tcgen05.mma is latency the tensor pipe waits for
    // (scripts/microbench/umma_rate.cu: rebuilding both descriptors per K-step costs ~155 cycles per MMA against the 128
    // the pipe needs).  Descriptors are built once; a K-step adds 16 address units (256 B) to the activation
    // descriptor and the ring stage's 512 units (8 KB) select the slab.
    if (lane == 0) {
      unsigned long long xcnt = 0;
      uint32_t tpar = 0;
      const uint32_t sboX = (uint32_t)(K1p / 8) * 128u, sboH = (uint32_t)(HID / 8) * 128u;
      const uint64_t dX0 = umma_desc(aX, 128, sboX), dX1 = umma_desc(aX + xbuf_bytes, 128, sboX), dH1 = umma_desc(aH1, 128, sboH),
                     dH2 = umma_desc(aH2, 128, sboH), dW3 = umma_desc(aW3, 128, sboH), dZ3 = umma_desc(aZ3, 128, 256),
                     dRing = umma_desc(aRing, 128, 256);
      constexpr uint32_t kIdH = umma_idesc(HID), kIdO = umma_idesc(kNOut);
      uint32_t st = 0, fpar = 0;          // ring stage and the parity of its next FULL completion
      // one streamed K-step: wait for the slab, issue, hand the stage back when the MMA has read it
      auto ring_mma = [&](uint32_t acc, uint64_t adesc, uint32_t accumulate) {
        mbar_wait(bar(B_FULL + (int)st), fpar);
        umma_bf16(acc, adesc, dRing + (uint64_t)(st * (kSlabBytes >> 4)), kIdH, accumulate);
        umma_commit(bar(B_EMPTY + (int)st));
        if (++st == (uint32_t)kStages) { st = 0; fpar ^= 1; }
      };
      mbar_wait(bar(B_W3), 0);
      bool first = true;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (!first) { mbar_wait(bar(B_TDONE), tpar ^ 1); }   // previous tile's last epilogue has drained acc0
        first = false;
        tc_fence_after();
        // ---- layer 1: acc0 = sum_c X_c W1_c^T
        for (int c = 0; c < C; ++c, ++xcnt) {
          const int xb = nxb == 2 ? (int)(xcnt & 1) : 0;
          mbar_wait(bar(B_XFULL + xb), (uint32_t)((nxb == 2 ? (xcnt >> 1) : xcnt) & 1));
          tc_fence_after();
          const uint64_t dX = xb ? dX1 : dX0;
          for (int s = 0; s < k1_steps; ++s) ring_mma(acc0, dX + (uint64_t)(16 * s), (uint32_t)((c | s) != 0));
          umma_commit(bar(B_XEMPTY + xb));
        }
        umma_commit(bar(B_L1));
        // ---- layer 2: acc1 = H1 W2^T, K-steps follow the layer-1 epilogue chunk by chunk
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          mbar_wait(bar(B_H1C + j), tpar);
          tc_fence_after();
#pragma unroll
          for (int h = 0; h < 4; ++h) ring_mma(acc1, dH1 + (uint64_t)(16 * (h * 4 + j)), (uint32_t)((j | h) != 0));
        }
        umma_commit(bar(B_L2));
        // ---- layer 3: acc0[:, 0:16] = H2 W3^T
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          mbar_wait(bar(B_H2C + j), tpar);
          tc_fence_after();
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            const uint64_t o = (uint64_t)(16 * (h * 4 + j));
            umma_bf16(acc0, dH2 + o, dW3 + o, kIdO, (uint32_t)((j | h) != 0));
          }
        }
        umma_commit(bar(B_L3));
        // ---- dH2 = dZ3 W3 : acc1 = Z3[128 x 16] . slab[256 j x 16 o]^T
        mbar_wait(bar(B_Z3), tpar);
        tc_fence_after();
        ring_mma(acc1, dZ3, 0u);
        umma_commit(bar(B_D2));
        // ---- dH1 = dZ2 W2 : acc0 = dZ2[128 x 256 j] . slab_s[256 i x 16 j]^T over the 16 j-steps
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          mbar_wait(bar(B_Z2C + j), tpar);
          tc_fence_after();
#pragma unroll
          for (int h = 0; h < 4; ++h) ring_mma(acc0, dH2 + (uint64_t)(16 * (h * 4 + j)), (uint32_t)((j | h) != 0));
        }
        umma_commit(bar(B_D1));
        tpar ^= 1;
      }
    }
  } else {
    // ================================ staging + epilogue threads ==================================
    const int row = tid & (kRows - 1), grp = tid >> 7;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const int rps = P.mode == MODE_CRITIC_TRAIN ? 1 : P.M;   // rows per sample
    const int n_pieces = K1p / 8;
    const bool vec4 = (D & 3) == 0;
    float4 xa[kMaxPieces], xb4[kMaxPieces];
    long long cur_sample = 0;

    // env-step index of the sample a tile row belongs to (-1: padding row)
    auto sample_of = [&](long long tile) -> long long {
      const long long r = tile * kRows + row;
      if (r >= P.rows) return -1;
      const long long s = r / rps;
      return P.idx != nullptr ? P.idx[s] : s;
    };
    auto load_x = [&](long long tile, int c, long long samp) {
      const long long r = tile * kRows + row;
      const int agent = (rps == 1) ? c : (int)(r % rps);
      const float* src = P.obs + ((size_t)samp * P.M + agent) * D;
#pragma unroll
      for (int i = 0; i < kMaxPieces; ++i) {
        const int k0 = (grp + i * 4) * 8;
        xa[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        xb4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k0 < D && samp >= 0) {
          if (vec4 && k0 + 8 <= D) {
            xa[i] = __ldg(reinterpret_cast<const float4*>(src + k0));
            xb4[i] = __ldg(reinterpret_cast<const float4*>(src + k0 + 4));
          } else {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = (k0 + j < D) ? __ldg(src + k0 + j) : 0.0f;
            xa[i] = make_float4(x[0], x[1], x[2], x[3]);
            xb4[i] = make_float4(x[4], x[5], x[6], x[7]);
          }
        }
      }
    };
    // MeanStdNormalizer on load (normalization.py:84-88) with the statistics of the slot the row was observed in
    auto normalise_x = [&](long long tile, int c, long long samp) {
      if (P.nmean == nullptr || samp < 0) return;
      const long long r = tile * kRows + row;
      const int agent = (rps == 1) ? c : (int)(r % rps);
      const size_t base = ((size_t)(samp / P.N) * P.M + agent) * D;
#pragma unroll
      for (int i = 0; i < kMaxPieces; ++i) {
        const int k0 = (grp + i * 4) * 8;
        if (k0 < D) {
          float x[8] = {xa[i].x, xa[i].y, xa[i].z, xa[i].w, xb4[i].x, xb4[i].y, xb4[i].z, xb4[i].w};
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (k0 + j < D) {
              const float v = (x[j] - __ldg(P.nmean + base + k0 + j)) * __ldg(P.nrstd + base + k0 + j);
              x[j] = fminf(fmaxf(v, -P.nclip), P.nclip);
            }
          }
          xa[i] = make_float4(x[0], x[1], x[2], x[3]);
          xb4[i] = make_float4(x[4], x[5], x[6], x[7]);
        }
      }
    };
    auto stage_x = [&](int xbuf, long long tile, int c) {
      bf16* dst = bufX + (size_t)xbuf * kRows * K1p;
      bf16* gdst = P.Xt + ((size_t)tile * C + c) * (size_t)kRows * K1p;
#pragma unroll
      for (int i = 0; i < kMaxPieces; ++i) {
        const int p = grp + i * 4;
        if (p < n_pieces) {
          const uint4 pk = make_uint4(pack_bf16(xa[i].x, xa[i].y), pack_bf16(xa[i].z, xa[i].w), pack_bf16(xb4[i].x, xb4[i].y),
                                      pack_bf16(xb4[i].z, xb4[i].w));
          const size_t off = canon_off(row, p * 8, K1p);
          *reinterpret_cast<uint4*>(dst + off) = pk;
          *reinterpret_cast<uint4*>(gdst + off) = pk;
        }
      }
    };
    // forward epilogue: acc row -> +bias, tanh -> bf16 -> activation tile (next layer's A operand) + global copy
    auto epi_forward = [&](uint32_t acc, const float* bias, bf16* sH, bf16* gH, int chunk_bar) {
      uint32_t va[16], vb[16];
      tmem_ld16_nowait(acc + lane_off + (uint32_t)(grp * 64), va);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c0 = grp * 64 + j * 16;
        uint32_t* cur = (j & 1) ? vb : va;
        uint32_t* nxt = (j & 1) ? va : vb;
        if (j < 3) tmem_ld16_nowait(acc + lane_off + (uint32_t)(c0 + 16), nxt);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float z[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) z[e] = __uint_as_float(cur[q * 8 + e]) + bias[c0 + q * 8 + e];
          const uint4 pk = make_uint4(tanh2_bf16(z[0], z[1]), tanh2_bf16(z[2], z[3]), tanh2_bf16(z[4], z[5]), tanh2_bf16(z[6], z[7]));
          const size_t off = canon_off(row, c0 + q * 8, HID);
          *reinterpret_cast<uint4*>(sH + off) = pk;
          *reinterpret_cast<uint4*>(gH + off) = pk;
        }
        proxy_fence();
        mbar_arrive(bar(chunk_bar + j));
        tmem_wait_ld();
      }
    };
    // backward epilogue: dZ = dH * (1 - H^2), in place over H (bf16), + global copy
    auto epi_backward = [&](uint32_t acc, bf16* sH, bf16* gZ, int chunk_bar) {
      uint32_t va[16], vb[16];
      tmem_ld16_nowait(acc + lane_off + (uint32_t)(grp * 64), va);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c0 = grp * 64 + j * 16;
        uint32_t* cur = (j & 1) ? vb : va;
        uint32_t* nxt = (j & 1) ? va : vb;
        if (j < 3) tmem_ld16_nowait(acc + lane_off + (uint32_t)(c0 + 16), nxt);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const size_t off = canon_off(row, c0 + q * 8, HID);
          const uint4 hv = *reinterpret_cast<const uint4*>(sH + off);
          const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float h0, h1;
            unpack_bf16(hw[e], h0, h1);
            const float d0 = __uint_as_float(cur[q * 8 + 2 * e]) * fmaf(-h0, h0, 1.0f);
            const float d1 = __uint_as_float(cur[q * 8 + 2 * e + 1]) * fmaf(-h1, h1, 1.0f);
            o[e] = pack_bf16(d0, d1);
          }
          const uint4 pk = make_uint4(o[0], o[1], o[2], o[3]);
          *reinterpret_cast<uint4*>(sH + off) = pk;
          *reinterpret_cast<uint4*>(gZ + off) = pk;
        }
        if (chunk_bar >= 0) {
          proxy_fence();
          mbar_arrive(bar(chunk_bar + j));
        }
        tmem_wait_ld();
      }
    };

    unsigned long long xcnt = 0;
    uint32_t tpar = 0;
    if ((long long)blockIdx.x < n_tiles) {
      cur_sample = sample_of(blockIdx.x);
      load_x(blockIdx.x, 0, cur_sample);
    }
    long long* const tr0 = (P.trace != nullptr && blockIdx.x == 0 && tid == 0) ? P.trace : nullptr;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const long long next = tile + gridDim.x, next2 = next + gridDim.x;
      const long long samp = cur_sample;
      long long* const tr = (tr0 != nullptr && tile / gridDim.x < 16) ? tr0 + (tile / gridDim.x) * 16 : nullptr;
      if (tr) tr[0] = clock64();     // tile start
      // The minibatch index of the NEXT tile's row is requested here and used after this tile's inputs are staged, and
      // the one of the tile after that is used in the middle of this tile to pull its observation row into L2: read at
      // the point of use, index -> row is a dependent pair of latencies inside the staging phase (update 140.7 -> 138.4
      // ms at configs[4]'s shape).  Reading the row at the start of its own tile instead of holding it in 24 registers
      // across the previous one was slower (141.5 ms): the staging phase is long (5-8 k cycles) because its loads queue
      // behind the previous epilogue's 64 KB of activation stores, not because of the gather's own latency.
      const long long nsamp = next < n_tiles ? sample_of(next) : -1;
      const long long n2samp = next2 < n_tiles ? sample_of(next2) : -1;
      // the row's loss inputs (a gather by sample index) are requested now and used two epilogues later: read at the
      // point of use they cost a DRAM latency on the tile's critical path (2 k of 35 k cycles in the phase trace)
      float pre_a[4] = {0.f, 0.f, 0.f, 0.f}, pre_lpo = 0.f, pre_adv = 0.f;
      if (grp == 0 && samp >= 0) {
        if (P.mode == MODE_ACTOR_TRAIN) {
          const size_t arow = (size_t)samp * P.M + (int)((tile * kRows + row) % rps);
          for (int k = 0; k < W.out_dim; ++k) pre_a[k] = ldg_f1_pinned(P.act + arow * W.out_dim + k);
          pre_lpo = ldg_f1_pinned(P.logp_old + arow);
          pre_adv = ldg_f1_pinned(P.adv + samp);
        } else {
          pre_adv = ldg_f1_pinned(P.ret + samp);
          if (P.use_clipped_value > 0.f && P.v_old != nullptr) pre_lpo = ldg_f1_pinned(P.v_old + samp);
        }
      }
      // ---- stage the input chunks (actor: one, critic: one per agent); the next chunk is already on its way
      for (int c = 0; c < C; ++c, ++xcnt) {
        const int xbuf = nxb == 2 ? (int)(xcnt & 1) : 0;
        const unsigned long long use = nxb == 2 ? (xcnt >> 1) : xcnt;       // how often this buffer has been filled before
        if (use >= 1) mbar_wait(bar(B_XEMPTY + xbuf), (uint32_t)((use & 1) ^ 1));
        normalise_x(tile, c, samp);
        stage_x(xbuf, tile, c);
        proxy_fence();
        mbar_arrive(bar(B_XFULL + xbuf));
        if (c + 1 < C) load_x(tile, c + 1, samp);
        else if (next < n_tiles) { cur_sample = nsamp; load_x(next, 0, cur_sample); }
      }
      const size_t tbase = (size_t)tile * kRows * HID;
      // ---- H1
      if (tr) tr[1] = clock64();     // inputs staged
      mbar_wait(bar(B_L1), tpar);
      tc_fence_after();
      if (tr) tr[2] = clock64();     // layer 1 complete
      epi_forward(acc0, sB1, bufH1, P.H1t + tbase, B_H1C);
      tc_fence_before();
      if (tr) tr[3] = clock64();     // H1 written
      if (n2samp >= 0) {             // the row (actor) / the sample's M rows (critic) of the tile after the next one -> L2
        const int agent0 = (rps == 1) ? 0 : (int)((next2 * kRows + row) % rps);
        const char* b0 = reinterpret_cast<const char*>(P.obs + ((size_t)n2samp * P.M + agent0) * D);
        const char* b1 = b0 + (size_t)(rps == 1 ? P.M : 1) * D * 4;
        for (const char* a = reinterpret_cast<const char*>(reinterpret_cast<uintptr_t>(b0) & ~(uintptr_t)127) + grp * 128; a < b1; a += 4 * 128)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
      }
      // ---- H2
      mbar_wait(bar(B_L2), tpar);
      tc_fence_after();
      if (tr) tr[4] = clock64();     // layer 2 complete
      epi_forward(acc1, sB2, bufH2, P.H2t + tbase, B_H2C);
      tc_fence_before();
      if (tr) tr[5] = clock64();     // H2 written
      // ---- output layer, loss, gradient at the output (column group 0 owns the rows)
      if (grp == 0) {
        mbar_wait(bar(B_L3), tpar);
        tc_fence_after();
        if (tr) tr[6] = clock64();   // layer 3 complete
        uint32_t v[16];
        tmem_ld16_nowait(acc0 + lane_off, v);
        tmem_wait_ld();
        float dz[4] = {0.f, 0.f, 0.f, 0.f};
        float loss = 0.f, kl = 0.f, dls[4] = {0.f, 0.f, 0.f, 0.f}, cntv = 0.f;
        if (samp >= 0) {
          cntv = 1.f;
          if (P.mode == MODE_ACTOR_TRAIN) {
            // agent.py:617-640 with torch.distributions.Normal.log_prob summed over the action dims
            float lp = 0.f, diff[4], ivar[4];
            for (int k = 0; k < W.out_dim; ++k) {
              const float mu = __uint_as_float(v[k]) + sB3[k];
              const float ls = sLs[k];
              ivar[k] = __expf(-2.0f * ls);
              diff[k] = pre_a[k] - mu;
              lp += -0.5f * diff[k] * diff[k] * ivar[k] - ls - 0.91893853320467f;
            }
            const float lpo = pre_lpo;
            if (tr) tr[12] = clock64();   // loss inputs have arrived
            const float ratio = __expf(lp - lpo);
            const float a = (pre_adv - P.adv_stats[0]) * P.adv_stats[1];
            const float s1 = ratio * a;
            const float s2 = fminf(fmaxf(ratio, 1.0f - P.clip), 1.0f + P.clip) * a;
            loss = -fminf(s1, s2);
            kl = lpo - lp;
            // d(-min(s1, s2))/d lp: inside the clip range both branches are ratio * a; outside it the gradient
            // flows only when the unclipped branch is the minimum
            const bool inside = ratio >= 1.0f - P.clip && ratio <= 1.0f + P.clip;
            const float g = (inside || s1 < s2) ? -a * ratio : 0.f;
            for (int k = 0; k < W.out_dim; ++k) {
              dz[k] = g * diff[k] * ivar[k];
              dls[k] = g * (diff[k] * diff[k] * ivar[k] - 1.0f);
            }
          } else {
            // agent.py:643-700, centralised critic: target = mean over agents of identical returns
            const float vv = __uint_as_float(v[0]) + sB3[0];
            const float rt = pre_adv;            // prefetched P.ret[samp]
            float e = vv - rt;
            float l = e * e;
            if (P.use_clipped_value > 0.f) {
              const float vo = pre_lpo;          // prefetched P.v_old[samp] (0 without stored values)
              const float dvc = fminf(fmaxf(vv - vo, -P.clip), P.clip);
              const float ec = vo + dvc - rt;
              if (ec * ec > l) { l = ec * ec; e = (fabsf(vv - vo) <= P.clip) ? ec : 0.f; }
            }
            loss = 0.5f * l;
            dz[0] = e;
          }
        }
        // dZ3 tile [128 x 16] bf16, K-major (K = 16): my row's 16 entries = two core-matrix rows
        const uint4 lo = make_uint4(pack_bf16(dz[0], dz[1]), pack_bf16(dz[2], dz[3]), 0u, 0u);
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        const size_t off = canon_off(row, 0, kNOut);
        *reinterpret_cast<uint4*>(bufZ3 + off) = lo;
        *reinterpret_cast<uint4*>(bufZ3 + off + 64) = zero;
        bf16* g3 = P.dZ3t + (size_t)tile * kRows * kNOut;
        *reinterpret_cast<uint4*>(g3 + off) = lo;
        *reinterpret_cast<uint4*>(g3 + off + 64) = zero;
        proxy_fence();
        tc_fence_before();
        mbar_arrive(bar(B_Z3));
        if (tr) tr[13] = clock64();     // dZ3 handed to the tensor core
        // tile statistics: warp reduce, then one shared-memory atomic per value and warp; the CTA's sums go to global
        // memory once, when the kernel ends (11 double atomics per warp and tile on the same 11 addresses from every
        // CTA cost ~4 k of a tile's 35 k cycles: profiles/r2_ppo_tile_trace_actor.txt)
        float red[11] = {loss, kl, cntv, dls[0], dls[1], dls[2], dls[3], dz[0], dz[1], dz[2], dz[3]};
#pragma unroll
        for (int i = 0; i < 11; ++i) {
          float x = red[i];
          for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
          if (lane == 0 && x != 0.f) atomicAdd(&s_red[i], x);
        }
      }
      if (tr) tr[7] = clock64();     // loss / output rows done
      // ---- dZ2 = dH2 * (1 - H2^2), in place over H2; its chunks feed the dH1 MMAs
      mbar_wait(bar(B_D2), tpar);
      tc_fence_after();
      if (tr) tr[8] = clock64();   // dH2 complete
      epi_backward(acc1, bufH2, P.dZ2t + tbase, B_Z2C);
      tc_fence_before();
      if (tr) tr[9] = clock64();   // dZ2 written
      // ---- dZ1 = dH1 * (1 - H1^2)
      mbar_wait(bar(B_D1), tpar);
      tc_fence_after();
      if (tr) tr[10] = clock64();  // dH1 complete
      epi_backward(acc0, bufH1, P.dZ1t + tbase, -1);
      if (tr) tr[11] = clock64();  // dZ1 written
      tc_fence_before();
      mbar_arrive(bar(B_TDONE));
      tpar ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid < 11 && s_red[tid] != 0.f) atomicAdd(P.stats + tid, (double)s_red[tid]);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// ---------------------------------------------------------------------------------------------
//                    forward only, TWO tiles in flight per CTA (rollout actor / critic values)
// ---------------------------------------------------------------------------------------------
// The forward chain of one tile is latency-bound: MMA -> TMEM read -> tanh -> shared memory -> next MMA.  Here a CTA
// works on a PAIR of tiles (slots A, B) in strict alternation — the tensor core runs layer l of tile B while the 512
// epilogue threads turn tile A's accumulator into the next layer's operand, and vice versa — so both units always have
// work: 2 x 256 TMEM columns, 2 x 64 KB activation buffers, one input buffer [128 x K1p] per slot (the NEXT tile's input is
// staged between the hidden-layer epilogues of the current pair, so layer 1 of the next pair starts as soon as the
// output accumulator has been read), weights through a TMA slab ring (as many 8 KB stages as the rest leaves room for).
// mode FWD: out (rows, out_dim).  mode SAMPLE (`MAPPOActorCritic.step`, agent.py:389-415): act = mean + exp(logstd) eps,
// logp = sum_k [-eps_k^2/2 - logstd_k - log(2 pi)/2], eps from `noise` or Philox4x32-10(seed; row, offset).
constexpr int kF2MaxStages = 8;
struct Fwd2Args {
  NetDev net;
  int sample;                // 0: FWD, 1: SAMPLE
  int stages;                // ring depth (<= kF2MaxStages)
  const float* obs;
  int N, M;
  const long long* idx;
  long long rows;
  int rows_per_sample;       // M: row = (sample, agent) (actor); 1: row = sample, C input chunks (critic)
  const float *nmean, *nrstd;
  float nclip;
  float* out;                // FWD: (rows, out_dim); SAMPLE: actions (rows, out_dim)
  float* logp;               // SAMPLE: (rows)
  float* mean_out;           // SAMPLE: optional (rows, out_dim)
  const float* noise;        // SAMPLE: optional (rows, out_dim) standard normals
  unsigned long long seed, offset;
  long long* trace;          // diagnostics: CTA 0 writes [pair][64] SM-clock stamps (0..31 epilogue thread 0, 32..63 MMA thread)
};
enum { F_W3 = 0, F_XFULL, F_XEMPTY = F_XFULL + 2, F_L1 = F_XEMPTY + 2, F_L2 = F_L1 + 2, F_L3 = F_L2 + 2, F_H1 = F_L3 + 2,
       F_H2 = F_H1 + 2, F_OUT = F_H2 + 2, F_FULL = F_OUT + 2, F_EMPTY = F_FULL + kF2MaxStages, F_COUNT = F_EMPTY + kF2MaxStages };

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

__global__ void __launch_bounds__(kThreads, 1)
mlp_fwd2_kernel(const __grid_constant__ Fwd2Args P) {
  extern __shared__ __align__(128) unsigned char smem_f2[];   // no swizzle anywhere: 128 B is all the operands need
  const NetDev& W = P.net;
  const int K1p = W.K1p, C = W.C, D = W.D, stages = P.stages;
  bf16* const bufT0 = reinterpret_cast<bf16*>(smem_f2);                         // 2 x 64 KB activations
  bf16* const bufX0 = bufT0 + 2 * (size_t)kRows * HID;                       // 2 x [128 x K1p] inputs
  const uint32_t xbytes = (uint32_t)kRows * (uint32_t)K1p * 2u;
  bf16* sW3 = bufX0 + 2 * (size_t)kRows * K1p;
  unsigned char* ring = reinterpret_cast<unsigned char*>(sW3 + (size_t)kNOut * HID);
  float* sB1 = reinterpret_cast<float*>(ring + (size_t)stages * kSlabBytes);
  float* sB2 = sB1 + HID;
  float* sB3 = sB2 + HID;
  float* sLs = sB3 + kNOut;
  // barriers and the TMEM base live in the dynamic region too: static shared memory is accounted in whole KB, which
  // would cost a ring stage
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sLs + kNOut);
  uint32_t& tmem_base_s = *reinterpret_cast<uint32_t*>(mbar + F_COUNT);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < HID; i += kThreads) { sB1[i] = W.b1[i]; sB2[i] = W.b2[i]; }
  if (tid < kNOut) { sB3[tid] = W.b3[tid]; sLs[tid] = W.logstd != nullptr ? W.logstd[tid] : 0.f; }
  if (tid == 0) {
    mbar_init(smem_u32(&mbar[F_W3]), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&mbar[F_XFULL + i]), kEpiThreads); mbar_init(smem_u32(&mbar[F_XEMPTY + i]), 1);
      mbar_init(smem_u32(&mbar[F_L1 + i]), 1); mbar_init(smem_u32(&mbar[F_L2 + i]), 1); mbar_init(smem_u32(&mbar[F_L3 + i]), 1);
      mbar_init(smem_u32(&mbar[F_H1 + i]), kEpiThreads); mbar_init(smem_u32(&mbar[F_H2 + i]), kEpiThreads);
      mbar_init(smem_u32(&mbar[F_OUT + i]), kRows);
    }
    for (int i = 0; i < kF2MaxStages; ++i) { mbar_init(smem_u32(&mbar[F_FULL + i]), 1); mbar_init(smem_u32(&mbar[F_EMPTY + i]), 1); }
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
  const uint32_t bar0 = smem_u32(&mbar[0]);
  auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const uint32_t aT0 = smem_u32(bufT0), aX0 = smem_u32(bufX0), aW3 = smem_u32(sW3), aRing = smem_u32(ring);
  const uint32_t tbytes = (uint32_t)kRows * HID * 2u;
  const long long n_tiles = (P.rows + kRows - 1) / kRows;
  // this CTA's tiles: blockIdx.x, + gridDim.x, ...; position 2j goes to slot 0, 2j + 1 to slot 1
  const long long my_tiles = n_tiles > (long long)blockIdx.x ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int k1_steps = K1p / 16;

  if (warp == kEpiThreads / 32 + 1) {
    // ===================================== TMA producer ===========================================
    if (lane == 0) {
      mbar_expect_tx(bar(F_W3), (uint32_t)(kNOut * HID * 2));
      bulk_g2s(aW3, W.w3f, (uint32_t)(kNOut * HID * 2), bar(F_W3));
      unsigned long long cnt = 0;
      int st = 0;
      uint32_t epar = 1;       // parity of the EMPTY completion the next use of stage `st` must see (first lap: none)
      auto push = [&](const bf16* src) {
        if (cnt >= (unsigned long long)stages) mbar_wait(bar(F_EMPTY + st), epar);
        mbar_expect_tx(bar(F_FULL + st), kSlabBytes);
        bulk_g2s(aRing + (uint32_t)st * kSlabBytes, src, kSlabBytes, bar(F_FULL + st));
        ++cnt;
        if (++st == stages) { st = 0; epar ^= 1; }
      };
      const bf16 *w1s = W.w1_slabs, *w2fs = W.w2f_slabs;
      for (long long p = 0; p < my_tiles; p += 2) {
        const int nt = (p + 1 < my_tiles) ? 2 : 1;
        for (int t = 0; t < nt; ++t)
          for (int q = 0; q < C * k1_steps; ++q) push(w1s + (size_t)q * (kSlabBytes / 2));
        for (int t = 0; t < nt; ++t)
          for (int q = 0; q < 16; ++q) push(w2fs + (size_t)q * (kSlabBytes / 2));
      }
    }
  } else if (warp == kEpiThreads / 32) {
    // ===================================== MMA issuer =============================================
    // (descriptors built once, a K-step adds a constant: see mlp_tile_kernel; the slot loop stays a loop, the K-steps
    // of a layer are unrolled)
    if (lane == 0) {
      uint32_t st = 0, fpar = 0;
      uint32_t xpar = 0;                 // bit t: parity of slot t's next XFULL completion
      const uint32_t sboX = (uint32_t)(K1p / 8) * 128u, sboH = (uint32_t)(HID / 8) * 128u;
      const uint64_t dX = umma_desc(aX0, 128, sboX), dT = umma_desc(aT0, 128, sboH), dW3 = umma_desc(aW3, 128, sboH),
                     dRing = umma_desc(aRing, 128, 256);
      const uint64_t xstep = (uint64_t)(xbytes >> 4), tstep = (uint64_t)(tbytes >> 4);
      constexpr uint32_t kIdH = umma_idesc(HID), kIdO = umma_idesc(kNOut);
      auto ring_mma = [&](uint32_t acc, uint64_t adesc, uint32_t accumulate) {
        mbar_wait(bar(F_FULL + (int)st), fpar);
        umma_bf16(acc, adesc, dRing + (uint64_t)(st * (kSlabBytes >> 4)), kIdH, accumulate);
        umma_commit(bar(F_EMPTY + (int)st));
        if (++st == (uint32_t)stages) { st = 0; fpar ^= 1; }
      };
      mbar_wait(bar(F_W3), 0);
      uint32_t ppar = 0;
      long long* tr = (P.trace != nullptr && blockIdx.x == 0) ? P.trace + 32 : nullptr;
      auto stamp = [&](long long p, int id) { if (tr != nullptr && p < 64) tr[(p >> 1) * 64 + id] = clock64(); };
      for (long long p = 0; p < my_tiles; p += 2, ppar ^= 1) {
        const int nt = (p + 1 < my_tiles) ? 2 : 1;
        stamp(p, 0);
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {                     // layer 1 of A, then of B
          const uint32_t acc = tmem_base + (uint32_t)t * HID;
          if (p > 0) { mbar_wait(bar(F_OUT + t), ppar ^ 1); tc_fence_after(); }   // the slot's previous output has been read
          stamp(p, 1 + t);
          const uint64_t dXt = dX + xstep * (uint64_t)t;
#pragma unroll 1
          for (int c = 0; c < C; ++c) {
            mbar_wait(bar(F_XFULL + t), (xpar >> t) & 1u);
            xpar ^= 1u << t;
            tc_fence_after();
            for (int s = 0; s < k1_steps; ++s) ring_mma(acc, dXt + (uint64_t)(16 * s), (uint32_t)((c | s) != 0));
            umma_commit(bar(F_XEMPTY + t));
          }
          umma_commit(bar(F_L1 + t));
          stamp(p, 3 + t);
        }
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {                     // layer 2
          const uint32_t acc = tmem_base + (uint32_t)t * HID;
          mbar_wait(bar(F_H1 + t), ppar);
          tc_fence_after();
          stamp(p, 5 + t);
          const uint64_t dTt = dT + tstep * (uint64_t)t;
#pragma unroll
          for (int i = 0; i < 16; ++i)                     // K-step 4 (i & 3) + (i >> 2): the slabs' issue order (pack_kernel)
            ring_mma(acc, dTt + (uint64_t)(16 * (4 * (i & 3) + (i >> 2))), (uint32_t)(i != 0));
          umma_commit(bar(F_L2 + t));
          stamp(p, 7 + t);
        }
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {                     // layer 3
          const uint32_t acc = tmem_base + (uint32_t)t * HID;
          mbar_wait(bar(F_H2 + t), ppar);
          tc_fence_after();
          stamp(p, 9 + t);
          const uint64_t dTt = dT + tstep * (uint64_t)t;
#pragma unroll
          for (int s = 0; s < 16; ++s) umma_bf16(acc, dTt + (uint64_t)(16 * s), dW3 + (uint64_t)(16 * s), kIdO, (uint32_t)(s != 0));
          umma_commit(bar(F_L3 + t));
          stamp(p, 11 + t);
        }
      }
    }
  } else {
    // ================================ staging + epilogue threads ==================================
    const int row = tid & (kRows - 1), grp = tid >> 7;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const int rps = P.rows_per_sample;
    const int n_pieces = K1p / 8;
    const bool vec4 = (D & 3) == 0;
    float4 xa[kMaxPieces], xb4[kMaxPieces];      // one input chunk in flight (global -> registers -> bf16 tile)
    uint32_t xe = 0;                             // bit t: parity of the XEMPTY completion slot t's next staging must see
    uint32_t xused = 0;                          // bit t: slot t's input buffer has been staged before

    auto tile_of = [&](long long pos) { return (long long)blockIdx.x + pos * gridDim.x; };
    auto sample_of = [&](long long tile) -> long long {
      const long long r = tile * kRows + row;
      if (r >= P.rows) return -1;
      const long long s = r / rps;
      return P.idx != nullptr ? P.idx[s] : s;
    };
    auto load_x = [&](long long tile, int c, long long sm) {
      const long long r = tile * kRows + row;
      const int agent = (rps == 1) ? c : (int)(r % rps);
      const float* src = P.obs + ((size_t)(sm < 0 ? 0 : sm) * P.M + agent) * D;
#pragma unroll
      for (int i = 0; i < kMaxPieces; ++i) {
        const int k0 = (grp + i * 4) * 8;
        xa[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        xb4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k0 < D && sm >= 0) {
          if (vec4 && k0 + 8 <= D) {
            xa[i] = __ldg(reinterpret_cast<const float4*>(src + k0));
            xb4[i] = __ldg(reinterpret_cast<const float4*>(src + k0 + 4));
          } else {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = (k0 + j < D) ? __ldg(src + k0 + j) : 0.0f;
            xa[i] = make_float4(x[0], x[1], x[2], x[3]);
            xb4[i] = make_float4(x[4], x[5], x[6], x[7]);
          }
        }
      }
    };
    // registers -> (normalise) -> bf16 canonical tile of slot t; waits until the tensor core has consumed the slot's
    // previous chunk
    auto stage_x = [&](int t, long long tile, int c, long long sm) {
      const long long r = tile * kRows + row;
      const int agent = (rps == 1) ? c : (int)(r % rps);
      if ((xused >> t) & 1u) { mbar_wait(bar(F_XEMPTY + t), (xe >> t) & 1u); xe ^= 1u << t; }
      xused |= 1u << t;
      bf16* dst = reinterpret_cast<bf16*>(reinterpret_cast<unsigned char*>(bufX0) + (size_t)t * xbytes);
      const bool norm = P.nmean != nullptr && sm >= 0;
      const size_t nb = norm ? ((size_t)(sm / P.N) * P.M + agent) * D : 0;
#pragma unroll
      for (int i = 0; i < kMaxPieces; ++i) {
        const int pc = grp + i * 4;
        if (pc < n_pieces) {
          float x[8] = {xa[i].x, xa[i].y, xa[i].z, xa[i].w, xb4[i].x, xb4[i].y, xb4[i].z, xb4[i].w};
          if (norm) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int k = pc * 8 + j;
              if (k < D) {
                const float v = (x[j] - __ldg(P.nmean + nb + k)) * __ldg(P.nrstd + nb + k);
                x[j] = fminf(fmaxf(v, -P.nclip), P.nclip);
              }
            }
          }
          *reinterpret_cast<uint4*>(dst + canon_off(row, pc * 8, K1p)) =
              make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
        }
      }
      proxy_fence();
      mbar_arrive(bar(F_XFULL + t));
    };
    auto epi_hidden = [&](uint32_t acc, const float* bias, bf16* sH, int done_bar) {
      uint32_t va[16], vb[16];
      tmem_ld16_nowait(acc + lane_off + (uint32_t)(grp * 64), va);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c0 = grp * 64 + j * 16;
        uint32_t* cur = (j & 1) ? vb : va;
        uint32_t* nxt = (j & 1) ? va : vb;
        if (j < 3) tmem_ld16_nowait(acc + lane_off + (uint32_t)(c0 + 16), nxt);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float z[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) z[e] = __uint_as_float(cur[q * 8 + e]) + bias[c0 + q * 8 + e];
          *reinterpret_cast<uint4*>(sH + canon_off(row, c0 + q * 8, HID)) =
              make_uint4(tanh2_bf16(z[0], z[1]), tanh2_bf16(z[2], z[3]), tanh2_bf16(z[4], z[5]), tanh2_bf16(z[6], z[7]));
        }
        tmem_wait_ld();
      }
      proxy_fence();
      tc_fence_before();
      mbar_arrive(bar(done_bar));
    };
    auto finish_row = [&](long long r, const uint32_t (&v)[16]) {
      if (!P.sample) {
        for (int k = 0; k < W.out_dim; ++k) P.out[(size_t)r * W.out_dim + k] = __uint_as_float(v[k]) + sB3[k];
        return;
      }
      float eps[4] = {0.f, 0.f, 0.f, 0.f};
      if (P.noise != nullptr) {
        for (int k = 0; k < W.out_dim; ++k) eps[k] = P.noise[(size_t)r * W.out_dim + k];
      } else {   // Philox4x32-10 keyed by the seed, counter = (row, call offset) -> 4 normals (Box-Muller)
        uint32_t c[4] = {(uint32_t)r, (uint32_t)((unsigned long long)r >> 32), (uint32_t)P.offset, (uint32_t)(P.offset >> 32)};
        philox4x32_10(c, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
        const float u0 = ((c[0] >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = (c[1] >> 8) * (1.0f / 16777216.0f);
        const float u2 = ((c[2] >> 8) + 0.5f) * (1.0f / 16777216.0f), u3 = (c[3] >> 8) * (1.0f / 16777216.0f);
        const float r0 = sqrtf(-2.0f * __logf(u0)), r1 = sqrtf(-2.0f * __logf(u2));
        float s0, c0, s1, c1;
        __sincosf(6.28318530718f * u1, &s0, &c0);
        __sincosf(6.28318530718f * u3, &s1, &c1);
        eps[0] = r0 * c0; eps[1] = r0 * s0; eps[2] = r1 * c1; eps[3] = r1 * s1;
      }
      float lp = 0.f;
      for (int k = 0; k < W.out_dim; ++k) {
        const float m = __uint_as_float(v[k]) + sB3[k];
        const float ls = sLs[k];
        P.out[(size_t)r * W.out_dim + k] = fmaf(__expf(ls), eps[k], m);
        if (P.mean_out != nullptr) P.mean_out[(size_t)r * W.out_dim + k] = m;
        lp += -0.5f * eps[k] * eps[k] - ls - 0.91893853320467f;
      }
      P.logp[r] = lp;
    };

    // prologue: chunk 0 of both slots' first tiles
#pragma unroll 1
    for (int t = 0; t < 2; ++t)
      if (t < my_tiles) {
        const long long tile = tile_of(t), sm = sample_of(tile);
        load_x(tile, 0, sm);
        stage_x(t, tile, 0, sm);
      }
    uint32_t ppar = 0;
    long long* tr = (P.trace != nullptr && blockIdx.x == 0 && tid == 0) ? P.trace : nullptr;
    auto stamp = [&](long long p, int id) { if (tr != nullptr && p < 64) tr[(p >> 1) * 64 + id] = clock64(); };
    for (long long p = 0; p < my_tiles; p += 2, ppar ^= 1) {
      const int nt = (p + 1 < my_tiles) ? 2 : 1;
      stamp(p, 0);
      if (C > 1) {
        // centralised critic: the remaining input chunks of the current tiles, one by one (each waits for the tensor core
        // to release the slot's input buffer)
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {
          const long long tile = tile_of(p + t), sm = sample_of(tile);
#pragma unroll 1
          for (int c = 1; c < C; ++c) { load_x(tile, c, sm); stage_x(t, tile, c, sm); }
        }
      }
      // hidden layers: H1 of A while the tensor core runs layer 1 of B, H1 of B during layer 2 of A, ...
#pragma unroll 1
      for (int lt = 0; lt < 4; ++lt) {
        const int layer = lt >> 1, t = lt & 1;
        if (t >= nt) continue;
        const bool has_next = layer == 0 && p + t + 2 < my_tiles;
        const long long ntile = tile_of(p + t + 2);
        long long nsm = -1;
        if (has_next) { nsm = sample_of(ntile); load_x(ntile, 0, nsm); }   // in flight during the epilogue below
        mbar_wait(bar(F_L1 + 2 * layer + t), ppar);
        tc_fence_after();
        stamp(p, 1 + 3 * lt);
        epi_hidden(tmem_base + (uint32_t)t * HID, layer ? sB2 : sB1, bufT0 + (size_t)t * kRows * HID, F_H1 + 2 * layer + t);
        stamp(p, 2 + 3 * lt);
        if (has_next) stage_x(t, ntile, 0, nsm);           // layer 1 of this tile is complete: its input buffer is free
        stamp(p, 3 + 3 * lt);
      }
      if (grp == 0) {
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {
          mbar_wait(bar(F_L3 + t), ppar);
          tc_fence_after();
          stamp(p, 13 + 2 * t);
          uint32_t v[16];
          tmem_ld16_nowait(tmem_base + (uint32_t)t * HID + lane_off, v);
          tmem_wait_ld();
          tc_fence_before();
          mbar_arrive(bar(F_OUT + t));                     // the slot's accumulator may be overwritten by the next layer 1
          const long long r = tile_of(p + t) * kRows + row;
          if (r < P.rows) finish_row(r, v);
          stamp(p, 14 + 2 * t);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}
// dynamic shared memory of mlp_fwd2_kernel with `stages` ring stages
size_t fwd2_kernel_smem(int K1p, int stages) {
  return (size_t)2 * kRows * HID * 2 + (size_t)2 * kRows * K1p * 2 + (size_t)kNOut * HID * 2 + (size_t)stages * kSlabBytes +
         (size_t)(2 * HID + 2 * kNOut) * 4 + (size_t)F_COUNT * 8 + 16;
}
constexpr size_t kF2SmemBudget = 227 * 1024;          // the opt-in maximum (the kernel has no static shared memory)
int fwd2_stages(int K1p) {
  int st = kF2MaxStages;
  while (st > 2 && fwd2_kernel_smem(K1p, st) > kF2SmemBudget) --st;
  return st;
}

// dynamic shared memory of mlp_tile_kernel for a net with C input chunks of K1p columns and `stages` ring stages
size_t tile_kernel_smem(int C, int K1p, int stages) {
  return (size_t)2 * kRows * HID * 2 + (size_t)(C > 1 ? 2 : 1) * kRows * K1p * 2 + (size_t)kRows * kNOut * 2 + (size_t)kNOut * HID * 2 +
         (size_t)stages * kSlabBytes + (size_t)(2 * HID + 2 * kNOut) * 4;
}
constexpr size_t kTileSmemBudget = 227 * 1024 - 1024;   // opt-in maximum minus the kernel's static shared memory (barriers)
int tile_stages(int C, int K1p) {
  int st = kMaxStages;
  while (st > 2 && tile_kernel_smem(C, K1p, st) > kTileSmemBudget) --st;
  return st;
}

// ---------------------------------------------------------------------------------------------
//                         weight gradients: out[j][n] += sum_r A[r][j] B[r][n]
// ---------------------------------------------------------------------------------------------
constexpr int kDwStages = 3;
constexpr int kDwStageBytes = 65536;   // 64 rows of A (32 KB) + up to 32 KB of B operands
constexpr int kDwThreads = 192;        // warp 0: TMA, warp 1: MMA, warps 2-5: bias sums + final epilogue
constexpr int kDwMaxB = 3;
// input chunks one role-1 job can hold: 2 * K1p TMEM columns each, 32 columns spare, at most kDwMaxB operands
inline int chunks_per_job(int K1p) { const int c = (512 - 2 * kNOut) / (2 * K1p); return c < kDwMaxB ? c : kDwMaxB; }

struct DwJob {
  const bf16* A;                 // tiles [128 r x 256 j] canonical, 64 KB apart
  const bf16* B[kDwMaxB];        // tiles [128 r x nB] canonical
  long long b_stride[kDwMaxB];   // bytes between tiles of B[b]
  int nB[kDwMaxB];
  int n_b;
  float* out[kDwMaxB];           // partials [n_cta][256][nB]
  float* bias_out;               // partials [n_cta][256] (column sums of A) or nullptr
  int cta0, n_cta;
};
struct DwArgs {
  DwJob jobs[12];
  int n_jobs;
  long long tiles;
};

enum { DB_FULL = 0, DB_EMPTY = kDwStages, DB_DONE = 2 * kDwStages, DB_COUNT };

__global__ void __launch_bounds__(kDwThreads, 1)
dw_kernel(const __grid_constant__ DwArgs P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) uint64_t mbar[DB_COUNT];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int ji = 0;
  for (int k = 0; k < P.n_jobs; ++k)
    if ((int)blockIdx.x >= P.jobs[k].cta0 && (int)blockIdx.x < P.jobs[k].cta0 + P.jobs[k].n_cta) ji = k;
  const DwJob& J = P.jobs[ji];
  const int local = (int)blockIdx.x - J.cta0;
  const long long t0 = P.tiles * local / J.n_cta, t1 = P.tiles * (local + 1) / J.n_cta;
  const long long n_half = (t1 - t0) * 2;   // stages = half tiles (64 rows)
  const bool has_bias = J.bias_out != nullptr;
  if (tid == 0) {
    for (int i = 0; i < kDwStages; ++i) {
      mbar_init(smem_u32(&mbar[DB_FULL + i]), 1);
      mbar_init(smem_u32(&mbar[DB_EMPTY + i]), has_bias ? 5 : 1);
    }
    mbar_init(smem_u32(&mbar[DB_DONE]), 1);
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
  const uint32_t bar0 = smem_u32(&mbar[0]);
  auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const uint32_t aS = smem_u32(smem);
  uint32_t b_off[kDwMaxB], col0[kDwMaxB];
  {
    uint32_t o = 32768, c = 0;
    for (int b = 0; b < J.n_b; ++b) { b_off[b] = o; o += 64u * J.nB[b] * 2u; col0[b] = c; c += 2u * J.nB[b]; }
  }

  if (warp == 0) {
    if (lane == 0) {
      for (long long h = 0; h < n_half; ++h) {
        const int st = (int)(h % kDwStages);
        if (h >= kDwStages) mbar_wait(bar(DB_EMPTY + st), (uint32_t)(((h / kDwStages) & 1) ^ 1));
        const long long tile = t0 + (h >> 1);
        const int half = (int)(h & 1);
        uint32_t bytes = 32768;
        for (int b = 0; b < J.n_b; ++b) bytes += 64u * J.nB[b] * 2u;
        mbar_expect_tx(bar(DB_FULL + st), bytes);
        const uint32_t sbase = aS + (uint32_t)st * kDwStageBytes;
        bulk_g2s(sbase, reinterpret_cast<const unsigned char*>(J.A) + (size_t)tile * 65536 + (size_t)half * 32768, 32768,
                 bar(DB_FULL + st));
        for (int b = 0; b < J.n_b; ++b) {
          const uint32_t hb = 64u * J.nB[b] * 2u;
          bulk_g2s(sbase + b_off[b], reinterpret_cast<const unsigned char*>(J.B[b]) + (size_t)tile * J.b_stride[b] + (size_t)half * hb,
                   hb, bar(DB_FULL + st));
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // descriptors and instruction descriptors once (the issuing thread's own instructions are the tensor pipe's idle
      // time: scripts/microbench/umma_rate.cu); a stage adds kDwStageBytes / 16 address units, the upper 128 output rows
      // 2048 / 16, a K = 16 step 8192 / 16 (A) or 2 row groups (B)
      // A: M = j (contiguous in a core-matrix row), K = r.  8-row groups are 4096 B apart, 8-j groups 128 B.
      // (MN-major descriptors: LBO = K direction, SBO = M / N direction; verified on the B200 against autograd)
      const uint64_t adesc0 = umma_desc(aS, 4096, 128);
      uint64_t bdesc0[kDwMaxB], bstep[kDwMaxB];
      uint32_t idesc[kDwMaxB];
#pragma unroll
      for (int b = 0; b < kDwMaxB; ++b) {
        const uint32_t nb = b < J.n_b ? (uint32_t)J.nB[b] : 16u;
        const uint32_t rg = (nb / 8u) * 128u;               // bytes between 8-row groups of the B operand
        bdesc0[b] = umma_desc(aS + (b < J.n_b ? b_off[b] : 0u), rg, 128);
        bstep[b] = (uint64_t)((2u * rg) >> 4);
        idesc[b] = umma_idesc((int)nb, 1, 1);
      }
      uint32_t st = 0, fpar = 0;
      for (long long h = 0; h < n_half; ++h) {
        mbar_wait(bar(DB_FULL + (int)st), fpar);
        tc_fence_after();
        const uint64_t soff = (uint64_t)(st * (uint32_t)(kDwStageBytes >> 4));
#pragma unroll
        for (int b = 0; b < kDwMaxB; ++b) {
          if (b < J.n_b) {
#pragma unroll
            for (int mh = 0; mh < 2; ++mh) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                umma_bf16(tmem_base + col0[b] + (uint32_t)mh * (uint32_t)J.nB[b], adesc0 + soff + (uint64_t)(mh * 128 + ks * 512),
                          bdesc0[b] + soff + bstep[b] * (uint64_t)ks, idesc[b], (uint32_t)((h | ks) != 0));
            }
          }
        }
        umma_commit(bar(DB_EMPTY + (int)st));
        if (++st == (uint32_t)kDwStages) { st = 0; fpar ^= 1; }
      }
      umma_commit(bar(DB_DONE));
    }
  } else {
    // ---- bias gradient = column sums of A over my row range, while the tensor core works
    const int bt = tid - 64;          // 0..127
    const int w4 = bt >> 5;           // warp 0..3 of this group
    float acc[2][8];
#pragma unroll
    for (int p = 0; p < 2; ++p)
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[p][e] = 0.f;
    if (has_bias) {
      const int r8 = lane & 7, cgl = lane >> 3;       // row within an 8-row group, column group within my block of 4
      for (long long h = 0; h < n_half; ++h) {
        const int st = (int)(h % kDwStages);
        mbar_wait(bar(DB_FULL + st), (uint32_t)((h / kDwStages) & 1));
        const unsigned char* sA = smem + (size_t)st * kDwStageBytes;
#pragma unroll
        for (int p = 0; p < 2; ++p) {
          const int cg = p * 16 + w4 * 4 + cgl;       // 8-column group 0..31
#pragma unroll
          for (int rgi = 0; rgi < 8; ++rgi) {
            const uint4 v = *reinterpret_cast<const uint4*>(sA + (size_t)rgi * 4096 + (size_t)cg * 128 + (size_t)r8 * 16);
            const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float a, b;
              unpack_bf16(u[e], a, b);
              acc[p][2 * e] += a;
              acc[p][2 * e + 1] += b;
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(DB_EMPTY + st));
      }
#pragma unroll
      for (int p = 0; p < 2; ++p) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float x = acc[p][e];
          x += __shfl_xor_sync(0xffffffffu, x, 1);
          x += __shfl_xor_sync(0xffffffffu, x, 2);
          x += __shfl_xor_sync(0xffffffffu, x, 4);
          acc[p][e] = x;
        }
        if (r8 == 0) {
          const int cg = p * 16 + w4 * 4 + cgl;
          float* o = J.bias_out + (size_t)local * 256 + cg * 8;
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = acc[p][e];
        }
      }
    }
    // ---- final epilogue: TMEM -> per-CTA partial gradient
    mbar_wait(bar(DB_DONE), 0);
    tc_fence_after();
    const int q = warp & 3;                           // my TMEM lane quarter
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    for (int b = 0; b < J.n_b; ++b) {
      const int nB = J.nB[b];
      for (int mh = 0; mh < 2; ++mh) {
        const int j = mh * 128 + q * 32 + lane;
        float* o = J.out[b] + ((size_t)local * 256 + j) * nB;
        for (int c0 = 0; c0 < nB; c0 += 16) {
          uint32_t v[16];
          tmem_ld16_nowait(tmem_base + lane_off + col0[b] + (uint32_t)(mh * nB + c0), v);
          tmem_wait_ld();
          if (n_half > 0) {
#pragma unroll
            for (int e = 0; e < 16; e += 4)
              *reinterpret_cast<float4*>(o + c0 + e) = make_float4(__uint_as_float(v[e]), __uint_as_float(v[e + 1]),
                                                                   __uint_as_float(v[e + 2]), __uint_as_float(v[e + 3]));
          } else {
#pragma unroll
            for (int e = 0; e < 16; e += 4) *reinterpret_cast<float4*>(o + c0 + e) = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      }
    }
    if (has_bias && n_half == 0 && bt < 32) {
      for (int e = 0; e < 8; ++e) J.bias_out[(size_t)local * 256 + bt * 8 + e] = 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// ---------------------------------------------------------------------------------------------
//                   partials -> flat gradient, Adam, bf16 slab packing (small kernels)
// ---------------------------------------------------------------------------------------------
// Flat parameter layout = GatedAdam's: [logstd (actor only)] W1 (256 x Din) b1 W2 (256 x 256) b2 W3 (out x 256) b3,
// Din = C * D (torch nn.Linear weights are row-major (out, in)).
struct NetShape {
  int C, D, K1p, out_dim, has_logstd;
  __host__ __device__ int din() const { return C * D; }
  __host__ __device__ long long off_w1() const { return has_logstd ? out_dim : 0; }
  __host__ __device__ long long off_b1() const { return off_w1() + (long long)HID * din(); }
  __host__ __device__ long long off_w2() const { return off_b1() + HID; }
  __host__ __device__ long long off_b2() const { return off_w2() + (long long)HID * HID; }
  __host__ __device__ long long off_w3() const { return off_b2() + HID; }
  __host__ __device__ long long off_b3() const { return off_w3() + (long long)out_dim * HID; }
  __host__ __device__ long long count() const { return off_b3() + out_dim; }
};

struct ReduceArgs {
  NetShape s;
  const float* pw1[16];   // per input chunk: partials [n1][256][K1p]
  const float* pw2;       // [n2][256][256]
  const float* pw3;       // [n3][256][16]   (dW3 transposed)
  const float* pb1;       // [n1][256]
  const float* pb2;       // [n2][256]
  int n1, n2, n3;
  const double* stats;    // tile-kernel statistics (rows at [2], dlogstd sums at [3..6], db3 sums at [7..10])
  double* run_acc;        // optional running statistics over minibatches: [0] += mean loss, [1] += mean kl, [2] += 1, [3] += entropy loss
  const float* logstd;    // packed logstd (entropy statistic)
  float entropy_coef;
  long long rows_global;  // rows of the minibatch over ALL ranks (the mean's denominator); 0 = use stats[10]
  float* grad;            // flat
};

// sum of n per-CTA partials of one element, `stride` floats apart: eight loads in flight and four accumulators (one
// thread per element and one dependent add per load kept 66-148 DRAM / L2 round trips in sequence: 14 us per actor net)
__device__ __forceinline__ float sum_partials(const float* __restrict__ p, size_t stride, int n) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int i = 0;
  for (; i + 8 <= n; i += 8) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = __ldg(p + (size_t)(i + u) * stride);
    a0 += v[0]; a1 += v[1]; a2 += v[2]; a3 += v[3];
    a0 += v[4]; a1 += v[5]; a2 += v[6]; a3 += v[7];
  }
  for (; i < n; ++i) a0 += __ldg(p + (size_t)i * stride);
  return (a0 + a1) + (a2 + a3);
}

__global__ void reduce_kernel(const __grid_constant__ ReduceArgs P) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const NetShape& s = P.s;
  if (i >= s.count()) return;
  if (i == 0 && P.run_acc != nullptr) {
    // per-minibatch statistics the reference averages over an update (agent.py:738-741, 763-771); local rows
    const double lr_ = P.stats[2] > 0.0 ? P.stats[2] : 1.0;
    P.run_acc[0] += P.stats[0] / lr_;
    P.run_acc[1] += P.stats[1] / lr_;
    P.run_acc[2] += 1.0;
    if (s.has_logstd && P.logstd != nullptr) {
      double ent = 0.0;
      for (int k = 0; k < s.out_dim; ++k) ent += 0.5 + 0.91893853320467 + (double)P.logstd[k];   // Normal.entropy summed
      P.run_acc[3] += -ent;
    }
  }
  const double rows = P.rows_global > 0 ? (double)P.rows_global : (P.stats[2] > 0.0 ? P.stats[2] : 1.0);
  const float scale = (float)(1.0 / rows);
  float g = 0.f;
  if (i < s.off_w1()) {                                   // logstd: policy part + entropy bonus (agent.py:629-633,736)
    g = (float)P.stats[3 + i] * scale - P.entropy_coef;
  } else if (i < s.off_b1()) {
    const long long k = i - s.off_w1();
    const int j = (int)(k / s.din()), col = (int)(k % s.din());
    const int c = col / s.D, kk = col % s.D;
    const float* p = P.pw1[c] + (size_t)j * s.K1p + kk;
    g = sum_partials(p, (size_t)HID * s.K1p, P.n1) * scale;
  } else if (i < s.off_w2()) {
    const int j = (int)(i - s.off_b1());
    g = sum_partials(P.pb1 + j, HID, P.n1) * scale;
  } else if (i < s.off_b2()) {
    const long long k = i - s.off_w2();
    const float* p = P.pw2 + k;
    g = sum_partials(p, (size_t)HID * HID, P.n2) * scale;
  } else if (i < s.off_w3()) {
    const int j = (int)(i - s.off_b2());
    g = sum_partials(P.pb2 + j, HID, P.n2) * scale;
  } else if (i < s.off_b3()) {
    const long long k = i - s.off_w3();
    const int o = (int)(k / HID), j = (int)(k % HID);
    const float* p = P.pw3 + (size_t)j * kNOut + o;
    g = sum_partials(p, (size_t)HID * kNOut, P.n3) * scale;
  } else {
    g = (float)P.stats[7 + (i - s.off_b3())] * scale;
  }
  P.grad[i] = g;
}

// torch.optim.Adam (defaults) on the flat buffers, applied only when the gate holds: the reference skips the whole
// optimiser step — parameters, both moments, the step count — when approx_kl > 1.5 target_kl (agent.py:731).
// kl_sum / kl_rows: device scalars (after the cross-rank reduction); target_kl <= 0 or kl_sum == nullptr: no gate.
struct AdamArgs {
  float *param, *m, *v;
  const float* grad;
  double* step;            // torch keeps it as a float tensor; fp64 here for the bias corrections
  long long n;
  float lr, b1, b2, eps;
  const double* kl_sum;
  const double* kl_rows;
  float target_kl;
  double* gate_out;        // optional: 1.0 / 0.0 (statistics)
};
__device__ __forceinline__ bool adam_gate(const AdamArgs& P) {
  if (P.kl_sum == nullptr || !(P.target_kl > 0.f)) return true;
  const double rows = *P.kl_rows > 0.0 ? *P.kl_rows : 1.0;
  return (float)(*P.kl_sum / rows) <= 1.5f * P.target_kl;
}
__global__ void adam_kernel(const __grid_constant__ AdamArgs P) {
  // the bias corrections (two fp64 pow) once per block, not once per parameter
  __shared__ float s_step_size, s_bias2_sqrt;
  __shared__ int s_on;
  if (threadIdx.x == 0) {
    s_on = adam_gate(P) ? 1 : 0;
    const double step = *P.step + 1.0;
    s_step_size = (float)((double)P.lr / (1.0 - pow((double)P.b1, step)));
    s_bias2_sqrt = (float)sqrt(1.0 - pow((double)P.b2, step));
  }
  __syncthreads();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n || !s_on) return;
  const float g = P.grad[i];
  const float m = P.m[i] + (g - P.m[i]) * (1.0f - P.b1);            // torch.lerp(exp_avg, grad, 1 - beta1)
  const float v = P.v[i] * P.b2 + (g * g) * (1.0f - P.b2);
  const float step_size = s_step_size, bias2_sqrt = s_bias2_sqrt;
  const float denom = sqrtf(v) / bias2_sqrt + P.eps;
  P.param[i] = P.param[i] - step_size * (m / denom);
  P.m[i] = m;
  P.v[i] = v;
}
// after adam_kernel (every thread of which reads the step count): advance it — one thread of the repack kernel that
// follows the Adam kernel in the stream (it was a launch of its own: 3 us, 256 times per train step; together with the
// multi-accumulator partial sums and the per-block bias corrections: 184 launches fewer per train step, no measurable change
// of the step time in an A/B on one box — 137.8 / 138.4 vs 137.8 / 137.3 ms of update — the graph hides these kernels)
__device__ __forceinline__ void adam_advance(const AdamArgs& P) {
  const bool on = adam_gate(P);
  if (on) *P.step = *P.step + 1.0;
  if (P.gate_out != nullptr) *P.gate_out += on ? 1.0 : 0.0;
}

// fp32 master weights (flat, torch layout) -> bf16 slabs the tile kernel streams
struct PackArgs {
  NetShape s;
  const float* param;
  bf16 *w1_slabs, *w2f_slabs, *w2b_slabs, *w3f, *w3b_slab;
  float *b1, *b2, *b3, *logstd;
  AdamArgs adam;             // adam.step != nullptr: thread 0 advances the optimiser's step count (bd_ppo_adam_step)
};
__global__ void pack_kernel(const __grid_constant__ PackArgs P) {
  const NetShape& s = P.s;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && P.adam.step != nullptr) adam_advance(P.adam);
  const int k1_steps = s.K1p / 16;
  const long long n_w1 = (long long)s.C * k1_steps * 4096, n_w2 = 16LL * 4096, n_w3 = (long long)kNOut * HID;
  if (i < n_w1) {                        // slab (c, ks): [256 n x 16 kk]
    const long long slab = i / 4096;
    const int e = (int)(i % 4096), n = e / 16, kk = e % 16;
    const int c = (int)(slab / k1_steps), ks = (int)(slab % k1_steps);
    const int col = ks * 16 + kk;
    const float v = col < s.D ? P.param[s.off_w1() + (long long)n * s.din() + c * s.D + col] : 0.f;
    P.w1_slabs[slab * 4096 + canon_off(n, kk, 16)] = __float2bfloat16(v);
    return;
  }
  long long k = i - n_w1;
  if (k < n_w2) {                        // forward slab i_issue -> K-step ks = 4 (i & 3) + (i >> 2): W2[n][ks*16 + kk]
    const int slab = (int)(k / 4096), e = (int)(k % 4096), n = e / 16, kk = e % 16;
    const int ks = 4 * (slab & 3) + (slab >> 2);
    P.w2f_slabs[(size_t)slab * 4096 + canon_off(n, kk, 16)] = __float2bfloat16(P.param[s.off_w2() + (long long)n * HID + ks * 16 + kk]);
    // backward slab, same issue order over j: element (i = n, jj = kk) = W2[ks*16 + kk][n]
    P.w2b_slabs[(size_t)slab * 4096 + canon_off(n, kk, 16)] = __float2bfloat16(P.param[s.off_w2() + (long long)(ks * 16 + kk) * HID + n]);
    return;
  }
  k -= n_w2;
  if (k < n_w3) {                        // W3 forward [16 o x 256 j] canonical; backward slab [256 j x 16 o]
    const int o = (int)(k / HID), j = (int)(k % HID);
    const float v = o < s.out_dim ? P.param[s.off_w3() + (long long)o * HID + j] : 0.f;
    P.w3f[canon_off(o, j, HID)] = __float2bfloat16(v);
    P.w3b_slab[canon_off(j, o, 16)] = __float2bfloat16(v);
    return;
  }
  k -= n_w3;
  if (k < HID) { P.b1[k] = P.param[s.off_b1() + k]; P.b2[k] = P.param[s.off_b2() + k]; return; }
  k -= HID;
  if (k < kNOut) {
    P.b3[k] = k < s.out_dim ? P.param[s.off_b3() + k] : 0.f;
    if (P.logstd != nullptr) P.logstd[k] = (s.has_logstd && k < s.out_dim) ? P.param[k] : 0.f;
  }
}
long long pack_threads(const NetShape& s) { return (long long)s.C * (s.K1p / 16) * 4096 + 16LL * 4096 + (long long)kNOut * HID + HID + kNOut; }

}  // namespace

// =================================================================================================
//                                          C-ABI
// =================================================================================================
struct bd_ppo_net {
  int device, sm_count;
  NetShape s;
  long long max_rows, max_tiles;
  // packed weights
  bf16 *w1_slabs = nullptr, *w2f_slabs = nullptr, *w2b_slabs = nullptr, *w3f = nullptr, *w3b_slab = nullptr;
  float *b1 = nullptr, *b2 = nullptr, *b3 = nullptr, *logstd = nullptr;
  // tile scratch
  bf16 *Xt = nullptr, *H1t = nullptr, *H2t = nullptr, *dZ2t = nullptr, *dZ1t = nullptr, *dZ3t = nullptr;
  // gradient partials
  float *pw1 = nullptr, *pw2 = nullptr, *pw3 = nullptr, *pb1 = nullptr, *pb2 = nullptr;
  int n1 = 0, n2 = 0;            // CTAs of the two weight-gradient roles
  int n3 = 0;                    // CTAs of the separate dW3 launch
  int n1_jobs = 1;               // input chunks are spread over this many role-1 jobs (TMEM: 512 columns)
  double* stats = nullptr;       // [kStatSlots]
  long long* trace = nullptr;    // diagnostics (bd_ppo_set_trace)
  int64_t launches = 0;
};

namespace {
void free_net(bd_ppo_net* n) {
  cudaFree(n->w1_slabs); cudaFree(n->w2f_slabs); cudaFree(n->w2b_slabs); cudaFree(n->w3f); cudaFree(n->w3b_slab);
  cudaFree(n->b1); cudaFree(n->b2); cudaFree(n->b3); cudaFree(n->logstd);
  cudaFree(n->Xt); cudaFree(n->H1t); cudaFree(n->H2t); cudaFree(n->dZ2t); cudaFree(n->dZ1t); cudaFree(n->dZ3t);
  cudaFree(n->pw1); cudaFree(n->pw2); cudaFree(n->pw3); cudaFree(n->pb1); cudaFree(n->pb2); cudaFree(n->stats);
}
NetDev net_dev(const bd_ppo_net* n) {
  NetDev d;
  d.w1_slabs = n->w1_slabs; d.w2f_slabs = n->w2f_slabs; d.w2b_slabs = n->w2b_slabs; d.w3f = n->w3f; d.w3b_slab = n->w3b_slab;
  d.b1 = n->b1; d.b2 = n->b2; d.b3 = n->b3; d.logstd = n->s.has_logstd ? n->logstd : nullptr;
  d.C = n->s.C; d.D = n->s.D; d.K1p = n->s.K1p; d.out_dim = n->s.out_dim;
  return d;
}
}  // namespace

extern "C" {

const char* bd_ppo_last_error(void) { return g_err; }

int bd_ppo_net_create(int in_dim, int chunks, int out_dim, int has_logstd, int64_t max_rows, int device, bd_ppo_net** out) {
  if (!out) return pfail(BD_EINVAL, "bd_ppo_net_create: null out");
  *out = nullptr;
  if (in_dim < 1 || in_dim > 96) return pfail(BD_EINVAL, "bd_ppo_net_create: in_dim (per chunk) must be in [1,96]");
  if (chunks < 1 || chunks > 16) return pfail(BD_EINVAL, "bd_ppo_net_create: chunks must be in [1,16]");
  if (out_dim < 1 || out_dim > 4) return pfail(BD_EINVAL, "bd_ppo_net_create: out_dim must be in [1,4]");
  if (max_rows < 1) return pfail(BD_EINVAL, "bd_ppo_net_create: max_rows must be positive");
  int prev = -1;
  if (cudaGetDevice(&prev) != cudaSuccess || cudaSetDevice(device) != cudaSuccess)
    return pfail(BD_ECUDA, "bd_ppo_net_create: cannot select device %d", device);
  bd_ppo_net* n = new (std::nothrow) bd_ppo_net();
  if (!n) return pfail(BD_ENOMEM, "bd_ppo_net_create: out of host memory");
  n->device = device;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  n->sm_count = prop.multiProcessorCount;
  n->s.C = chunks; n->s.D = in_dim; n->s.K1p = (in_dim + 15) & ~15; n->s.out_dim = out_dim; n->s.has_logstd = has_logstd ? 1 : 0;
  n->max_rows = max_rows;
  n->max_tiles = (max_rows + kRows - 1) / kRows;
  // weight-gradient roles: role 2 = dW2 (512 TMEM columns); role 1 = dW1 chunks + dW3, as many jobs as the 512 columns need
  const int per_job = chunks_per_job(n->s.K1p);
  n->n1_jobs = (chunks + per_job - 1) / per_job;
  const int sms = n->sm_count;
  int n2 = (int)(sms * 0.45), n1 = (sms - n2) / n->n1_jobs;
  if (n1 < 1) n1 = 1;
  n2 = sms - n1 * n->n1_jobs;
  if (n2 < 1) n2 = 1;
  n->n1 = n1; n->n2 = n2;
  // dW3^T = H2^T dZ3 streams the whole H2 tile array through a 256 x 16 accumulator: bandwidth-bound, so it runs on every SM
  // (it used the role-1 CTA count: 82 CTAs for the actor, 13 for the 16-agent critic = 23 us for 17 MB)
  n->n3 = sms;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes); };
  const size_t k1s = n->s.K1p / 16;
  alloc((void**)&n->w1_slabs, (size_t)chunks * k1s * kSlabBytes);
  alloc((void**)&n->w2f_slabs, 16 * (size_t)kSlabBytes); alloc((void**)&n->w2b_slabs, 16 * (size_t)kSlabBytes);
  alloc((void**)&n->w3f, (size_t)kNOut * HID * 2); alloc((void**)&n->w3b_slab, kSlabBytes);
  alloc((void**)&n->b1, HID * 4); alloc((void**)&n->b2, HID * 4); alloc((void**)&n->b3, kNOut * 4); alloc((void**)&n->logstd, kNOut * 4);
  const size_t T = (size_t)n->max_tiles;
  alloc((void**)&n->Xt, T * chunks * kRows * n->s.K1p * 2);
  alloc((void**)&n->H1t, T * kRows * HID * 2); alloc((void**)&n->H2t, T * kRows * HID * 2);
  alloc((void**)&n->dZ2t, T * kRows * HID * 2); alloc((void**)&n->dZ1t, T * kRows * HID * 2);
  alloc((void**)&n->dZ3t, T * kRows * kNOut * 2);
  alloc((void**)&n->pw1, (size_t)chunks * n1 * HID * n->s.K1p * 4);
  alloc((void**)&n->pw2, (size_t)n2 * HID * HID * 4);
  alloc((void**)&n->pw3, (size_t)n->n3 * HID * kNOut * 4);
  alloc((void**)&n->pb1, (size_t)n1 * HID * 4); alloc((void**)&n->pb2, (size_t)n2 * HID * 4);
  alloc((void**)&n->stats, kStatSlots * sizeof(double));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mlp_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmemBudget);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(mlp_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kF2SmemBudget);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDwStages * kDwStageBytes);
  if (prev >= 0 && prev != device) cudaSetDevice(prev);
  if (e != cudaSuccess) {
    free_net(n); delete n;
    return pfail(e == cudaErrorMemoryAllocation ? BD_ENOMEM : BD_ECUDA, "bd_ppo_net_create: %s", cudaGetErrorString(e));
  }
  *out = n;
  return BD_OK;
}

void bd_ppo_net_destroy(bd_ppo_net* n) {
  if (!n) return;
  free_net(n);
  delete n;
}

/* Diagnostics: CTA 0 of the following forward / sample launches writes SM-clock stamps of its pipeline phases,
 * [tile pair][64] int64 (0..31: epilogue thread 0, 32..63: MMA thread; see mlp_fwd2_kernel); NULL switches it off. */
int bd_ppo_set_trace(bd_ppo_net* n, long long* trace_dev) {
  if (!n) return pfail(BD_EINVAL, "bd_ppo_set_trace: null net");
  n->trace = trace_dev;
  return BD_OK;
}
int64_t bd_ppo_net_param_count(const bd_ppo_net* n) { return n ? n->s.count() : 0; }
int64_t bd_ppo_launch_count(const bd_ppo_net* n) { return n ? n->launches : 0; }
double* bd_ppo_net_stats(bd_ppo_net* n) { return n ? n->stats : nullptr; }

/* fp32 master weights (flat, torch parameter order) -> bf16 slabs.  Stream ordered. */
static int pack_impl(bd_ppo_net* n, const float* flat_params_dev, void* stream, const AdamArgs* adam) {
  if (!n || !flat_params_dev) return pfail(BD_EINVAL, "bd_ppo_net_pack: null argument");
  PackArgs a;
  memset(&a, 0, sizeof(a));
  if (adam != nullptr) a.adam = *adam;
  a.s = n->s; a.param = flat_params_dev;
  a.w1_slabs = n->w1_slabs; a.w2f_slabs = n->w2f_slabs; a.w2b_slabs = n->w2b_slabs; a.w3f = n->w3f; a.w3b_slab = n->w3b_slab;
  a.b1 = n->b1; a.b2 = n->b2; a.b3 = n->b3; a.logstd = n->logstd;
  const long long t = pack_threads(n->s);
  pack_kernel<<<(unsigned)((t + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  n->launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_net_pack: %s", cudaGetErrorString(e));
  return BD_OK;
}
int bd_ppo_net_pack(bd_ppo_net* n, const float* flat_params_dev, void* stream) { return pack_impl(n, flat_params_dev, stream, nullptr); }

namespace {
// forward-only launches: mlp_fwd2_kernel, two tiles in flight per CTA
int launch_fwd2(bd_ppo_net* n, Fwd2Args& a, void* stream, const char* who) {
  a.net = net_dev(n);
  const long long tiles = (a.rows + kRows - 1) / kRows;
  // one CTA per SM, every CTA an even number of tiles where possible (a CTA works on pairs)
  long long grid = tiles < n->sm_count ? tiles : n->sm_count;
  if (tiles < 2LL * n->sm_count) grid = (tiles + 1) / 2;
  if (grid < 1) grid = 1;
  a.stages = fwd2_stages(n->s.K1p);
  a.trace = n->trace;
  mlp_fwd2_kernel<<<(unsigned)grid, kThreads, fwd2_kernel_smem(n->s.K1p, a.stages), (cudaStream_t)stream>>>(a);
  n->launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "%s: %s", who, cudaGetErrorString(e));
  return BD_OK;
}
}  // namespace

/* Forward only: out (rows, out_dim) = MLP(rows of obs).  rows_per_sample: M for the actor (row = (sample, agent)),
 * 1 for the critic (row = sample, input = the M agents' observations).  idx may be NULL (identity). */
int bd_ppo_forward(bd_ppo_net* n, const float* obs_dev, int n_envs, int n_agents, const int64_t* idx_dev, int64_t rows,
                   const float* nmean_dev, const float* nrstd_dev, float nclip, float* out_dev, void* stream) {
  if (!n || !obs_dev || !out_dev) return pfail(BD_EINVAL, "bd_ppo_forward: null argument");
  if (rows <= 0) return BD_OK;
  Fwd2Args f;
  memset(&f, 0, sizeof(f));
  f.sample = 0;
  f.obs = obs_dev; f.N = n_envs; f.M = n_agents; f.idx = (const long long*)idx_dev; f.rows = rows;
  f.rows_per_sample = n->s.C > 1 ? 1 : n_agents;
  f.nmean = nmean_dev; f.nrstd = nrstd_dev; f.nclip = nclip;
  f.out = out_dev;
  return launch_fwd2(n, f, stream, "bd_ppo_forward");
}

/* Rollout-time policy step of an actor net (`MAPPOActorCritic.step`, agent.py:389-415), one launch: mean = MLP(row),
 * act = mean + exp(logstd) eps, logp = sum_k log N(act_k; mean_k, exp(logstd_k)).  obs_dev (n_envs, n_agents, D) = ONE slot,
 * rows = n_envs * n_agents; nmean / nrstd: that slot's (n_agents * D) statistics or NULL.  eps = noise_dev (rows, out_dim)
 * standard normals, or NULL: Philox4x32-10(seed; row, offset) + Box-Muller. */
int bd_ppo_sample(bd_ppo_net* n, const float* obs_dev, int n_envs, int n_agents, const float* nmean_dev, const float* nrstd_dev,
                  float nclip, const float* noise_dev, uint64_t seed, uint64_t offset, float* act_dev, float* logp_dev,
                  float* mean_dev, void* stream) {
  if (!n || !obs_dev || !act_dev || !logp_dev) return pfail(BD_EINVAL, "bd_ppo_sample: null argument");
  if (n->s.C != 1 || !n->s.has_logstd) return pfail(BD_EINVAL, "bd_ppo_sample: needs an actor net (1 input chunk, logstd)");
  const long long rows = (long long)n_envs * n_agents;
  if (rows <= 0) return BD_OK;
  Fwd2Args f;
  memset(&f, 0, sizeof(f));
  f.sample = 1;
  f.obs = obs_dev; f.N = n_envs; f.M = n_agents; f.idx = nullptr; f.rows = rows; f.rows_per_sample = n_agents;
  f.nmean = nmean_dev; f.nrstd = nrstd_dev; f.nclip = nclip;
  f.out = act_dev; f.logp = logp_dev; f.mean_out = mean_dev; f.noise = noise_dev; f.seed = seed; f.offset = offset;
  return launch_fwd2(n, f, stream, "bd_ppo_sample");
}

/* One minibatch: forward, loss, backward (tile kernel), weight gradients (dw kernel), reduction of the per-CTA partials
 * into grad_dev (flat, torch parameter order, mean over rows_global rows — pass the minibatch rows of ALL ranks so that
 * a following all-reduce SUM gives the global mean; 0 = this call's rows).  Statistics of the call are left in
 * bd_ppo_net_stats: [0] sum of per-row losses, [1] sum of (logp_old - logp), [2] rows; run_acc_dev (optional, 4 doubles)
 * accumulates per-minibatch means: [0] += loss, [1] += approx_kl, [2] += 1, [3] += entropy loss. */
int bd_ppo_grad(bd_ppo_net* n, int critic, const float* obs_dev, int n_envs, int n_agents, const int64_t* idx_dev,
                int64_t samples, const float* act_dev, const float* logp_old_dev, const float* adv_dev,
                const float* adv_stats_dev, const float* ret_dev, const float* v_old_dev, float clip, int use_clipped_value,
                float entropy_coef, const float* nmean_dev, const float* nrstd_dev, float nclip, int64_t rows_global,
                float* grad_dev, double* run_acc_dev, void* stream) {
  if (!n || !obs_dev || !grad_dev) return pfail(BD_EINVAL, "bd_ppo_grad: null argument");
  if (!critic && (!act_dev || !logp_old_dev || !adv_dev || !adv_stats_dev)) return pfail(BD_EINVAL, "bd_ppo_grad: actor inputs missing");
  if (critic && !ret_dev) return pfail(BD_EINVAL, "bd_ppo_grad: critic inputs missing");
  const long long rows = critic ? samples : samples * n_agents;
  if (rows < 1 || rows > n->max_rows) return pfail(BD_EINVAL, "bd_ppo_grad: rows %lld outside [1,%lld]", rows, n->max_rows);
  if ((critic ? n_agents : 1) != n->s.C) return pfail(BD_EINVAL, "bd_ppo_grad: net has %d input chunks", n->s.C);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(n->stats, 0, kStatSlots * sizeof(double), st);
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_grad: %s", cudaGetErrorString(e));
  TileArgs a;
  memset(&a, 0, sizeof(a));
  a.net = net_dev(n);
  a.mode = critic ? MODE_CRITIC_TRAIN : MODE_ACTOR_TRAIN;
  a.obs = obs_dev; a.N = n_envs; a.M = n_agents; a.idx = (const long long*)idx_dev; a.rows = rows;
  a.act = act_dev; a.logp_old = logp_old_dev; a.adv = adv_dev; a.adv_stats = adv_stats_dev;
  a.ret = ret_dev; a.v_old = v_old_dev; a.clip = clip; a.use_clipped_value = use_clipped_value ? 1.f : 0.f;
  a.nmean = nmean_dev; a.nrstd = nrstd_dev; a.nclip = nclip;
  a.Xt = n->Xt; a.H1t = n->H1t; a.H2t = n->H2t; a.dZ2t = n->dZ2t; a.dZ1t = n->dZ1t; a.dZ3t = n->dZ3t;
  a.stats = n->stats;
  const long long tiles = (rows + kRows - 1) / kRows;
  const int grid = (int)(tiles < n->sm_count ? tiles : n->sm_count);
  a.stages = tile_stages(n->s.C, n->s.K1p);
  a.trace = n->trace;
  mlp_tile_kernel<<<grid, kThreads, tile_kernel_smem(n->s.C, n->s.K1p, a.stages), st>>>(a);
  e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_grad (tile kernel): %s", cudaGetErrorString(e));
  // ---- weight gradients
  DwArgs d;
  memset(&d, 0, sizeof(d));
  d.tiles = tiles;
  const int C = n->s.C, K1p = n->s.K1p;
  const int per_job = chunks_per_job(K1p);
  int cta = 0, nj = 0;
  for (int jb = 0; jb < n->n1_jobs; ++jb) {          // role 1: A = dZ1 (or H2 for dW3), B = X chunks
    DwJob& J = d.jobs[nj++];
    J.A = n->dZ1t;
    J.n_b = 0;
    for (int c = jb * per_job; c < C && c < (jb + 1) * per_job; ++c) {
      J.B[J.n_b] = n->Xt + (size_t)c * kRows * K1p;
      J.b_stride[J.n_b] = (long long)C * kRows * K1p * 2;
      J.nB[J.n_b] = K1p;
      J.out[J.n_b] = n->pw1 + (size_t)c * n->n1 * HID * K1p;
      J.n_b++;
    }
    J.bias_out = jb == 0 ? n->pb1 : nullptr;
    J.cta0 = cta; J.n_cta = n->n1; cta += n->n1;
  }
  {                                                   // role 2: dW2 = dZ2^T H1 (+ db2), all 512 TMEM columns
    DwJob& J = d.jobs[nj++];
    J.A = n->dZ2t; J.n_b = 1; J.B[0] = n->H1t; J.b_stride[0] = (long long)kRows * HID * 2; J.nB[0] = HID; J.out[0] = n->pw2;
    J.bias_out = n->pb2; J.cta0 = cta; J.n_cta = n->n2; cta += n->n2;
  }
  d.n_jobs = nj;
  dw_kernel<<<cta, kDwThreads, kDwStages * kDwStageBytes, st>>>(d);
  e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_grad (dw kernel): %s", cudaGetErrorString(e));
  // dW3^T = H2^T dZ3: a second, small launch of the same kernel (A = H2) on every SM
  DwArgs d3;
  memset(&d3, 0, sizeof(d3));
  d3.tiles = tiles; d3.n_jobs = 1;
  {
    DwJob& J = d3.jobs[0];
    J.A = n->H2t; J.n_b = 1; J.B[0] = n->dZ3t; J.b_stride[0] = (long long)kRows * kNOut * 2; J.nB[0] = kNOut; J.out[0] = n->pw3;
    J.bias_out = nullptr; J.cta0 = 0; J.n_cta = n->n3;
  }
  dw_kernel<<<n->n3, kDwThreads, kDwStages * kDwStageBytes, st>>>(d3);
  e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_grad (dw3 kernel): %s", cudaGetErrorString(e));
  // ---- flat gradient
  ReduceArgs r;
  memset(&r, 0, sizeof(r));
  r.s = n->s;
  for (int c = 0; c < C; ++c) r.pw1[c] = n->pw1 + (size_t)c * n->n1 * HID * K1p;
  r.pw2 = n->pw2; r.pw3 = n->pw3; r.pb1 = n->pb1; r.pb2 = n->pb2; r.n1 = n->n1; r.n2 = n->n2; r.n3 = n->n3;
  r.stats = n->stats; r.entropy_coef = critic ? 0.f : entropy_coef; r.rows_global = rows_global; r.grad = grad_dev;
  r.run_acc = run_acc_dev; r.logstd = n->logstd;
  const long long np = n->s.count();
  reduce_kernel<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(r);
  e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_grad (reduce kernel): %s", cudaGetErrorString(e));
  n->launches += 4;
  return BD_OK;
}

/* torch.optim.Adam's step on flat fp32 buffers with the reference's KL gate evaluated on the device, then the bf16
 * repack of the network for the next minibatch.  kl_sum_dev / kl_rows_dev: device doubles (e.g. stats + 1, stats + 10,
 * or their cross-rank sums); NULL or target_kl <= 0: unconditional step.  step_dev: device double (step count). */
int bd_ppo_adam_step(bd_ppo_net* n, float* param_dev, float* exp_avg_dev, float* exp_avg_sq_dev, const float* grad_dev,
                     double* step_dev, float lr, float beta1, float beta2, float eps, const double* kl_sum_dev,
                     const double* kl_rows_dev, float target_kl, double* gate_count_dev, void* stream) {
  if (!n || !param_dev || !exp_avg_dev || !exp_avg_sq_dev || !grad_dev || !step_dev) return pfail(BD_EINVAL, "bd_ppo_adam_step: null argument");
  AdamArgs a;
  a.param = param_dev; a.m = exp_avg_dev; a.v = exp_avg_sq_dev; a.grad = grad_dev; a.step = step_dev; a.n = n->s.count();
  a.lr = lr; a.b1 = beta1; a.b2 = beta2; a.eps = eps; a.kl_sum = kl_sum_dev; a.kl_rows = kl_rows_dev; a.target_kl = target_kl;
  a.gate_out = gate_count_dev;
  cudaStream_t st = (cudaStream_t)stream;
  adam_kernel<<<(unsigned)((a.n + 255) / 256), 256, 0, st>>>(a);
  n->launches += 1;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_adam_step: %s", cudaGetErrorString(e));
  return pack_impl(n, param_dev, stream, &a);     // repack + advance the step count
}

/* Returns and advantages of a whole rollout in one launch (mappo/buffer.py:561-614), plus the buffer-wide advantage
 * moments: acc3_dev += (sum adv, sum adv^2, count).  rew (T,N) float, term / trunc (T,N) uint8, vals (T+1,N). */
int bd_ppo_gae(const float* rew_dev, const uint8_t* term_dev, const uint8_t* trunc_dev, const float* vals_dev, int T, int N,
               float gamma, float lam, int use_gae, float* ret_dev, float* adv_dev, double* acc3_dev, void* stream) {
  if (!rew_dev || !term_dev || !trunc_dev || !vals_dev || !ret_dev || !adv_dev || !acc3_dev) return pfail(BD_EINVAL, "bd_ppo_gae: null argument");
  if (T < 1 || N < 1) return pfail(BD_EINVAL, "bd_ppo_gae: T and N must be positive");
  gae_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rew_dev, term_dev, trunc_dev, vals_dev, T, N, gamma, lam, use_gae,
                                                                ret_dev, adv_dev, acc3_dev);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_gae: %s", cudaGetErrorString(e));
  return BD_OK;
}
/* (sum, sum of squares, count) -> stats2_dev = (mean, 1 / (std + 1e-8)) per normalize_advantages (buffer.py:666-695). */
int bd_ppo_adv_stats(const double* acc3_dev, float* stats2_dev, void* stream) {
  if (!acc3_dev || !stats2_dev) return pfail(BD_EINVAL, "bd_ppo_adv_stats: null argument");
  adv_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(acc3_dev, stats2_dev);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(BD_ECUDA, "bd_ppo_adv_stats: %s", cudaGetErrorString(e));
  return BD_OK;
}

}  // extern "C"
