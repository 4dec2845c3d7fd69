// Memory skeleton of one control step (no arithmetic): which structure moves the step's
// bytes fastest?  read 4 state planes + action + 14 history planes; write 4 state planes,
// one ring slot and complete 288-B observation rows.
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o step_skeleton step_skeleton.cu
// ./step_skeleton [n]            structure sweep at n drones (default 262 144)
// ./step_skeleton l2 n1 n2 ...   L2 eviction-policy sweep at each size (see residency_sweep)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1);} } while (0)
constexpr int B = 15, NS = 14, D = 72;

struct Bufs { float4 *s0, *s1, *s2, *s3, *hist; const float4* act; float* obs; size_t n; int head; };

__device__ __forceinline__ void bulk_store(void* g, const void* s, unsigned bytes) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(s);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(g), "r"(sa), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}

// ROWS per CTA = blockDim; persistent loop over tiles; MODE 0: cooperative STG, 1: TMA bulk store
template <int ROWS, int MODE>
__global__ void __launch_bounds__(ROWS) k_skel(Bufs b, int ntiles) {
  extern __shared__ __align__(128) float tile[];   // [ROWS][D]
  const int tid = threadIdx.x;
  for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const size_t g = (size_t)t * ROWS + tid;
    float4 a0 = b.s0[g], a1 = b.s1[g], a2 = b.s2[g], a3 = b.s3[g], ac = b.act[g];
    float4 v[NS];
    int slot = b.head;
#pragma unroll
    for (int k = 0; k < NS; ++k) { slot = (slot + 1 == B) ? 0 : slot + 1; v[k] = b.hist[(size_t)slot * b.n + g]; }
    if (MODE == 1) { if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
    __syncthreads();
    float4* row = reinterpret_cast<float4*>(tile + (size_t)tid * D);
    row[0] = a0; row[1] = a1; row[2] = a2;
#pragma unroll
    for (int k = 0; k < NS; ++k) row[3 + k] = v[k];
    row[17] = ac;
    b.hist[(size_t)b.head * b.n + g] = ac;
    a0.x += 1.f; a1.x += 1.f; a2.x += 1.f; a3.x += 1.f;
    b.s0[g] = a0; b.s1[g] = a1; b.s2[g] = a2; b.s3[g] = a3;
    float* gob = b.obs + (size_t)t * ROWS * D;
    if (MODE == 0) {
      __syncthreads();
      const float4* s4 = reinterpret_cast<const float4*>(tile);
      float4* g4 = reinterpret_cast<float4*>(gob);
      for (int i = tid; i < ROWS * D / 4; i += ROWS) g4[i] = s4[i];
    } else {
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
      __syncthreads();
      if (tid == 0) bulk_store(gob, tile, ROWS * D * 4);
    }
  }
  if (MODE == 1 && tid == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
}

// ---- L2 residency sweep (`step_skeleton l2 [n ...]`) -------------------------------------------------------------
// The fast step kernel's shape: one CTA per 128-row tile (a different SM every launch), ring planes by cp.async
// straight into the row, state / action by 128-bit loads, whole rows out as one evict-first TMA bulk store.  Many
// back-to-back steps run on the same state and ring planes while actions and observation rows rotate through pools
// larger than the L2.  Policy (keep_state, keep_k): state loads / stores evict_last when keep_state; a ring slot of
// age a (0 = the slot written this step, read again at ages 1..14) evict_last when a < keep_k, evict_first otherwise
// (evict_normal for both when the policy is off); actions evict_first.
__device__ __forceinline__ uint64_t pol_last() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t pol_first() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t pol_normal() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;\n" : "=l"(p)); return p; }
__device__ __forceinline__ float4 ld_pol(const float4* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ void st_pol(float4* p, float4 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;\n" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__global__ void __launch_bounds__(128, 6) k_res(Bufs b, int keep_state, int keep_k) {
  extern __shared__ __align__(128) float tile[];   // [128][D]
  const int tid = threadIdx.x;
  const size_t g = (size_t)blockIdx.x * 128 + tid;
  const bool on = keep_state || keep_k > 0;
  const uint64_t last = pol_last(), drop = on ? pol_first() : pol_normal();
  const uint64_t ps = keep_state ? last : pol_normal();
  float* row = tile + (size_t)tid * D;
  int slot = b.head;
#pragma unroll
  for (int j = 0; j < NS; ++j) {   // entry j = slot head+1+j, age NS - j
    slot = (slot + 1 == B) ? 0 : slot + 1;
    const unsigned d = (unsigned)__cvta_generic_to_shared(row + 12 + 4 * j);
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;\n" ::"r"(d), "l"(b.hist + (size_t)slot * b.n + g),
                 "l"(NS - j < keep_k ? last : drop) : "memory");
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  float4 a0 = ld_pol(b.s0 + g, ps), a1 = ld_pol(b.s1 + g, ps), a2 = ld_pol(b.s2 + g, ps), a3 = ld_pol(b.s3 + g, ps);
  const float4 ac = ld_pol(b.act + g, pol_first());
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  float4* r4 = reinterpret_cast<float4*>(row);
  r4[0] = a0; r4[1] = a1; r4[2] = a2; r4[17] = ac;
  st_pol(b.hist + (size_t)b.head * b.n + g, ac, keep_k > 0 ? last : drop);
  a0.x += 1.f; a1.x += 1.f; a2.x += 1.f; a3.x += 1.f;
  st_pol(b.s0 + g, a0, ps); st_pol(b.s1 + g, a1, ps); st_pol(b.s2 + g, a2, ps); st_pol(b.s3 + g, a3, ps);
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  __syncthreads();
  if (tid == 0) {
    bulk_store(b.obs + (size_t)blockIdx.x * 128 * D, tile, 128 * D * 4);
    asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
  }
}

static int residency_sweep(int argc, char** argv) {
  int dev = 0, l2 = 0, pmax = 0;
  size_t plim = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev));
  CK(cudaDeviceGetAttribute(&pmax, cudaDevAttrMaxPersistingL2CacheSize, dev));
  CK(cudaDeviceGetLimit(&plim, cudaLimitPersistingL2CacheSize));
  cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, dev));
  printf("# %s  L2 %d B  persisting max %d B  persisting limit %zu B\n", prop.name, l2, pmax, plim);
  const int pol[][2] = {{0, 0}, {1, 0}, {1, 1}, {1, 2}, {1, 4}, {1, 7}, {1, 14}};
  const int npol = sizeof(pol) / sizeof(pol[0]), reps = 3, warm = 60, iters = 300;
  CK(cudaFuncSetAttribute(k_res, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * D * 4));
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  for (int a = 2; a < argc; ++a) {
    const size_t n = (size_t)atoll(argv[a]) / 128 * 128;
    // pools: actions and observation rows rotate through more than 2 x L2, so they never hit
    const int act_slots = (int)((2 * (size_t)l2) / (n * 16) + 2), obs_slots = (int)((2 * (size_t)l2) / (n * D * 4) + 2);
    Bufs b; b.n = n;
    float4* act;
    float* obs;
    CK(cudaMalloc(&b.s0, n * 16)); CK(cudaMalloc(&b.s1, n * 16)); CK(cudaMalloc(&b.s2, n * 16)); CK(cudaMalloc(&b.s3, n * 16));
    CK(cudaMalloc(&b.hist, (size_t)B * n * 16)); CK(cudaMalloc(&act, (size_t)act_slots * n * 16));
    CK(cudaMalloc(&obs, (size_t)obs_slots * n * D * 4));
    CK(cudaMemset(b.s0, 0, n * 16)); CK(cudaMemset(b.s1, 0, n * 16)); CK(cudaMemset(b.s2, 0, n * 16)); CK(cudaMemset(b.s3, 0, n * 16));
    CK(cudaMemset(b.hist, 0, (size_t)B * n * 16)); CK(cudaMemset(act, 0, (size_t)act_slots * n * 16));
    const double alg = (double)n * 675.0;   // algorithmic bytes per drone (ISSUE table: state, ring, action, row, counters)
    double us[16][8];
    int step = 0;
    for (int r = 0; r < reps; ++r) {
      for (int p = 0; p < npol; ++p) {
        auto launch = [&]() {
          b.head = step % B;
          b.act = act + (size_t)(step % act_slots) * n;
          b.obs = obs + (size_t)(step % obs_slots) * n * D;
          k_res<<<(unsigned)(n / 128), 128, 128 * D * 4>>>(b, pol[p][0], pol[p][1]);
          ++step;
        };
        for (int i = 0; i < warm; ++i) launch();
        CK(cudaEventRecord(e0));
        for (int i = 0; i < iters; ++i) launch();
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1)); CK(cudaGetLastError());
        float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
        us[p][r] = ms * 1e3 / iters;
      }
    }
    for (int p = 0; p < npol; ++p) {
      double v[8];
      for (int r = 0; r < reps; ++r) v[r] = us[p][r];
      for (int i = 0; i < reps; ++i) for (int j = i + 1; j < reps; ++j) if (v[j] < v[i]) { double t = v[i]; v[i] = v[j]; v[j] = t; }
      const double kept = (pol[p][0] ? 64.0 : 0.0) * n + 16.0 * pol[p][1] * n;
      printf("n %8zu  state %d  k %2d  evict_last %6.1f MB  median %8.2f us  [%7.2f .. %7.2f]  %7.1f GB/s algorithmic\n", n, pol[p][0],
             pol[p][1], kept / 1e6, v[reps / 2], v[0], v[reps - 1], alg / (v[reps / 2] * 1e-6) / 1e9);
    }
    CK(cudaFree(b.s0)); CK(cudaFree(b.s1)); CK(cudaFree(b.s2)); CK(cudaFree(b.s3)); CK(cudaFree(b.hist)); CK(cudaFree(act)); CK(cudaFree(obs));
  }
  return 0;
}

int main(int argc, char** argv) {
  if (argc > 1 && argv[1][0] == 'l') return residency_sweep(argc, argv);
  const size_t n = argc > 1 ? atoll(argv[1]) : 262144;
  const int slots = 8, iters = 100;
  Bufs b; b.n = n;
  float4* act;
  CK(cudaMalloc(&b.s0, n * 16)); CK(cudaMalloc(&b.s1, n * 16)); CK(cudaMalloc(&b.s2, n * 16)); CK(cudaMalloc(&b.s3, n * 16));
  CK(cudaMalloc(&b.hist, (size_t)B * n * 16)); CK(cudaMalloc(&act, (size_t)slots * n * 16));
  CK(cudaMalloc(&b.obs, (size_t)slots * n * D * 4));
  CK(cudaMemset(b.s0, 0, n * 16)); CK(cudaMemset(b.s1, 0, n * 16)); CK(cudaMemset(b.s2, 0, n * 16)); CK(cudaMemset(b.s3, 0, n * 16));
  CK(cudaMemset(b.hist, 0, (size_t)B * n * 16)); CK(cudaMemset(act, 0, (size_t)slots * n * 16));
  float* obs0 = b.obs;
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  const double alg = (double)n * 647.5, act_bytes = (double)n * (304 + 368);
  auto run = [&](const char* name, auto&& launch) {
    for (int i = 0; i < 10; ++i) launch(i);
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(e0));
    for (int i = 0; i < iters; ++i) launch(i);
    CK(cudaEventRecord(e1));
    CK(cudaDeviceSynchronize()); CK(cudaGetLastError());
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    const double t = ms * 1e-3 / iters;
    printf("%-46s %8.2f us  algorithmic %7.1f GB/s (frac of 6553: %.3f)  actual %7.1f GB/s\n", name, t * 1e6, alg / t / 1e9, alg / t / 6553e9, act_bytes / t / 1e9);
  };
  auto prep = [&](int i) { b.head = i % B; b.act = act + (size_t)(i % slots) * n; b.obs = obs0 + (size_t)(i % slots) * n * D; };
#define RUN(ROWS, MODE, GRID, label) { CK(cudaFuncSetAttribute(k_skel<ROWS, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, ROWS * D * 4)); \
    run(label, [&](int i) { prep(i); k_skel<ROWS, MODE><<<GRID, ROWS, ROWS * D * 4>>>(b, (int)(n / ROWS)); }); }
  RUN(128, 0, (int)(n / 128), "128 rows/CTA, STG, one CTA per tile");
  RUN(128, 0, 148 * 6, "128 rows/CTA, STG, persistent 148x6");
  RUN(128, 1, (int)(n / 128), "128 rows/CTA, TMA store, one CTA per tile");
  RUN(128, 1, 148 * 6, "128 rows/CTA, TMA store, persistent 148x6");
  RUN(64, 1, 148 * 12, "64 rows/CTA, TMA store, persistent 148x12");
  RUN(32, 1, 148 * 24, "32 rows/CTA, TMA store, persistent 148x24");
  RUN(32, 1, (int)(n / 32), "32 rows/CTA, TMA store, one CTA per tile");
  RUN(256, 1, 148 * 3, "256 rows/CTA, TMA store, persistent 148x3");
  RUN(256, 0, 148 * 3, "256 rows/CTA, STG, persistent 148x3");
  return 0;
}
