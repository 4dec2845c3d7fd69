// Fast step kernel (float, DYN with optional ground effect / drag / downwash, M <= 32): one CTA per tile of up to 128 drones
// (a warp holds 32 / M whole envs on consecutive lanes).
//
// Measured facts that shape it (scripts/microbench/*.cu, profiles/README.md):
//   * observation rows must leave the SM as complete, contiguous rows: 16-byte or
//     partial-sector row pieces write at 1.6-1.9 TB/s, whole rows at 5-6 TB/s;
//   * the memory skeleton of a step (read 4 state planes + action + 14 ring planes, write
//     state, one ring slot and whole rows) runs at 0.85-0.96 of the measured HBM peak with
//     exactly this shape — 128 rows per CTA, every load issued before anything is consumed,
//     a row-major shared-memory tile — and slower with 32-row tiles or persistent CTAs;
//   * shared memory, not registers, bounds occupancy: the 128 x D tile must be the ONLY
//     shared memory of the CTA for 6 CTAs (24 warps) to fit on an SM.
//
// Per CTA: (1) 4 state planes, action and step counter with 128-bit coalesced loads, then
// the B-1 ring planes with cp.async (no registers) straight into the thread's own row of
// the tile; (2) S substeps in registers while the history lands; (3) kinematic part, task
// terms and the new action complete the row; per-env reward / termination reductions and
// the MultiHover re-spawn rule use warp shuffles (envs are lane groups, M | 32), so there
// is no reduction scratch; (4) one __syncthreads, then the 128 finished rows (36 864 B for
// D = 72) leave as ONE TMA bulk store issued by thread 0; state planes and the ring slot
// are 128-bit stores.  Every global access carries an L2 eviction priority (L2Hints): what
// the tile reads again next step is kept in L2 as far as the handle's budget allows.
// Dependency on the previous control step (0): per tile, not per grid.  A CTA waits (ld.acquire) for the
// epoch its own tile's previous CTA published (st.release) instead of griddepcontrol.wait, so back-to-back
// launches overlap tile by tile; a per-launch decision (bd_device.cuh: pipe_gate) falls back to the
// grid-wide wait when a foreign kernel ran between two steps.  DESIGN.md section 4 has the protocol.
// The global step count (ring head, Philox stream id) is a host-tracked parameter; a device-resident copy
// (advanced by tile 0's CTA, or by the last CTA out under CUDA-graph replay) keeps the launch replayable.
// Tasks: Hover, MultiHover, Spiral, and the swarm tasks (Meetup / Flock / LeaderFollower) through warp-shuffle
// exchange inside the env's lane group (swarm_reward_shfl).
#pragma once
#include "bd_device.cuh"

namespace bd {

template <int A>
struct TileIn {
  float4 s0, s1, s2, s3;
  float4 act;   // A == 1: only .x is used
  int stepc;
  float ep_ret;
};

// the handle's own data (written by the previous step of this tile) ...   HINT: with the L2 policies of L2Hints
template <int A, bool HINT = false>
__device__ __forceinline__ void load_state(const Params<float>& P, long long g, int env, bool active, TileIn<A>& in,
                                           const L2Hints& h = L2Hints{}) {
  if (active) {
    if constexpr (HINT) {
      in.s0 = ld_hint(P.s0 + g, h.state); in.s1 = ld_hint(P.s1 + g, h.state);
      in.s2 = ld_hint(P.s2 + g, h.state); in.s3 = ld_hint(P.s3 + g, h.state);
      in.stepc = ld_hint(P.stepc + env, h.state);
      in.ep_ret = P.ep_ret != nullptr ? ld_hint(P.ep_ret + env, h.state) : 0.f;
    } else {
      in.s0 = P.s0[g]; in.s1 = P.s1[g]; in.s2 = P.s2[g]; in.s3 = P.s3[g];
      in.stepc = P.stepc[env];
      in.ep_ret = P.ep_ret != nullptr ? P.ep_ret[env] : 0.f;
    }
  } else {
    in.s0 = in.s1 = in.s2 = in.s3 = make_float4(0.f, 0.f, 0.f, 0.f);
    in.s1.z = 1.0f;
    in.stepc = 0;
    in.ep_ret = 0.f;
  }
}
// ... and the caller's (possibly written by the kernel enqueued just before this launch)
template <int A, bool HINT = false>
__device__ __forceinline__ void load_action(const Params<float>& P, long long g, bool active, TileIn<A>& in,
                                            const L2Hints& h = L2Hints{}) {
  if (active) {
    if constexpr (HINT) {
      if constexpr (A == 4) in.act = ld_hint(reinterpret_cast<const float4*>(P.actions) + g, h.once);
      else in.act = make_float4(ld_hint(reinterpret_cast<const float*>(P.actions) + g, h.once), 0.f, 0.f, 0.f);
    } else {
      if constexpr (A == 4) in.act = reinterpret_cast<const float4*>(P.actions)[g];
      else in.act = make_float4(reinterpret_cast<const float*>(P.actions)[g], 0.f, 0.f, 0.f);
    }
  } else {
    in.act = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// Swarm tasks (Meetup / Flock / LeaderFollower, bd_device.cuh: swarm_terms / swarm_reward) on the fast kernel: the env's
// drones are a lane group of M, so partners' final positions / velocities arrive by warp shuffle and the env-level
// sums by xor butterflies.  Executed by every lane of the warp (inactive lanes carry zeros); returns the env's
// reward, sets this drone's flag bits (bit1: truncation bound, bit2: my pair has not met).
__device__ __forceinline__ float swarm_reward_shfl(const Params<float>& P, const Drone<float>& d, float roll, float pitch,
                                                   int lane, int M, int drone, int& flags) {
  const unsigned full = 0xffffffffu;
  const int base = lane & ~(M - 1);
  const bool tilt = fabsf(roll) > .4f || fabsf(pitch) > .4f;
  flags = 0;
  float contrib = 0.f;
  if (P.task == TASK_MEETUP) {
    const int src = base | (M - 1 - drone);
    const float ox = __shfl_sync(full, d.px, src), oy = __shfl_sync(full, d.py, src), oz = __shfl_sync(full, d.pz, src);
    if (drone < M / 2) {                                                         // MeetupAviary.py:88-93
      const float dx = d.px - ox, dy = d.py - oy, dz = d.pz - oz;
      const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
      contrib = (-1.f * (dist * dist)) * 2.f;
      if (dist > 0.1f) flags |= 4;                                               // :115-118
    }
    if (fabsf(d.px) > 5.0f || fabsf(d.py) > 5.0f || d.pz > 3.0f || d.pz < 0.1f || tilt) flags |= 2;   // :142-147
  } else if (P.task == TASK_LEADERFOLLOWER) {
    const float z0 = __shfl_sync(full, d.pz, base);
    if (drone == 0) {                                                            // LeaderFollowerAviary.py:88
      const float ex = 0.f - d.px, ey = 0.f - d.py, ez = 0.5f - d.pz;
      const float n = sqrtf(ex * ex + ey * ey + ez * ez);
      contrib = -1.f * (n * n);
    } else {                                                                     // :91-97
      const float dz = z0 - d.pz;
      const float n = sqrtf(dz * dz);
      contrib = -(1.f / (float)M) * (n * n);
    }
    if (fabsf(d.px) > 2.0f || fabsf(d.py) > 2.0f || d.pz > 2.0f || tilt) flags |= 2;   // :135-140
  } else {                                                                       // FlockAviary.py:75-150
    const float eps = 1e-3f;
    const float ni = sqrtf(d.vx * d.vx + d.vy * d.vy + d.vz * d.vz);
    float ali = 0.f, sp = 0.f;
#pragma unroll 1
    for (int o = 1; o < M; ++o) {
      const int src = base | ((lane + o) & (M - 1));
      const float ox = __shfl_sync(full, d.px, src), oy = __shfl_sync(full, d.py, src), oz = __shfl_sync(full, d.pz, src);
      const float ux = __shfl_sync(full, d.vx, src), uy = __shfl_sync(full, d.vy, src), uz = __shfl_sync(full, d.vz, src);
      const float nj = __shfl_sync(full, ni, src);
      const float dot = d.vx * ux + d.vy * uy + d.vz * uz;
      ali += dot / (ni + eps) / (nj + eps);                                      // :98-103
      const float dx = ox - d.px, dy = oy - d.py, dz = oz - d.pz;
      const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
      sp = (o == 1 || dist < sp) ? dist : sp;                                    // :121-125 nearest neighbour
    }
    if (fabsf(d.px) > 10.0f || fabsf(d.py) > 10.0f || d.pz > 10.0f || tilt) flags |= 2;   // :181-184
    float cx = d.vx, cy = d.vy, cz = d.vz, ssp = sp;
#pragma unroll 1
    for (int o = M >> 1; o > 0; o >>= 1) {
      ali += __shfl_xor_sync(full, ali, o);
      cx += __shfl_xor_sync(full, cx, o); cy += __shfl_xor_sync(full, cy, o); cz += __shfl_xor_sync(full, cz, o);
      ssp += __shfl_xor_sync(full, ssp, o);
    }
    cx /= (float)M; cy /= (float)M; cz /= (float)M;                              // :111-112
    const float speed = sqrtf(cx * cx + cy * cy + cz * cz);
    if (M == 1) return speed;
    const float avg = ssp / (float)M;
    float var = (sp - avg) * (sp - avg);
#pragma unroll 1
    for (int o = M >> 1; o > 0; o >>= 1) var += __shfl_xor_sync(full, var, o);
    var /= (float)M;                                                             // np.var (:131)
    float pen = 0.f;
    if (!(1.0f < avg && avg < 3.0f)) {                                           // :137-141
      const float a = fabsf(avg - 1.0f), b = fabsf(avg - 3.0f);
      pen = a < b ? a : b;
    }
    return ((ali / (float)(M * (M - 1)) + speed) - pen) - var;                   // :145
  }
#pragma unroll 1
  for (int o = M >> 1; o > 0; o >>= 1) contrib += __shfl_xor_sync(full, contrib, o);
  return contrib;
}

// AERO: 0 plain DYN, 1 downwash only, 2 any aero combination (run-time P.aero) — see fast_substeps.
// Lane packing: a warp holds EW = 32 / M whole envs on its first EW * M lanes (an env = M consecutive lanes), the
// left-over lanes idle: nothing for the power-of-two team sizes, 2 of 32 lanes for M = 3 or 5 (a first version padded
// every env to a power-of-two lane group and left 3 of 8 lanes idle at M = 5).  A tile = 4 EW envs = 4 EW M rows.
template <int TASK, int A, bool VEC, int AERO>
__global__ void __launch_bounds__(kBlock, 6)
step_kernel_tile(const __grid_constant__ Params<float> P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int M = P.M, B = P.B, D = P.D, EW = P.EW;
  const bool pow2 = (M & (M - 1)) == 0;
  constexpr bool vec = VEC;   // A == 4 and D % 4 == 0: 128-bit row accesses
  float* tile_s = reinterpret_cast<float*>(smem_raw);   // [tile rows][D] row-major, dense
  const int env_w = pow2 ? (lane >> (31 - __clz(M))) : lane / M;    // env within the warp
  const int group_base = env_w * M;
  const int drone = lane - group_base;
  const int tile = blockIdx.x + P.block0;               // block0 > 0: sub-range launch (bd_step_host chunks)
  const int env_l = (tid >> 5) * EW + env_w;
  const int env = tile * (4 * EW) + env_l;
  const bool active = env_w < EW && env < P.N;
  const long long g0 = (long long)tile * (4 * EW) * M;
  const long long g = (long long)env * M + drone;       // meaningful for active lanes only
  float* myrow = tile_s + (size_t)(env_w < EW ? env_l * M + drone : 0) * D;   // idle lanes alias a live row, never write
  const bool jit = (TASK == TASK_MULTIHOVER) && (P.reset_mode != RESET_FIXED);
  const long long gh = active ? g : P.n_total;          // idle lanes issue no history copies
  const L2Hints l2 = l2_hints(P);

  // ---- 1. every load of the tile is issued before anything is consumed ------------------------
  // Programmatic dependent launch: this grid may become resident while the previous kernel of
  // the stream is still in its last wave.  Before griddepcontrol.wait only data that no earlier
  // kernel can be writing is touched: the ring planes except the one the previous step wrote
  // (its slot `head-1`, time index B-2).  68 % of the step's reads are in flight before the
  // previous kernel has even finished.
  pdl_launch_dependents();
  int total, head;
  const bool pipe = P.pipe_wait && P.host_total >= 0;   // wait on my tile's epoch instead of the whole previous grid
  if (pipe) {
    // Tile-level step pipelining: everything this CTA reads that an earlier launch wrote belongs to ITS tile
    // (whole environments), and was written by the CTA that stepped this tile in the previous control step.
    // So instead of griddepcontrol.wait (the whole previous grid finished and flushed) the CTA waits for its own
    // tile's epoch: launches overlap tile by tile, no lock-step start, no idle tail.  (All CTAs of the previous
    // launch are resident or done before any CTA of this one starts, so the spin cannot deadlock.)  pipe_gate
    // also decides, once per launch, whether the grid-wide wait is needed after all (a foreign kernel, e.g. the
    // one that produced the actions, ran between the two steps).
    total = P.host_total;
    head = P.host_head;
    if (pipe_gate(P, tile, total, tid)) pdl_wait();
    issue_history<float, A, VEC, true>(P, gh, head, myrow, 0, B - 2, l2);
  } else if (P.host_total >= 0 && P.early_prefetch) {
    total = P.host_total;
    head = P.host_head;   // = total % B (ring slot overwritten by this step's action), divided on the host
    issue_history<float, A, VEC, true>(P, gh, head, myrow, 0, B - 2, l2);
    pdl_wait();
  } else {              // CUDA-graph mode (the step count is read from device memory), or a grid smaller than the
    pdl_wait();         // resident capacity (several earlier launches could still be in flight: no early reads)
    total = P.host_total >= 0 ? P.host_total : P.gsteps[0];   // only the last CTA to finish modifies it, after every read
    head = total % B;
    issue_history<float, A, VEC, true>(P, gh, head, myrow, 0, B - 2, l2);
  }
  TileIn<A> cur;
  load_state<A, true>(P, g, env, active, cur, l2);
  issue_history<float, A, VEC, true>(P, gh, head, myrow, B - 2, B - 1, l2);
  cp_async_commit();
  load_action<A, true>(P, g, active, cur, l2);
  const int stepc = cur.stepc;
  // drag reads last_clipped_action during the first substep (BaseAviary.py:359,372): the previous step's action,
  // i.e. ring slot head-1; zero right after a reset (:468)
  float last_sum = 0.f;
  if constexpr (AERO == 2) {
    if ((P.aero & AERO_DRAG) && active && stepc > 0) {
      const int prev = head == 0 ? B - 1 : head - 1;
      const float* lp = P.hist + ((size_t)prev * P.n_total + g) * A;
      if constexpr (A == 4) {
        const float4 pa = *reinterpret_cast<const float4*>(lp);
        last_sum = (__fadd_rn(1.0f, __fmul_rn(0.05f, pa.x)) + __fadd_rn(1.0f, __fmul_rn(0.05f, pa.y))) +
                   (__fadd_rn(1.0f, __fmul_rn(0.05f, pa.z)) + __fadd_rn(1.0f, __fmul_rn(0.05f, pa.w)));
      } else {
        last_sum = 4.0f * __fadd_rn(1.0f, __fmul_rn(0.05f, lp[0]));
      }
    }
  }

  Drone<float> d;
  d.px = cur.s0.x; d.py = cur.s0.y; d.pz = cur.s0.z; d.qx = cur.s0.w;
  d.qy = cur.s1.x; d.qz = cur.s1.y; d.qw = cur.s1.z; d.vx = cur.s1.w;
  d.vy = cur.s2.x; d.vz = cur.s2.y; d.wx = cur.s2.z; d.wy = cur.s2.w;
  d.wz = cur.s3.x; d.tx = cur.s3.y; d.ty = cur.s3.z; d.tz = cur.s3.w;
  float onep[4];
  if constexpr (A == 4) {
    // numpy evaluates 1 + 0.05*a in float32 for float32 actions (two roundings, BaseRLAviary.py:192)
    onep[0] = __fadd_rn(1.0f, __fmul_rn(0.05f, cur.act.x));
    onep[1] = __fadd_rn(1.0f, __fmul_rn(0.05f, cur.act.y));
    onep[2] = __fadd_rn(1.0f, __fmul_rn(0.05f, cur.act.z));
    onep[3] = __fadd_rn(1.0f, __fmul_rn(0.05f, cur.act.w));
  } else {
    onep[0] = onep[1] = onep[2] = onep[3] = __fadd_rn(1.0f, __fmul_rn(0.05f, cur.act.x));   // :225
  }

  // ---- 2. S substeps in registers while the history lands --------------------------------------
  float avx = 0.f, avy = 0.f, avz = 0.f;
  fast_substeps<AERO>(P, d, onep, avx, avy, avz, group_base, drone, last_sum);
  float roll, pitch, yaw;
  quat_to_euler_fast(d.qx, d.qy, d.qz, d.qw, roll, pitch, yaw);

  // ---- 3. complete my observation row ------------------------------------------------------------
  cp_async_wait_all();
  float contrib = 0.f;
  int flags = 0;
  if (active) {
    if (vec) {
      float4* r4 = reinterpret_cast<float4*>(myrow);
      r4[0] = make_float4(d.px, d.py, d.pz, roll);
      r4[1] = make_float4(pitch, yaw, d.vx, d.vy);
      r4[2] = make_float4(d.vz, avx, avy, avz);
    } else {
      myrow[0] = d.px; myrow[1] = d.py; myrow[2] = d.pz; myrow[3] = roll; myrow[4] = pitch; myrow[5] = yaw;
      myrow[6] = d.vx; myrow[7] = d.vy; myrow[8] = d.vz; myrow[9] = avx; myrow[10] = avy; myrow[11] = avz;
    }
    if constexpr (TASK != TASK_SWARM)
      task_terms<float, TASK>(P, d, roll, pitch, stepc, drone, myrow + 12 + B * A, contrib, flags);
    // newest history entry: tail of the row and ring slot `head`
    if constexpr (A == 4) {
      if (vec) *reinterpret_cast<float4*>(myrow + 12 + (B - 1) * 4) = cur.act;
      else { float* o = myrow + 12 + (B - 1) * 4; o[0] = cur.act.x; o[1] = cur.act.y; o[2] = cur.act.z; o[3] = cur.act.w; }
      st_hint(reinterpret_cast<float4*>(P.hist + ((size_t)head * P.n_total + g) * 4), cur.act, l2_slot_pol(l2, 0));
    } else {
      myrow[12 + B - 1] = cur.act.x;
      st_hint(P.hist + (size_t)head * P.n_total + g, cur.act.x, l2_slot_pol(l2, 0));
    }
  }

  float swarm_reward_env = 0.f;
  if constexpr (TASK == TASK_SWARM) {
    int fl = 0;
    swarm_reward_env = swarm_reward_shfl(P, d, roll, pitch, lane, M, drone, fl);   // swarm tasks: G == M (host side)
    flags = active ? fl : 0;
  }
  // ---- per-env reduction with shuffles (envs are lane groups of M) --------------------------------
  if (pow2) {
#pragma unroll 1
    for (int o = M >> 1; o > 0; o >>= 1) {
      contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
      flags |= __shfl_xor_sync(0xffffffffu, flags, o);
    }
  } else {        // team sizes that are not a power of two: every lane gathers its M - 1 partners
    const float c0 = contrib;
    const int f0 = flags;
#pragma unroll 1
    for (int o = 1; o < M; ++o) {
      int t = drone + o;
      t -= (t >= M) ? M : 0;
      contrib += __shfl_sync(0xffffffffu, c0, group_base + t);
      flags |= __shfl_sync(0xffffffffu, f0, group_base + t);
    }
  }
  const float reward = (TASK == TASK_SWARM) ? swarm_reward_env : ((TASK == TASK_HOVER) ? contrib : contrib / (float)M);
  const bool time_up = stepc >= P.trunc_counter;   // step_counter/PYB_FREQ > EPISODE_LEN_SEC, pre-increment (:379,:382)
  // Meetup terminates when every pair has met (MeetupAviary.py:115-121; no pairs at M = 1: always)
  const bool terminated = (TASK == TASK_SWARM) ? (P.task == TASK_MEETUP && (flags & 4) == 0) : (flags & 1) != 0;
  const bool truncated = ((flags & 2) != 0) || time_up;
  const bool done_reset = active && (terminated || truncated) && P.auto_reset;
  if (active && drone == 0) {
    P.reward[env] = reward;
    P.terminated[env] = terminated ? 1 : 0;
    P.truncated[env] = truncated ? 1 : 0;
    st_hint(P.stepc + env, done_reset ? 0 : stepc + P.S, l2.state);
    // episode statistics on the device (record_episode_statistics.py:144-171)
    if (P.ep_ret != nullptr) {
      float ep = cur.ep_ret + reward;   // loaded up front with the other inputs
      if (terminated || truncated) {
        atomicAdd(P.ep_acc + 0, (double)ep);
        atomicAdd(P.ep_acc + 1, (double)(stepc / P.S + 1));
        atomicAdd(P.ep_acc + 2, 1.0);
        ep = 0.f;
      }
      st_hint(P.ep_ret + env, ep, l2.state);
    }
  }

  // ---- reset-on-done (subproc_vec_env.py:195-206), rare -------------------------------------------
  if (__any_sync(0xffffffffu, done_reset)) {
    float cx = 0.f, cy = 0.f, cz = 0.f;
    if (jit) {   // MultiHoverAviary.py:83-102, every lane draws its own drone's jitter
      const long long ib = (long long)env * P.init_env_stride + drone * 3;
      bool retry = done_reset;
#pragma unroll 1
      for (int attempt = 0; attempt <= kMaxJitterTries; ++attempt) {
        const bool last = attempt == kMaxJitterTries;
        if (retry) {
          float j0 = 0.f, j1 = 0.f, j2 = 0.f;
          if (!last) {
            if (P.reset_mode == RESET_BUFFER && P.jitter != nullptr) {
              j0 = P.jitter[g * 3]; j1 = P.jitter[g * 3 + 1]; j2 = P.jitter[g * 3 + 2];
            } else {
              uint32_t c[4] = {(uint32_t)env, (uint32_t)total + P.philox_base, (uint32_t)(attempt * M + drone), 0u};
              uint32_t c2[4] = {c[0], c[1], c[2], 1u};
              philox4x32_10(c, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
              philox4x32_10(c2, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
              j0 = -0.25f + 0.5f * u01(c[0], c[1], 0.f);
              j1 = -0.25f + 0.5f * u01(c[2], c[3], 0.f);
              j2 = -0.25f + 0.5f * u01(c2[0], c2[1], 0.f);
            }
          }
          cx = P.init_xyz[ib] + j0;
          cy = P.init_xyz[ib + 1] + j1;
          cz = P.init_xyz[ib + 2] + j2;
          cz = cz < 0.1f ? 0.1f : (cz > 1.0f ? 1.0f : cz);
        }
        int bad = 0;
#pragma unroll 1
        for (int o = 1; o < M; ++o) {
          int t = drone + o;
          t -= (t >= M) ? M : 0;
          const int src = group_base + t;
          const float ox = __shfl_sync(0xffffffffu, cx, src), oy = __shfl_sync(0xffffffffu, cy, src),
                      oz = __shfl_sync(0xffffffffu, cz, src);
          const float dx = cx - ox, dy = cy - oy, dz = cz - oz;
          bad |= (sqrtf(dx * dx + dy * dy + dz * dz) < 0.5f) ? 1 : 0;
        }
        {   // any drone of the env too close -> the whole env redraws
          const int b0 = bad;
#pragma unroll 1
          for (int o = 1; o < M; ++o) {
            int t = drone + o;
            t -= (t >= M) ? M : 0;
            bad |= __shfl_sync(0xffffffffu, b0, group_base + t);
          }
        }
        if (last || P.reset_mode == RESET_BUFFER) bad = 0;
        retry = retry && (bad != 0);
        if (!__any_sync(0xffffffffu, retry)) break;
      }
    }
    if (done_reset) {
      if (P.terminal_obs != nullptr) {
        float* to = P.terminal_obs + (size_t)g * D;
        for (int k = 0; k < D; ++k) to[k] = myrow[k];
      }
      const float cand[3] = {cx, cy, cz};
      float kin[12];
      reset_drone<float, TASK>(P, env, drone, jit ? cand : nullptr, d, kin);
#pragma unroll
      for (int k = 0; k < 12; ++k) myrow[k] = kin[k];
      if (TASK == TASK_SPIRAL) {   // reset obs is evaluated at step_counter = 0
        float rp[3], rv[3], sphi, cphi;
        spiral_reference(P, 0, drone, rp, rv, sphi, cphi);
        spiral_extras(myrow + 12 + B * A, d, rp, rv, sphi, cphi);
      }
    }
  }

  // ---- 4. the finished rows leave as one TMA bulk store; state planes as 128-bit stores ------------
  const long long left = P.n_total - g0;
  const int tile_rows = 4 * EW * M;
  const int rows = (int)(left < (long long)tile_rows ? left : (long long)tile_rows);
  const uint32_t bytes = (uint32_t)rows * (uint32_t)D * 4u;
  float* gobs = P.obs + (size_t)g0 * D;
  const bool bulk = P.obs_aligned && (bytes & 15u) == 0;
  if (bulk) fence_proxy_async_smem();    // my generic-proxy writes -> visible to the async proxy
  __syncthreads();
  if (bulk) {
    if (tid == 0) bulk_store_s2g(gobs, tile_s, bytes);
  } else {                               // ragged last tile whose byte count is not a multiple of 16
    for (int i = tid; i < rows * D; i += kBlock) gobs[i] = tile_s[i];
  }
  if (active) {
    st_hint(P.s0 + g, make_float4(d.px, d.py, d.pz, d.qx), l2.state);
    st_hint(P.s1 + g, make_float4(d.qy, d.qz, d.qw, d.vx), l2.state);
    st_hint(P.s2 + g, make_float4(d.vy, d.vz, d.wx, d.wy), l2.state);
    st_hint(P.s3 + g, make_float4(d.wz, d.tx, d.ty, d.tz), l2.state);
  }
  // ---- advance the global step count: last CTA out.  Every thread of this CTA consumed
  // gsteps[0] (ring addresses) before the __syncthreads above, so the ticket needs no fence:
  // a __threadfence here would hold the CTA — and its shared memory — until all of its stores
  // have drained (measured: ~half of the CTA's lifetime).  Kernel completion publishes the data.
  if (P.pipeline) {    // publish this tile's epoch (every launch of a pipelining handle does, however it waited)
    __syncthreads();   // every thread's state / ring / reward stores are issued (and ordered before thread 0's release)
    if (tid == 0) {
      if (bulk) bulk_wait_all0();   // the observation rows are written
      // device-resident step count (what a later CUDA-graph replay starts from).  Eager launches overlap, so a
      // "last CTA out" ticket could mix launches; they do not read the counter either, so tile 0's CTA — ordered
      // after tile 0 of the previous step by the epoch chain — simply writes it.  Graph replays (which read the
      // counter, and never overlap) keep the ticket.
      if (P.host_total >= 0) {
        if (tile == 0) P.gsteps[0] = (total + 1 >= P.total_wrap) ? 0 : total + 1;
      } else {
        const unsigned ticket = atomicAdd(reinterpret_cast<unsigned*>(P.gsteps + 1), 1u);
        if (ticket == gridDim.x - 1) {
          P.gsteps[1] = 0;
          if (P.advance) P.gsteps[0] = (total + 1 >= P.total_wrap) ? 0 : total + 1;
        }
      }
      st_release_gpu(P.tile_epoch + tile, total + 1);   // cumulative: the CTA's stores are visible before the epoch
      atomicAdd(P.finished, 1ull);
    }
    return;
  }
  if (tid == 0) {
    const unsigned ticket = atomicAdd(reinterpret_cast<unsigned*>(P.gsteps + 1), 1u);
    if (ticket == gridDim.x - 1) {
      P.gsteps[1] = 0;
      if (P.advance) P.gsteps[0] = (total + 1 >= P.total_wrap) ? 0 : total + 1;
    }
    if (bulk) bulk_wait_read0();   // shared memory must outlive the bulk store's reads
  }
}


// ---------------------------------------------------------------------------------------------------------------
// K control steps in ONE launch (bd_step_many): the action tape of all K steps is known up front and tiles are whole
// environments, so a CTA can take its tile through all K steps without ever meeting another CTA.  The drone states stay
// in registers from step to step, the action history stays in shared memory (two tiles, used alternately: the next row
// is the previous row shifted by one ring slot while the TMA engine still reads the previous tile), and per step only
// the new action comes in and the finished observation rows, reward and flags go out.  What bounds a small batch
// (BASELINE configs[3] as literally sharded: 8 192 envs per GPU = 256 tiles on 148 SMs) is the latency of one step's
// chain launch -> loads -> 8 substeps -> stores -> next launch (16 us, 0.20 of the HBM peak); here the chain is the
// substeps alone.  Results are bit-identical to K single launches (same device functions, same order).
// Not supported here (the caller falls back to K launches): terminal observations, rows that cannot leave as a TMA
// bulk store.
struct ManySpan {
  int K;
  long long act_step;   // elements between consecutive steps' action sets
  long long obs_step;   // floats between consecutive observation slots
  long long out_step;   // elements between consecutive reward / flag slots
};
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory"); }

template <int TASK, int A, bool VEC, int AERO>
__global__ void __launch_bounds__(kBlock, 3)
step_kernel_tile_many(const __grid_constant__ Params<float> P, const ManySpan Q) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int M = P.M, B = P.B, D = P.D, EW = P.EW;
  const bool pow2 = (M & (M - 1)) == 0;
  constexpr bool vec = VEC;
  const int env_w = pow2 ? (lane >> (31 - __clz(M))) : lane / M;
  const int group_base = env_w * M;
  const int drone = lane - group_base;
  const int tile = blockIdx.x;
  const int env_l = (tid >> 5) * EW + env_w;
  const int env = tile * (4 * EW) + env_l;
  const bool active = env_w < EW && env < P.N;
  const long long g0 = (long long)tile * (4 * EW) * M;
  const long long g = (long long)env * M + drone;
  const int tile_rows = 4 * EW * M;
  const size_t tile_floats = (size_t)tile_rows * D;            // a multiple of 4 floats (checked on the host)
  float* const tiles = reinterpret_cast<float*>(smem_raw);     // [2][tile rows][D]
  const size_t rowoff = (size_t)(env_w < EW ? env_l * M + drone : 0) * D;
  const bool jit = (TASK == TASK_MULTIHOVER) && (P.reset_mode != RESET_FIXED);
  const long long gh = active ? g : P.n_total;
  const long long left = P.n_total - g0;
  const int rows = (int)(left < (long long)tile_rows ? left : (long long)tile_rows);
  const uint32_t bytes = (uint32_t)rows * (uint32_t)D * 4u;

  pdl_wait();     // everything earlier launches wrote (state, ring, counters) is complete and visible
  int total = P.host_total >= 0 ? P.host_total : P.gsteps[0];
  int head = total % B;
  TileIn<A> cur;
  load_state<A>(P, g, env, active, cur);
  issue_history<float, A, VEC>(P, gh, head, tiles + rowoff, 0, B - 1);
  cp_async_commit();
  load_action<A>(P, g, active, cur);
  int stepc = cur.stepc;
  float ep = cur.ep_ret;
  float last_sum = 0.f;
  if constexpr (AERO == 2) {
    if ((P.aero & AERO_DRAG) && active && stepc > 0) {
      const int prev = head == 0 ? B - 1 : head - 1;
      const float* lp = P.hist + ((size_t)prev * P.n_total + g) * A;
      if constexpr (A == 4) {
        const float4 pa = *reinterpret_cast<const float4*>(lp);
        last_sum = (__fadd_rn(1.0f, __fmul_rn(0.05f, pa.x)) + __fadd_rn(1.0f, __fmul_rn(0.05f, pa.y))) +
                   (__fadd_rn(1.0f, __fmul_rn(0.05f, pa.z)) + __fadd_rn(1.0f, __fmul_rn(0.05f, pa.w)));
      } else {
        last_sum = 4.0f * __fadd_rn(1.0f, __fmul_rn(0.05f, lp[0]));
      }
    }
  }
  Drone<float> d;
  d.px = cur.s0.x; d.py = cur.s0.y; d.pz = cur.s0.z; d.qx = cur.s0.w;
  d.qy = cur.s1.x; d.qz = cur.s1.y; d.qw = cur.s1.z; d.vx = cur.s1.w;
  d.vy = cur.s2.x; d.vz = cur.s2.y; d.wx = cur.s2.z; d.wy = cur.s2.w;
  d.wz = cur.s3.x; d.tx = cur.s3.y; d.ty = cur.s3.z; d.tz = cur.s3.w;
  float4 act = cur.act;

#pragma unroll 1
  for (int k = 0; k < Q.K; ++k) {
    float* const tile_s = tiles + (size_t)(k & 1) * tile_floats;
    float* const myrow = tile_s + rowoff;
    // the next step's action is on its way while this step computes
    float4 act_next = make_float4(0.f, 0.f, 0.f, 0.f);
    if (k + 1 < Q.K && active) {
      if constexpr (A == 4) act_next = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(P.actions) + (size_t)(k + 1) * Q.act_step)[g];
      else act_next.x = (reinterpret_cast<const float*>(P.actions) + (size_t)(k + 1) * Q.act_step)[g];
    }
    if (k > 0) {
      // this tile buffer was handed to the TMA engine two steps ago: its reads must be over before it is rewritten
      if (k > 1) {
        if (tid == 0) bulk_wait_read1();
        __syncthreads();
      }
      // history = the previous row's, one slot older (oldest entry drops out); thread-private rows, no barrier
      const float* prow = tiles + (size_t)((k - 1) & 1) * tile_floats + rowoff;
      if (active) {
        if constexpr (A == 4) {
          if (vec) {
#pragma unroll 4
            for (int j = 0; j < B - 1; ++j)
              *reinterpret_cast<float4*>(myrow + 12 + j * 4) = *reinterpret_cast<const float4*>(prow + 12 + (j + 1) * 4);
          } else {
            for (int j = 0; j < (B - 1) * 4; ++j) myrow[12 + j] = prow[12 + 4 + j];
          }
        } else {
          for (int j = 0; j < B - 1; ++j) myrow[12 + j] = prow[12 + 1 + j];
        }
      }
    }
    float onep[4];
    if constexpr (A == 4) {
      onep[0] = __fadd_rn(1.0f, __fmul_rn(0.05f, act.x));
      onep[1] = __fadd_rn(1.0f, __fmul_rn(0.05f, act.y));
      onep[2] = __fadd_rn(1.0f, __fmul_rn(0.05f, act.z));
      onep[3] = __fadd_rn(1.0f, __fmul_rn(0.05f, act.w));
    } else {
      onep[0] = onep[1] = onep[2] = onep[3] = __fadd_rn(1.0f, __fmul_rn(0.05f, act.x));
    }
    float avx = 0.f, avy = 0.f, avz = 0.f;
    fast_substeps<AERO>(P, d, onep, avx, avy, avz, group_base, drone, last_sum);
    float roll, pitch, yaw;
    quat_to_euler_fast(d.qx, d.qy, d.qz, d.qw, roll, pitch, yaw);
    if (k == 0) cp_async_wait_all();
    float contrib = 0.f;
    int flags = 0;
    if (active) {
      if (vec) {
        float4* r4 = reinterpret_cast<float4*>(myrow);
        r4[0] = make_float4(d.px, d.py, d.pz, roll);
        r4[1] = make_float4(pitch, yaw, d.vx, d.vy);
        r4[2] = make_float4(d.vz, avx, avy, avz);
      } else {
        myrow[0] = d.px; myrow[1] = d.py; myrow[2] = d.pz; myrow[3] = roll; myrow[4] = pitch; myrow[5] = yaw;
        myrow[6] = d.vx; myrow[7] = d.vy; myrow[8] = d.vz; myrow[9] = avx; myrow[10] = avy; myrow[11] = avz;
      }
      if constexpr (TASK != TASK_SWARM)
        task_terms<float, TASK>(P, d, roll, pitch, stepc, drone, myrow + 12 + B * A, contrib, flags);
      if constexpr (A == 4) {
        if (vec) *reinterpret_cast<float4*>(myrow + 12 + (B - 1) * 4) = act;
        else { float* o = myrow + 12 + (B - 1) * 4; o[0] = act.x; o[1] = act.y; o[2] = act.z; o[3] = act.w; }
        *reinterpret_cast<float4*>(P.hist + ((size_t)head * P.n_total + g) * 4) = act;
      } else {
        myrow[12 + B - 1] = act.x;
        P.hist[(size_t)head * P.n_total + g] = act.x;
      }
    }
    float swarm_reward_env = 0.f;
    if constexpr (TASK == TASK_SWARM) {
      int fl = 0;
      swarm_reward_env = swarm_reward_shfl(P, d, roll, pitch, lane, M, drone, fl);
      flags = active ? fl : 0;
    }
    if (pow2) {
#pragma unroll 1
      for (int o = M >> 1; o > 0; o >>= 1) {
        contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        flags |= __shfl_xor_sync(0xffffffffu, flags, o);
      }
    } else {
      const float c0 = contrib;
      const int f0 = flags;
#pragma unroll 1
      for (int o = 1; o < M; ++o) {
        int t = drone + o;
        t -= (t >= M) ? M : 0;
        contrib += __shfl_sync(0xffffffffu, c0, group_base + t);
        flags |= __shfl_sync(0xffffffffu, f0, group_base + t);
      }
    }
    const float reward = (TASK == TASK_SWARM) ? swarm_reward_env : ((TASK == TASK_HOVER) ? contrib : contrib / (float)M);
    const bool time_up = stepc >= P.trunc_counter;
    const bool terminated = (TASK == TASK_SWARM) ? (P.task == TASK_MEETUP && (flags & 4) == 0) : (flags & 1) != 0;
    const bool truncated = ((flags & 2) != 0) || time_up;
    const bool done_reset = active && (terminated || truncated) && P.auto_reset;
    if (active && drone == 0) {
      const size_t o = (size_t)k * Q.out_step + env;
      P.reward[o] = reward;
      P.terminated[o] = terminated ? 1 : 0;
      P.truncated[o] = truncated ? 1 : 0;
      if (P.ep_ret != nullptr) {
        ep += reward;
        if (terminated || truncated) {
          atomicAdd(P.ep_acc + 0, (double)ep);
          atomicAdd(P.ep_acc + 1, (double)(stepc / P.S + 1));
          atomicAdd(P.ep_acc + 2, 1.0);
          ep = 0.f;
        }
      }
    }
    // the drag model's last_clipped_action of the next step: this step's action, zero after a reset
    if constexpr (AERO == 2) last_sum = done_reset ? 0.f : (onep[0] + onep[1]) + (onep[2] + onep[3]);
    stepc = done_reset ? 0 : stepc + P.S;

    if (__any_sync(0xffffffffu, done_reset)) {
      float cx = 0.f, cy = 0.f, cz = 0.f;
      if (jit) {
        const long long ib = (long long)env * P.init_env_stride + drone * 3;
        bool retry = done_reset;
#pragma unroll 1
        for (int attempt = 0; attempt <= kMaxJitterTries; ++attempt) {
          const bool last = attempt == kMaxJitterTries;
          if (retry) {
            float j0 = 0.f, j1 = 0.f, j2 = 0.f;
            if (!last) {
              if (P.reset_mode == RESET_BUFFER && P.jitter != nullptr) {
                j0 = P.jitter[g * 3]; j1 = P.jitter[g * 3 + 1]; j2 = P.jitter[g * 3 + 2];
              } else {
                uint32_t c[4] = {(uint32_t)env, (uint32_t)total + P.philox_base, (uint32_t)(attempt * M + drone), 0u};
                uint32_t c2[4] = {c[0], c[1], c[2], 1u};
                philox4x32_10(c, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
                philox4x32_10(c2, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
                j0 = -0.25f + 0.5f * u01(c[0], c[1], 0.f);
                j1 = -0.25f + 0.5f * u01(c[2], c[3], 0.f);
                j2 = -0.25f + 0.5f * u01(c2[0], c2[1], 0.f);
              }
            }
            cx = P.init_xyz[ib] + j0;
            cy = P.init_xyz[ib + 1] + j1;
            cz = P.init_xyz[ib + 2] + j2;
            cz = cz < 0.1f ? 0.1f : (cz > 1.0f ? 1.0f : cz);
          }
          int bad = 0;
#pragma unroll 1
          for (int o = 1; o < M; ++o) {
            int t = drone + o;
            t -= (t >= M) ? M : 0;
            const int src = group_base + t;
            const float ox = __shfl_sync(0xffffffffu, cx, src), oy = __shfl_sync(0xffffffffu, cy, src),
                        oz = __shfl_sync(0xffffffffu, cz, src);
            const float dx = cx - ox, dy = cy - oy, dz = cz - oz;
            bad |= (sqrtf(dx * dx + dy * dy + dz * dz) < 0.5f) ? 1 : 0;
          }
          {
            const int b0 = bad;
#pragma unroll 1
            for (int o = 1; o < M; ++o) {
              int t = drone + o;
              t -= (t >= M) ? M : 0;
              bad |= __shfl_sync(0xffffffffu, b0, group_base + t);
            }
          }
          if (last || P.reset_mode == RESET_BUFFER) bad = 0;
          retry = retry && (bad != 0);
          if (!__any_sync(0xffffffffu, retry)) break;
        }
      }
      if (done_reset) {
        const float cand[3] = {cx, cy, cz};
        float kin[12];
        reset_drone<float, TASK>(P, env, drone, jit ? cand : nullptr, d, kin);
#pragma unroll
        for (int q = 0; q < 12; ++q) myrow[q] = kin[q];
        if (TASK == TASK_SPIRAL) {
          float rp[3], rv[3], sphi, cphi;
          spiral_reference(P, 0, drone, rp, rv, sphi, cphi);
          spiral_extras(myrow + 12 + B * A, d, rp, rv, sphi, cphi);
        }
      }
    }
    // this step's rows leave as one TMA bulk store while the next step computes
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) bulk_store_s2g(P.obs + (size_t)k * Q.obs_step + (size_t)g0 * D, tile_s, bytes);
    act = act_next;
    total = (total + 1 >= P.total_wrap) ? 0 : total + 1;
    head = head + 1 == B ? 0 : head + 1;
  }

  if (active) {
    P.s0[g] = make_float4(d.px, d.py, d.pz, d.qx);
    P.s1[g] = make_float4(d.qy, d.qz, d.qw, d.vx);
    P.s2[g] = make_float4(d.vy, d.vz, d.wx, d.wy);
    P.s3[g] = make_float4(d.wz, d.tx, d.ty, d.tz);
    if (drone == 0) {
      P.stepc[env] = stepc;
      if (P.ep_ret != nullptr) P.ep_ret[env] = ep;
    }
  }
  __syncthreads();   // every thread's stores are issued (and ordered before thread 0's release)
  if (tid == 0) {
    bulk_wait_all0();
    if (P.host_total >= 0) {
      if (tile == 0) P.gsteps[0] = total;
    } else {            // CUDA-graph replay: other CTAs read the counter when they start, the last one out advances it
      const unsigned ticket = atomicAdd(reinterpret_cast<unsigned*>(P.gsteps + 1), 1u);
      if (ticket == gridDim.x - 1) { P.gsteps[1] = 0; P.gsteps[0] = total; }
    }
    if (P.pipeline) {   // later pipelined launches wait on this tile's epoch / count finished (tile, step) pairs
      st_release_gpu(P.tile_epoch + tile, total);
      atomicAdd(P.finished, (unsigned long long)Q.K);
    }
  }
}

}  // namespace bd
