// Batched drone-step kernels for sm_100a.
//
// One thread per drone, one CTA = E = 128/M whole environments, so the O(M^2)
// downwash term and the per-env reward / termination reductions never leave the
// CTA.  A control step is ONE launch of step_kernel:
//
//   action -> rpm (BaseRLAviary.py:191-192,224-225)
//   S substeps of explicit dynamics with the state in registers
//       (BaseAviary.py:343-374, _dynamics :815-877, _integrateQ :879-892,
//        Bullet quaternion round trip of _updateAndStoreKinematicInformation :509-519)
//   KIN observation (BaseRLAviary.py:307-319, SpiralAviary.py:120-146)
//   reward / terminated / truncated of the task
//       (HoverAviary.py:77-117, MultiHoverAviary.py:128-268, SpiralAviary.py:150-196)
//   step-counter advance (:382) and SubprocVecEnv's reset-on-done
//       (subproc_vec_env.py:195-206; MultiHoverAviary.py:75-110 jitter)
//
// HBM traffic per drone-step is the algorithmic minimum + one ring slot:
// 4 x 128-bit state loads/stores (SoA planes), the action, B-1 history slots
// (cp.async straight into the shared-memory observation tile), and the
// observation rows, which leave the CTA as one contiguous, fully coalesced block.
//
// Two arithmetic flavours are compiled from the same source:
//   exact  (double, or float with GENERIC): the reference's formulas verbatim
//          (s = 2/|q|^2 rotation, Bullet matrix->quaternion branches, sqrt/sin/cos
//          quaternion step with the 1e-8 early-out) — the fp64 parity mode.
//   fast   (float, !GENERIC): same maths re-associated for throughput: rotation
//          column only, per-step thrust/torque hoisting, polynomial sinc/cos for
//          the quaternion step, rsqrt normalisation with Bullet's sign rule.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "bd_device.cuh"
#include "bd_params.h"

namespace bd {

template <typename R, bool GENERIC> struct Bounds { static constexpr int kMinBlocks = 1; };
template <> struct Bounds<float, false> { static constexpr int kMinBlocks = 6; };
template <> struct Bounds<float, true> { static constexpr int kMinBlocks = 3; };

// =========================================================================
//                     generic step kernel (any configuration)
// =========================================================================
// Same shape as the fast kernel (bd_step_tile.cuh): one CTA per tile of E = 128/M whole
// environments, every load issued up front (ring planes with cp.async into the thread's row of
// a dense row-major shared-memory tile), the finished rows leave as one contiguous block.
// Differences: any M <= 128 (per-env reductions through shared memory instead of shuffles),
// double or float, the exact arithmetic flavour, ground effect / drag / downwash (positions of
// the env's drones staged in shared memory per substep), Euler-angle integrator, optional
// world angular velocity plane.
template <typename R, int TASK, int A, bool GENERIC>
__global__ void __launch_bounds__(kBlock, Bounds<R, GENERIC>::kMinBlocks)
step_kernel(const __grid_constant__ Params<R> P) {
  using R4 = typename V4<R>::type;
  constexpr bool FAST = (sizeof(R) == 4) && !GENERIC;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int M = P.M, E = P.E, B = P.B, D = P.D;
  float* tile_s = reinterpret_cast<float*>(smem_raw);                         // [kBlock][D] dense
  R* sred = reinterpret_cast<R*>(smem_raw + (((size_t)kBlock * D * 4 + 15) & ~(size_t)15));   // [kBlock]
  R* spos = sred + kBlock;                                                    // [kBlock][3]
  int* sflag = reinterpret_cast<int*>(spos + 3 * kBlock);                     // [kBlock]
  int* sdone = sflag + kBlock;                                                // [kBlock]
  R* svel = reinterpret_cast<R*>(sdone + kBlock);                             // [kBlock][3]  (swarm tasks only)
  R* saux = svel + 3 * kBlock;                                                // [kBlock]     (swarm tasks only)
  float* myrow = tile_s + (size_t)tid * D;
  const bool vec = (A == 4) && ((D & 3) == 0);

  const int env_l = tid / M;
  const int drone = tid - env_l * M;
  const int bid = blockIdx.x + P.block0;   // block0 > 0: a launch over a sub-range of tiles (bd_step_host pipelines chunks)
  const int env = bid * E + env_l;
  const bool active = (env_l < E) && (env < P.N);
  const long long g0 = (long long)bid * E * M;
  const long long g = g0 + tid;

  // ---- 0. dependency on the previous control step (see bd_step_tile.cuh): tile-level when this launch fills the
  // GPU, else grid-wide.  Everything below reads only this tile's data.
  const bool pipe = P.pipe_wait && P.host_total >= 0;
  if (P.pipeline) {
    pdl_launch_dependents();
    if (pipe) {
      if (pipe_gate(P, bid, P.host_total, tid)) pdl_wait();
    } else {
      pdl_wait();
    }
  }
  // ---- 1. every load of the tile is issued before anything is consumed ----------------------
  const int total = P.host_total >= 0 ? P.host_total : P.gsteps[0];
  const int head = total % B;   // ring slot overwritten by this step's action
  if (active) {
    if (vec) issue_history<R, A, (A == 4)>(P, g, head, myrow, 0, B - 1);
    else issue_history<R, A, false>(P, g, head, myrow, 0, B - 1);
  }
  cp_async_commit();

  Drone<R> d;
  R rpm[4] = {R(0), R(0), R(0), R(0)};
  float af[4] = {0.f, 0.f, 0.f, 0.f};
  float onep[4] = {1.f, 1.f, 1.f, 1.f};   // fl32(1 + 0.05 a) per motor (float actions)
  R last_rpm[4] = {R(0), R(0), R(0), R(0)};
  int stepc = 0;
  float ep_in = 0.f;
  if (active) {
    const R4 a0 = P.s0[g], a1 = P.s1[g], a2 = P.s2[g], a3 = P.s3[g];
    bool from_double = false;
    if constexpr (sizeof(R) == 8) from_double = !P.action_is_f32;
    double ad[4] = {0, 0, 0, 0};
    if (from_double) {
      const double* ap = reinterpret_cast<const double*>(P.actions) + g * A;
#pragma unroll
      for (int k = 0; k < A; ++k) ad[k] = ap[k];
    } else {
      const float* ap = reinterpret_cast<const float*>(P.actions) + g * A;
      if constexpr (A == 4) {
        const float4 v = *reinterpret_cast<const float4*>(ap);
        af[0] = v.x; af[1] = v.y; af[2] = v.z; af[3] = v.w;
      } else {
#pragma unroll
        for (int k = 0; k < A; ++k) af[k] = ap[k];
      }
    }
    stepc = P.stepc[env];
    if (P.ep_ret != nullptr) ep_in = P.ep_ret[env];
    d.px = a0.x; d.py = a0.y; d.pz = a0.z; d.qx = a0.w;
    d.qy = a1.x; d.qz = a1.y; d.qw = a1.z; d.vx = a1.w;
    d.vy = a2.x; d.vz = a2.y; d.wx = a2.z; d.wy = a2.w;
    d.wz = a3.x; d.tx = a3.y; d.ty = a3.z; d.tz = a3.w;
    bool pid = false;
    if constexpr (GENERIC) pid = P.act_type >= ACT_PID;
    if (from_double) {
#pragma unroll
      for (int k = 0; k < A; ++k) af[k] = (float)ad[k];
    }
    if (pid) {
      if constexpr (GENERIC) {
        // DSL PID in the loop (BaseRLAviary.py:193-235): state at the start of the step -> rpm
        R roll0, pitch0, yaw0;
        quat_to_euler(d.qx, d.qy, d.qz, d.qw, roll0, pitch0, yaw0);
        R tp[3], tv[3], tyaw, c[9];
        pid_targets(P, d, yaw0, af, ad, from_double, tp, tyaw, tv);
#pragma unroll
        for (int k = 0; k < 9; ++k) c[k] = P.ctrl[(size_t)k * P.n_total + g];
        if ((P.aero & AERO_DRAG) && stepc > 0) {   // last_clipped_action (BaseAviary.py:372,468)
#pragma unroll
          for (int k = 0; k < 4; ++k) last_rpm[k] = P.ctrl[(size_t)(9 + k) * P.n_total + g];
        }
        dsl_pid(P, d, roll0, pitch0, yaw0, tp, tyaw, tv, c, rpm);
#pragma unroll
        for (int k = 0; k < 9; ++k) P.ctrl[(size_t)k * P.n_total + g] = c[k];
#pragma unroll
        for (int k = 0; k < 4; ++k) P.ctrl[(size_t)(9 + k) * P.n_total + g] = rpm[k];
      }
    } else if (from_double) {
      if constexpr (A != 3) {
#pragma unroll
        for (int k = 0; k < A; ++k) {
          const R r = P.hover_rpm * (R(1) + R(0.05) * (R)ad[k]);               // BaseRLAviary.py:192
          if constexpr (A == 4) rpm[k] = r; else rpm[0] = rpm[1] = rpm[2] = rpm[3] = r;
        }
      }
    } else {
      if constexpr (A != 3) {
#pragma unroll
        for (int k = 0; k < A; ++k) {
          // numpy evaluates 1 + 0.05*a in float32 for float32 actions (two roundings)
          const float s = __fadd_rn(1.0f, __fmul_rn(0.05f, af[k]));
          const R r = P.hover_rpm * (R)s;
          if constexpr (A == 4) { rpm[k] = r; onep[k] = s; }
          else { rpm[0] = rpm[1] = rpm[2] = rpm[3] = r; onep[0] = onep[1] = onep[2] = onep[3] = s; }
        }
      }
    }
    // newest history entry: ring slot `head` (the stale slot) and the tail of the row
    float* hp = P.hist + ((size_t)head * P.n_total + g) * A;
    float* newest = myrow + 12 + (B - 1) * A;
#pragma unroll
    for (int k = 0; k < A; ++k) { hp[k] = af[k]; newest[k] = af[k]; }
    if (GENERIC && !pid && (P.aero & AERO_DRAG) && stepc > 0) {
      // last_clipped_action (BaseAviary.py:372,468): previous step's rpm, zero after a reset
      const int prev = head == 0 ? B - 1 : head - 1;
      const float* lp = P.hist + ((size_t)prev * P.n_total + g) * A;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float a = lp[A == 4 ? k : 0];
        float s = __fadd_rn(1.0f, __fmul_rn(0.05f, a));
        last_rpm[k] = P.hover_rpm * (R)s;
      }
    }
  } else {
    rpm[0] = rpm[1] = rpm[2] = rpm[3] = R(0);
    d = Drone<R>{};
    d.qw = R(1);
    rpm[0] = rpm[1] = rpm[2] = rpm[3] = R(0);
  }

  // ---- 2. S substeps of explicit dynamics ------------------------------------
  const R dt = P.dt;
  R avx = R(0), avy = R(0), avz = R(0);   // world angular velocity R_old * w_new (:873)

  if constexpr (FAST) {
    fast_substeps<0>(P, d, onep, avx, avy, avz);
  } else {
#pragma unroll 1
    for (int s = 0; s < P.S; ++s) {
      if (GENERIC && (P.aero & AERO_DW)) {   // Jacobi snapshot of the env's positions (:346-347,799-800)
        __syncthreads();
        spos[tid * 3 + 0] = d.px; spos[tid * 3 + 1] = d.py; spos[tid * 3 + 2] = d.pz;
        __syncthreads();
      }
      R m[9];
      quat_to_mat(d.qx, d.qy, d.qz, d.qw, m);
      R f[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) f[k] = rpm[k] * rpm[k] * P.kf;                      // :838
      R fx_extra = R(0), fy_extra = R(0), fz_extra = R(0);
      if (GENERIC && P.aero) {
        if (P.aero & AERO_GND) {             // :739-742, added to the propeller thrusts
          if (tilt_below_half_pi(d.qx, d.qy, d.qz, d.qw)) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              R h = d.pz + (m[6] * P.prop_x[k] + m[7] * P.prop_y[k]);
              h = h < P.gnd_h_clip ? P.gnd_h_clip : h;
              const R ratio = P.prop_radius / (R(4) * h);
              f[k] += rpm[k] * rpm[k] * P.kf * P.gnd_coeff * (ratio * ratio);
            }
          }
        }
        if (P.aero & AERO_DRAG) {            // :773-774 -> world force k (.) v
          const R* lr = (s == 0) ? last_rpm : rpm;
          const R two_pi = R(2) * R(3.14159265358979323846);
          const R sum = two_pi * lr[0] / R(60) + two_pi * lr[1] / R(60) + two_pi * lr[2] / R(60) +
                        two_pi * lr[3] / R(60);
          fx_extra += R(-1) * P.drag_xy * sum * d.vx;
          fy_extra += R(-1) * P.drag_xy * sum * d.vy;
          fz_extra += R(-1) * P.drag_z * sum * d.vz;
        }
        if (P.aero & AERO_DW) {              // :798-804, body-z force -> R [0,0,F]
          R dw = R(0);
          const R* ep = spos + (size_t)env_l * M * 3;
          for (int i = 0; i < M; ++i) {
            const R dz = ep[i * 3 + 2] - d.pz;
            const R ddx = ep[i * 3] - d.px, ddy = ep[i * 3 + 1] - d.py;
            const R dxy = sqrt_(ddx * ddx + ddy * ddy);
            if (dz > R(0) && dxy < R(10)) {
              const R ratio = P.prop_radius / (R(4) * dz);
              const R alpha = P.dw1 * (ratio * ratio);
              const R beta = P.dw2 * dz + P.dw3;
              const R q_ = dxy / beta;
              dw += -alpha * exp_(R(-0.5) * (q_ * q_));
            }
          }
          fx_extra += m[2] * dw; fy_extra += m[5] * dw; fz_extra += m[8] * dw;
        }
      }
      const R thrust = ((f[0] + f[1]) + f[2]) + f[3];
      const R Fx = m[2] * thrust + fx_extra;
      const R Fy = m[5] * thrust + fy_extra;
      const R Fz = (m[8] * thrust - P.gravity) + fz_extra;                        // :839-841
      R zt[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) zt[k] = rpm[k] * rpm[k] * P.km;
      R tx, ty, tz;
      if (P.model == MODEL_RACE) {
        tz = ((zt[0] - zt[1]) + zt[2]) - zt[3];
        tx = (f[0] + f[1] - f[2] - f[3]) * P.arm;
        ty = (-f[0] + f[1] + f[2] - f[3]) * P.arm;
      } else if (P.model == MODEL_CF2X) {
        tz = ((-zt[0] + zt[1]) - zt[2]) + zt[3];
        tx = -(f[0] + f[1] - f[2] - f[3]) * P.arm;
        ty = (-f[0] + f[1] + f[2] - f[3]) * P.arm;
      } else {
        tz = ((-zt[0] + zt[1]) - zt[2]) + zt[3];
        tx = (f[1] - f[3]) * P.arm;
        ty = (-f[0] + f[2]) * P.arm;
      }
      // torques - w x (J w), J diagonal (:856-857)
      const R jwx = P.jx * d.wx, jwy = P.jy * d.wy, jwz = P.jz * d.wz;
      tx -= d.wy * jwz - d.wz * jwy;
      ty -= d.wz * jwx - d.wx * jwz;
      tz -= d.wx * jwy - d.wy * jwx;
      d.vx += dt * (Fx * P.inv_m);                                                // :860
      d.vy += dt * (Fy * P.inv_m);
      d.vz += dt * (Fz * P.inv_m);
      d.wx += dt * (P.ijx * tx);                                                  // :861
      d.wy += dt * (P.ijy * ty);
      d.wz += dt * (P.ijz * tz);
      d.px += dt * d.vx;                                                          // :862
      d.py += dt * d.vy;
      d.pz += dt * d.vz;
      if (!GENERIC || P.integrator == 0) {
        avx = m[0] * d.wx + m[1] * d.wy + m[2] * d.wz;                            // :873
        avy = m[3] * d.wx + m[4] * d.wy + m[5] * d.wz;
        avz = m[6] * d.wx + m[7] * d.wy + m[8] * d.wz;
        integrate_q_exact(d.qx, d.qy, d.qz, d.qw, d.wx, d.wy, d.wz, dt);          // :863
      } else {  // Euler-angle integrator (scg base_aviary.py:499-508)
        R roll, pitch, yaw;
        quat_to_euler(d.qx, d.qy, d.qz, d.qw, roll, pitch, yaw);
        euler_to_quat(roll + dt * d.wx, pitch + dt * d.wy, yaw + dt * d.wz, d.qx, d.qy, d.qz, d.qw);
        avx = d.wx; avy = d.wy; avz = d.wz;
      }
      bullet_roundtrip(d.qx, d.qy, d.qz, d.qw);                                   // :347 / :374
    }
  }

  // ---- 3. complete my observation row, reward terms, flags ---------------------
  R roll, pitch, yaw;
  quat_to_euler(d.qx, d.qy, d.qz, d.qw, roll, pitch, yaw);
  R contrib = R(0);
  int flags = 0;   // bit0: terminated condition, bit1: truncated condition (hover bounds)
  cp_async_wait_all();
  if (active) {
    // [pos rpy vel ang_v] (BaseRLAviary.py:314-315)
    myrow[0] = (float)d.px; myrow[1] = (float)d.py; myrow[2] = (float)d.pz;
    myrow[3] = (float)roll; myrow[4] = (float)pitch; myrow[5] = (float)yaw;
    myrow[6] = (float)d.vx; myrow[7] = (float)d.vy; myrow[8] = (float)d.vz;
    myrow[9] = (float)avx; myrow[10] = (float)avy; myrow[11] = (float)avz;
    if constexpr (TASK != TASK_SWARM)
      task_terms<R, TASK>(P, d, roll, pitch, stepc, drone, myrow + 12 + B * A, contrib, flags);
  }
  if constexpr (TASK == TASK_SWARM) {
    // rewards couple the env's drones: stage final positions / velocities, then per-drone parts in parallel
    __syncthreads();   // the last substep's downwash loop may still be reading spos
    spos[tid * 3 + 0] = d.px; spos[tid * 3 + 1] = d.py; spos[tid * 3 + 2] = d.pz;
    svel[tid * 3 + 0] = d.vx; svel[tid * 3 + 1] = d.vy; svel[tid * 3 + 2] = d.vz;
    __syncthreads();
    R aux = R(0);
    if (active)
      swarm_terms(P, spos + (size_t)env_l * M * 3, svel + (size_t)env_l * M * 3, M, drone, d, roll, pitch, contrib, aux, flags);
    saux[tid] = aux;
  }
  sred[tid] = contrib;
  sflag[tid] = flags;
  __syncthreads();

  // ---- 4. per-env reduction by the env's first drone --------------------------
  int done_reset = 0;
  if (active && drone == 0) {
    R sum = R(0);
    int fl = 0;
    for (int i = 0; i < M; ++i) { sum += sred[tid + i]; fl |= sflag[tid + i]; }
    R reward = (TASK == TASK_HOVER) ? sum : sum / R(M);
    if constexpr (TASK == TASK_SWARM) reward = swarm_reward(P, M, sred + tid, saux + tid, svel + (size_t)tid * 3);
    const bool time_up = stepc >= P.trunc_counter;   // step_counter/PYB_FREQ > EPISODE_LEN_SEC, pre-increment (:379,:382)
    // Meetup terminates when every pair has met (MeetupAviary.py:115-121; no pairs at M = 1: always)
    const bool terminated = (TASK == TASK_SWARM) ? (P.task == TASK_MEETUP && (fl & 4) == 0) : (fl & 1) != 0;
    const bool truncated = ((fl & 2) != 0) || time_up;
    P.reward[env] = reward;
    P.terminated[env] = terminated ? 1 : 0;
    P.truncated[env] = truncated ? 1 : 0;
    done_reset = ((terminated || truncated) && P.auto_reset) ? 1 : 0;
    P.stepc[env] = done_reset ? 0 : stepc + P.S;
    sdone[env_l] = done_reset;
    // episode statistics on the device (record_episode_statistics.py:144-171)
    if (P.ep_ret != nullptr) {
      float ep = ep_in + (float)reward;
      if (terminated || truncated) {
        atomicAdd(P.ep_acc + 0, (double)ep);
        atomicAdd(P.ep_acc + 1, (double)(stepc / P.S + 1));
        atomicAdd(P.ep_acc + 2, 1.0);
        ep = 0.f;
      }
      P.ep_ret[env] = ep;
    }
  }
  const int any_reset = __syncthreads_or(done_reset);

  // ---- 5. reset-on-done (subproc_vec_env.py:195-206), rare ----------------------
  if (any_reset) {
    const bool my_reset = active && sdone[env_l];
    const bool jit = (TASK == TASK_MULTIHOVER) && (P.reset_mode != RESET_FIXED);
    if (jit) {
      if (my_reset && drone == 0) sample_jitter(P, env, total, 0, spos + (size_t)tid * 3);
      __syncthreads();
    }
    if (my_reset) {
      if (P.terminal_obs != nullptr) {   // info['terminal_observation']: the full last row of the episode
        float* to = P.terminal_obs + (size_t)g * D;
        for (int k = 0; k < D; ++k) to[k] = myrow[k];
      }
      float kin[12];
      reset_drone<R, TASK>(P, env, drone, jit ? spos + (size_t)tid * 3 : nullptr, d, kin);
#pragma unroll
      for (int k = 0; k < 12; ++k) myrow[k] = kin[k];
      avx = avy = avz = R(0);
      if (GENERIC && P.ctrl != nullptr && P.ctrl_reset) {   // optional: DSLPIDControl.reset() with the env
        for (int k = 0; k < 9; ++k) P.ctrl[(size_t)k * P.n_total + g] = R(0);
      }
      if (TASK == TASK_SPIRAL) {   // reset obs is evaluated at step_counter = 0
        R rp[3], rv[3], sphi, cphi;
        spiral_reference(P, 0, drone, rp, rv, sphi, cphi);
        spiral_extras(myrow + 12 + B * A, d, rp, rv, sphi, cphi);
      }
    }
  }

  // ---- 6. the finished rows leave as one contiguous block; state planes -------------------
  const long long left = P.n_total - g0;
  const int rows = (int)(left < (long long)E * M ? left : (long long)E * M);
  const uint32_t bytes = (uint32_t)rows * (uint32_t)D * 4u;
  float* gobs = P.obs + (size_t)g0 * D;
  const bool bulk = P.obs_aligned && ((bytes & 15u) == 0) && ((((size_t)g0 * D * 4) & 15) == 0);
  if (bulk) fence_proxy_async_smem();
  __syncthreads();
  if (bulk) {
    if (tid == 0) bulk_store_s2g(gobs, tile_s, bytes);
  } else {
    for (int i = tid; i < rows * D; i += kBlock) gobs[i] = tile_s[i];
  }
  if (active) {
    P.s0[g] = make4(d.px, d.py, d.pz, d.qx);
    P.s1[g] = make4(d.qy, d.qz, d.qw, d.vx);
    P.s2[g] = make4(d.vy, d.vz, d.wx, d.wy);
    P.s3[g] = make4(d.wz, d.tx, d.ty, d.tz);
    if (GENERIC && P.keep_angv) P.s4[g] = make4(avx, avy, avz, R(0));
  }
  if (P.pipeline) {    // publish this tile's epoch (bd_step_tile.cuh)
    __syncthreads();
    if (tid == 0) {
      if (bulk) bulk_wait_all0();
      // device-resident step count (what a later CUDA-graph replay starts from).  Eager launches overlap, so a
      // "last CTA out" ticket could mix launches; they do not read the counter either, so tile 0's CTA — ordered
      // after tile 0 of the previous step by the epoch chain — simply writes it.  Graph replays (which read the
      // counter, and never overlap) keep the ticket.
      if (P.host_total >= 0) {
        if (bid == 0) P.gsteps[0] = (total + 1 >= P.total_wrap) ? 0 : total + 1;
      } else {
        const unsigned ticket = atomicAdd(reinterpret_cast<unsigned*>(P.gsteps + 1), 1u);
        if (ticket == gridDim.x - 1) {
          P.gsteps[1] = 0;
          if (P.advance) P.gsteps[0] = (total + 1 >= P.total_wrap) ? 0 : total + 1;
        }
      }
      st_release_gpu(P.tile_epoch + bid, total + 1);
      atomicAdd(P.finished, 1ull);
    }
    return;
  }
  // advance the device-resident step count: last CTA out (every thread consumed `total` before
  // the barrier above; no fence, see bd_step_tile.cuh)
  if (tid == 0) {
    const unsigned ticket = atomicAdd(reinterpret_cast<unsigned*>(P.gsteps + 1), 1u);
    if (ticket == gridDim.x - 1) {
      P.gsteps[1] = 0;
      if (P.advance) P.gsteps[0] = (total + 1 >= P.total_wrap) ? 0 : total + 1;
    }
    if (bulk) bulk_wait_read0();   // shared memory must outlive the bulk store's reads
  }
}

// =========================================================================
//                    reset / state access kernels (cold paths)
// =========================================================================
template <typename R, int TASK, int A>
__global__ void __launch_bounds__(kBlock)
reset_kernel(const __grid_constant__ Params<R> P) {
  using R4 = typename V4<R>::type;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  R* spos = reinterpret_cast<R*>(smem_raw);   // [kBlock][3]
  const int tid = threadIdx.x;
  const int M = P.M, E = P.E, B = P.B;
  const int env_l = tid / M, drone = tid - env_l * M;
  const int env = blockIdx.x * E + env_l;
  const bool active = (env_l < E) && (env < P.N) && (P.reset_mask == nullptr || P.reset_mask[env] != 0);
  const long long g = (long long)env * M + drone;
  const int total = P.host_total >= 0 ? P.host_total : P.gsteps[0];
  const bool jit = (TASK == TASK_MULTIHOVER) && (P.reset_mode != RESET_FIXED);
  if (jit) {
    if (active && drone == 0) sample_jitter(P, env, total, P.reset_epoch, spos + (size_t)tid * 3);
    __syncthreads();
  }
  if (!active) return;
  Drone<R> d;
  float kin[12];
  reset_drone<R, TASK>(P, env, drone, jit ? spos + (size_t)tid * 3 : nullptr, d, kin);
  P.s0[g] = make4(d.px, d.py, d.pz, d.qx);
  P.s1[g] = make4(d.qy, d.qz, d.qw, d.vx);
  P.s2[g] = make4(d.vy, d.vz, d.wx, d.wy);
  P.s3[g] = make4(d.wz, d.tx, d.ty, d.tz);
  if (P.keep_angv) P.s4[g] = make4(R(0), R(0), R(0), R(0));
  if (drone == 0) { P.stepc[env] = 0; if (P.ep_ret != nullptr) P.ep_ret[env] = 0.f; }   // the ring head (total steps) is untouched by a reset
  if (P.ctrl != nullptr && P.ctrl_reset) {
    for (int k = 0; k < 9; ++k) P.ctrl[(size_t)k * P.n_total + g] = R(0);
  }
  if (P.obs != nullptr) {
    float* row = P.obs + (size_t)g * P.D;
    for (int k = 0; k < 12; ++k) row[k] = kin[k];
    const int head = total % B;   // oldest entry lives in slot `head`
    int slot = head;
    for (int j = 0; j < B; ++j) {
      const float* hp = P.hist + ((size_t)slot * P.n_total + g) * A;
      for (int k = 0; k < A; ++k) row[12 + j * A + k] = hp[k];
      slot = (slot + 1 == B) ? 0 : slot + 1;
    }
    if (TASK == TASK_SPIRAL) {
      R rp[3], rv[3], sphi, cphi;
      spiral_reference(P, 0, drone, rp, rv, sphi, cphi);
      spiral_extras(row + 12 + B * A, d, rp, rv, sphi, cphi);
    }
  }
}

template <typename R>
__global__ void get_state_kernel(const __grid_constant__ Params<R> P, R* state20, R* rates,
                                 int32_t* step_counter) {
  using R4 = typename V4<R>::type;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.n_total) return;
  const int env = (int)(g / P.M);
  const R4 a0 = P.s0[g], a1 = P.s1[g], a2 = P.s2[g], a3 = P.s3[g];
  const int stepc = P.stepc[env];
  const int head = (P.host_total >= 0 ? P.host_total : P.gsteps[0]) % P.B;
  if (state20 != nullptr) {
    R* o = state20 + g * 20;
    o[0] = a0.x; o[1] = a0.y; o[2] = a0.z;
    o[3] = a0.w; o[4] = a1.x; o[5] = a1.y; o[6] = a1.z;
    R roll, pitch, yaw;
    quat_to_euler(a0.w, a1.x, a1.y, a1.z, roll, pitch, yaw);
    o[7] = roll; o[8] = pitch; o[9] = yaw;
    o[10] = a1.w; o[11] = a2.x; o[12] = a2.y;
    if (P.keep_angv) { const R4 av = P.s4[g]; o[13] = av.x; o[14] = av.y; o[15] = av.z; }
    else { const R nanv = R(nan("")); o[13] = o[14] = o[15] = nanv; }
    // last_clipped_action: rpm of the newest ring entry, zero right after a reset (:468)
    const int newest = head == 0 ? P.B - 1 : head - 1;
    const float* hp = P.hist + ((size_t)newest * P.n_total + g) * P.A;
    for (int k = 0; k < 4; ++k) {
      if (P.act_type >= ACT_PID) {
        o[16 + k] = stepc > 0 ? P.ctrl[(size_t)(9 + k) * P.n_total + g] : R(0);
        continue;
      }
      const float a = hp[P.A == 4 ? k : 0];
      const float s = __fadd_rn(1.0f, __fmul_rn(0.05f, a));
      o[16 + k] = stepc > 0 ? P.hover_rpm * (R)s : R(0);
    }
  }
  if (rates != nullptr) { rates[g * 3] = a2.z; rates[g * 3 + 1] = a2.w; rates[g * 3 + 2] = a3.x; }
  if (step_counter != nullptr && g % P.M == 0) step_counter[env] = stepc;
}

template <typename R>
__global__ void set_state_kernel(const __grid_constant__ Params<R> P, const R* kin13,
                                 const R* targets, const int32_t* step_counter) {
  using R4 = typename V4<R>::type;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.n_total) return;
  const int env = (int)(g / P.M);
  if (kin13 != nullptr) {
    const R* k = kin13 + g * 13;
    const R4 old3 = P.s3[g];
    P.s0[g] = make4(k[0], k[1], k[2], k[3]);
    P.s1[g] = make4(k[4], k[5], k[6], k[7]);
    P.s2[g] = make4(k[8], k[9], k[10], k[11]);
    P.s3[g] = make4(k[12], old3.y, old3.z, old3.w);
    if (P.keep_angv) P.s4[g] = make4(R(0), R(0), R(0), R(0));
  }
  if (targets != nullptr) {
    const R4 old3 = P.s3[g];
    P.s3[g] = make4(old3.x, targets[g * 3], targets[g * 3 + 1], targets[g * 3 + 2]);
  }
  if (step_counter != nullptr && g % P.M == 0) {
    P.stepc[env] = step_counter[env];
  }
}

// Simulator snapshot, both directions (bd_save_snapshot / bd_load_snapshot).  One thread per drone: the four (five)
// state planes as 128-bit (Real4) accesses, the controller planes, and the B ring slots stored by AGE (age a = ring slot
// (total-1-a) mod B of this handle), each age plane copied coalesced over drones; threads g < N also carry env g's step
// counter and episode return.  A masked load touches only the drones / envs with mask[env] != 0.
template <typename R>
__global__ void __launch_bounds__(256)
snapshot_kernel(const __grid_constant__ Params<R> P, unsigned char* snap, const __grid_constant__ SnapLayout L,
                const __grid_constant__ SnapHeader hdr, const uint8_t* mask, int save, int full) {
  using R4 = typename V4<R>::type;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int total = P.host_total >= 0 ? P.host_total : P.gsteps[0];
  if (g == 0) {
    SnapHeader* h = reinterpret_cast<SnapHeader*>(snap);
    if (save) {
      SnapHeader o = hdr;
      o.rng[1] = (uint64_t)(uint32_t)(P.philox_base + (uint32_t)total);   // the device count in graph mode
      for (int k = 0; k < 3; ++k) o.ep_acc[k] = P.ep_acc[k];
      *h = o;
    } else if (full) {
      for (int k = 0; k < 3; ++k) P.ep_acc[k] = h->ep_acc[k];
    }
  }
  if (g < P.N && (save || mask == nullptr || mask[g])) {
    int* sc = reinterpret_cast<int*>(snap + L.stepc);
    float* er = L.ep_ret >= 0 ? reinterpret_cast<float*>(snap + L.ep_ret) : nullptr;
    if (save) {
      sc[g] = P.stepc[g];
      if (er != nullptr) er[g] = P.ep_ret[g];
    } else {
      P.stepc[g] = sc[g];
      if (P.ep_ret != nullptr) P.ep_ret[g] = er[g];   // the host refused a snapshot without the plane
    }
  }
  if (g >= P.n_total) return;
  if (!save && mask != nullptr && !mask[g / P.M]) return;
  R4* k0 = reinterpret_cast<R4*>(snap + L.kin[0]);
  R4* k1 = reinterpret_cast<R4*>(snap + L.kin[1]);
  R4* k2 = reinterpret_cast<R4*>(snap + L.kin[2]);
  R4* k3 = reinterpret_cast<R4*>(snap + L.kin[3]);
  R4* av = L.angv >= 0 ? reinterpret_cast<R4*>(snap + L.angv) : nullptr;
  const int A = P.A, B = P.B;
  const int newest = (int)(((long long)total + B - 1) % B);
  if (save) {
    k0[g] = P.s0[g]; k1[g] = P.s1[g]; k2[g] = P.s2[g]; k3[g] = P.s3[g];
    if (av != nullptr) av[g] = P.s4[g];
  } else {
    P.s0[g] = k0[g]; P.s1[g] = k1[g]; P.s2[g] = k2[g]; P.s3[g] = k3[g];
    if (P.keep_angv) P.s4[g] = av[g];
  }
  if (P.ctrl != nullptr) {
    for (int k = 0; k < kCtrlPlanesHost; ++k) {
      R* c = reinterpret_cast<R*>(snap + L.ctrl + k * L.ctrl_stride);
      R* s = P.ctrl + (size_t)k * P.n_total;
      if (save) c[g] = s[g]; else s[g] = c[g];
    }
  }
  for (int a = 0; a < B; ++a) {
    int slot = newest - a;
    if (slot < 0) slot += B;
    float* hs = P.hist + ((size_t)slot * P.n_total + g) * A;
    float* rs = reinterpret_cast<float*>(snap + L.ring + a * L.ring_stride) + g * A;
    const float* src = save ? hs : rs;
    float* dst = save ? rs : hs;
    if (A == 4) {
      *reinterpret_cast<float4*>(dst) = *reinterpret_cast<const float4*>(src);
    } else {
      for (int k = 0; k < A; ++k) dst[k] = src[k];
    }
  }
}

// DSL PID memory (N,M,9): [integral_pos_e, integral_rpy_e, last_rpy]; src == nullptr zeroes it
// (DSLPIDControl.reset, DSLPIDControl.py:64-79)
template <typename R>
__global__ void ctrl_state_kernel(const __grid_constant__ Params<R> P, R* dst, const R* src, int write) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.n_total) return;
  for (int k = 0; k < 9; ++k) {
    if (write) P.ctrl[(size_t)k * P.n_total + g] = src != nullptr ? src[g * 9 + k] : R(0);
    else dst[g * 9 + k] = P.ctrl[(size_t)k * P.n_total + g];
  }
}

template <typename R>
__global__ void get_targets_kernel(const __grid_constant__ Params<R> P, R* targets) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.n_total) return;
  const auto a3 = P.s3[g];
  targets[g * 3] = a3.y; targets[g * 3 + 1] = a3.z; targets[g * 3 + 2] = a3.w;
}

// =========================================================================
//                              host-side dispatch
// =========================================================================
size_t step_smem_bytes(int precision, int A, int B, int D, int task) {
  (void)A; (void)B;
  const size_t real = precision ? 8 : 4;
  const size_t tile = ((size_t)kBlock * D * 4 + 15) & ~(size_t)15;
  const size_t swarm = task >= TASK_SWARM ? (size_t)kBlock * real * 4 : 0;   // svel + saux
  return tile + (size_t)kBlock * real * 4 + (size_t)kBlock * 8 + swarm;
}

template <typename R, int TASK, int A, bool GENERIC>
static cudaError_t launch_step_t(const Params<R>& P, const LaunchSpec& ls, cudaStream_t st) {
  const int device = ls.device;
  const size_t smem = step_smem_bytes(sizeof(R) == 8, A, P.B, P.D, P.task);
  auto kern = step_kernel<R, TASK, A, GENERIC>;
  static size_t configured[64] = {0};   // per device: the attribute is per context
  static int per_sm[64] = {0};
  if (smem > configured[device & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured[device & 63] = smem;
    per_sm[device & 63] = 0;
  }
  const int grid = P.grid_blocks > 0 ? P.grid_blocks : (P.N + P.E - 1) / P.E;
  if (!P.pipeline) {
    kern<<<grid, kBlock, smem, st>>>(P);
    return cudaGetLastError();
  }
  int& occ = per_sm[device & 63];
  if (occ == 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kBlock, smem) != cudaSuccess || occ < 1) occ = 1;
  }
  Params<R> Q = P;
  Q.pipe_wait = (grid >= occ * ls.sm_count) ? 1 : 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kBlock);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, Q);
}

template <typename R, int TASK, int A>
static cudaError_t launch_reset_t(const Params<R>& P, cudaStream_t st) {
  const int grid = (P.N + P.E - 1) / P.E;
  reset_kernel<R, TASK, A><<<grid, kBlock, kBlock * 3 * sizeof(R), st>>>(P);
  return cudaGetLastError();
}

template <typename R, int TASK, int A>
static cudaError_t step_g(const LaunchSpec& ls, const void* p, cudaStream_t st) {
  const Params<R>& P = *static_cast<const Params<R>*>(p);
  if constexpr (sizeof(R) == 4) {
    if (ls.impl == 1) return launch_step_tile(TASK, A, P, ls, st);
  }
  return ls.generic ? launch_step_t<R, TASK, A, true>(P, ls, st)
                    : launch_step_t<R, TASK, A, false>(P, ls, st);
}
template <typename R, int TASK>
static cudaError_t step_a(const LaunchSpec& ls, const void* p, cudaStream_t st) {
  if (ls.act_a == 3)   // ActionType.PID: waypoint actions, always the generic kernel
    return launch_step_t<R, TASK, 3, true>(*static_cast<const Params<R>*>(p), ls, st);
  return ls.act_a == 4 ? step_g<R, TASK, 4>(ls, p, st) : step_g<R, TASK, 1>(ls, p, st);
}
template <typename R>
static cudaError_t step_t(const LaunchSpec& ls, const void* p, cudaStream_t st) {
  switch (ls.task) {
    case TASK_HOVER: return step_a<R, TASK_HOVER>(ls, p, st);
    case TASK_MULTIHOVER: return step_a<R, TASK_MULTIHOVER>(ls, p, st);
    case TASK_SPIRAL: return step_a<R, TASK_SPIRAL>(ls, p, st);
    default: {   // swarm tasks: the fast tile kernel where it applies, else the generic kernel (never the non-generic CTA kernel)
      const Params<R>& P = *static_cast<const Params<R>*>(p);
      if constexpr (sizeof(R) == 4) {
        if (ls.impl == 1 && ls.act_a != 3)
          return launch_step_tile(TASK_SWARM, ls.act_a, P, ls, st);
      }
      if (ls.act_a == 3) return launch_step_t<R, TASK_SWARM, 3, true>(P, ls, st);
      return ls.act_a == 4 ? launch_step_t<R, TASK_SWARM, 4, true>(P, ls, st)
                           : launch_step_t<R, TASK_SWARM, 1, true>(P, ls, st);
    }
  }
}
cudaError_t launch_step(const LaunchSpec& ls, const void* params, cudaStream_t st) {
  return ls.precision ? step_t<double>(ls, params, st) : step_t<float>(ls, params, st);
}

template <typename R, int TASK>
static cudaError_t reset_a(const LaunchSpec& ls, const void* p, cudaStream_t st) {
  const Params<R>& P = *static_cast<const Params<R>*>(p);
  if (ls.act_a == 3) return launch_reset_t<R, TASK, 3>(P, st);
  return ls.act_a == 4 ? launch_reset_t<R, TASK, 4>(P, st) : launch_reset_t<R, TASK, 1>(P, st);
}
template <typename R>
static cudaError_t reset_t(const LaunchSpec& ls, const void* p, cudaStream_t st) {
  switch (ls.task) {
    case TASK_HOVER: return reset_a<R, TASK_HOVER>(ls, p, st);
    case TASK_MULTIHOVER: return reset_a<R, TASK_MULTIHOVER>(ls, p, st);
    case TASK_SPIRAL: return reset_a<R, TASK_SPIRAL>(ls, p, st);
    default: return reset_a<R, TASK_SWARM>(ls, p, st);
  }
}
cudaError_t launch_reset(const LaunchSpec& ls, const void* params, cudaStream_t st) {
  return ls.precision ? reset_t<double>(ls, params, st) : reset_t<float>(ls, params, st);
}

template <typename R>
static int flat_grid(const Params<R>& P) { return (int)((P.n_total + 255) / 256); }

cudaError_t launch_get_state(int precision, const void* p, void* state20, void* rates,
                             int32_t* step_counter, cudaStream_t st) {
  if (precision) {
    const auto& P = *static_cast<const Params<double>*>(p);
    get_state_kernel<double><<<flat_grid(P), 256, 0, st>>>(P, (double*)state20, (double*)rates, step_counter);
  } else {
    const auto& P = *static_cast<const Params<float>*>(p);
    get_state_kernel<float><<<flat_grid(P), 256, 0, st>>>(P, (float*)state20, (float*)rates, step_counter);
  }
  return cudaGetLastError();
}

cudaError_t launch_set_state(int precision, const void* p, const void* kin13, const void* targets,
                             const int32_t* step_counter, cudaStream_t st) {
  if (precision) {
    const auto& P = *static_cast<const Params<double>*>(p);
    set_state_kernel<double><<<flat_grid(P), 256, 0, st>>>(P, (const double*)kin13, (const double*)targets, step_counter);
  } else {
    const auto& P = *static_cast<const Params<float>*>(p);
    set_state_kernel<float><<<flat_grid(P), 256, 0, st>>>(P, (const float*)kin13, (const float*)targets, step_counter);
  }
  return cudaGetLastError();
}

cudaError_t launch_ctrl_state(int precision, const void* p, void* dst, const void* src, int write, cudaStream_t st) {
  if (precision) {
    const auto& P = *static_cast<const Params<double>*>(p);
    ctrl_state_kernel<double><<<flat_grid(P), 256, 0, st>>>(P, (double*)dst, (const double*)src, write);
  } else {
    const auto& P = *static_cast<const Params<float>*>(p);
    ctrl_state_kernel<float><<<flat_grid(P), 256, 0, st>>>(P, (float*)dst, (const float*)src, write);
  }
  return cudaGetLastError();
}

cudaError_t launch_snapshot(int precision, const void* p, void* snap, const SnapLayout& L, const SnapHeader& hdr,
                            const uint8_t* mask, int save, int full, cudaStream_t st) {
  unsigned char* s = static_cast<unsigned char*>(snap);
  if (precision) {
    const auto& P = *static_cast<const Params<double>*>(p);
    snapshot_kernel<double><<<flat_grid(P), 256, 0, st>>>(P, s, L, hdr, mask, save, full);
  } else {
    const auto& P = *static_cast<const Params<float>*>(p);
    snapshot_kernel<float><<<flat_grid(P), 256, 0, st>>>(P, s, L, hdr, mask, save, full);
  }
  return cudaGetLastError();
}

__global__ void episode_stats_kernel(double* acc, double* out3, int reset) {
  if (threadIdx.x < 3) {
    if (out3 != nullptr) out3[threadIdx.x] = acc[threadIdx.x];
    if (reset) acc[threadIdx.x] = 0.0;
  }
}
cudaError_t launch_episode_stats(double* ep_acc, double* out3, int reset, cudaStream_t st) {
  episode_stats_kernel<<<1, 32, 0, st>>>(ep_acc, out3, reset);
  return cudaGetLastError();
}

// ---- compact terminal observations (subproc_vec_env.py:195-206: only finished envs carry one) ----------
// Works on an env range [e0, e1) (one chunk of bd_step_host's pipeline, so the compaction of chunk k hides behind the
// device->host copy of its observations): pass 1 counts the finished envs per block of kCompactBlock envs, pass 2 turns
// the counts into offsets (running total of the earlier chunks in *total + the counts of the blocks before it), scans
// its own flags and copies the finished envs' (M,D) rows — in ascending env order, so the result is deterministic — to
// `rows_out` (at most `cap` envs) and their indices to `idx_out[1..]`; pass 3 adds the chunk's count to *total and
// mirrors it to idx_out[0].  The outputs may live in mapped pinned host memory.
constexpr int kCompactBlock = 1024;
__global__ void __launch_bounds__(kCompactBlock)
count_done_kernel(const uint8_t* __restrict__ term, const uint8_t* __restrict__ trunc, int e0, int e1, int* __restrict__ blockcnt) {
  const int e = e0 + blockIdx.x * kCompactBlock + threadIdx.x;
  const int done = (e < e1) && (term[e] | trunc[e]);
  const int c = __syncthreads_count(done);
  if (threadIdx.x == 0) blockcnt[blockIdx.x] = c;
}
__global__ void __launch_bounds__(kCompactBlock)
gather_done_kernel(const uint8_t* __restrict__ term, const uint8_t* __restrict__ trunc, int e0, int e1,
                   const int* __restrict__ blockcnt, const int* __restrict__ total, const float* __restrict__ tobs,
                   int row_floats, int cap, int* __restrict__ idx_out, float* __restrict__ rows_out) {
  __shared__ int s_warp[kCompactBlock / 32];
  __shared__ int s_base;
  __shared__ int s_list[kCompactBlock];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int before = 0;
  for (int b = tid; b < (int)blockIdx.x; b += kCompactBlock) before += blockcnt[b];
  for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
  if (tid == 0) s_base = *total;
  __syncthreads();
  if (lane == 0 && before != 0) atomicAdd(&s_base, before);
  const int e = e0 + blockIdx.x * kCompactBlock + tid;
  const int done = (e < e1) && (term[e] | trunc[e]);
  const unsigned bal = __ballot_sync(0xffffffffu, done);
  if (lane == 0) s_warp[warp] = __popc(bal);
  __syncthreads();
  int woff = 0, mine = 0;
  for (int w = 0; w < kCompactBlock / 32; ++w) { if (w < warp) woff += s_warp[w]; mine += s_warp[w]; }
  const int pos = woff + __popc(bal & ((1u << lane) - 1u));
  if (done) s_list[pos] = e;
  __syncthreads();
  const int base = s_base;
  for (int k = tid; k < mine; k += kCompactBlock)
    if (base + k < cap) idx_out[1 + base + k] = s_list[k];
  // rows: the block copies its finished envs one after the other, 128-bit where the row allows it
  for (int k = 0; k < mine; ++k) {
    if (base + k >= cap) break;
    const float* src = tobs + (size_t)s_list[k] * row_floats;
    float* dst = rows_out + (size_t)(base + k) * row_floats;
    if ((row_floats & 3) == 0 && ((((uintptr_t)src) | ((uintptr_t)dst)) & 15) == 0) {
      for (int i = tid; i < row_floats / 4; i += kCompactBlock)
        reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(src)[i];
    } else {
      for (int i = tid; i < row_floats; i += kCompactBlock) dst[i] = src[i];
    }
  }
}
__global__ void compact_total_kernel(const int* __restrict__ blockcnt, int blocks, int* __restrict__ total, int* __restrict__ idx_out,
                                     int reset_first) {
  int c = 0;
  for (int b = threadIdx.x; b < blocks; b += 32) c += blockcnt[b];
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (threadIdx.x == 0) {
    const int t = (reset_first ? 0 : *total) + c;
    *total = t;
    idx_out[0] = t;
  }
}
int compact_blocks(int n) { return (n + kCompactBlock - 1) / kCompactBlock; }
// reset_total: 1 for the first chunk of a step (the running total restarts at 0)
cudaError_t launch_compact_done(const uint8_t* term, const uint8_t* trunc, int e0, int e1, int reset_total, int* blockcnt, int* total,
                                const float* tobs, int row_floats, int cap, int* idx_out, float* rows_out, cudaStream_t st) {
  const int blocks = compact_blocks(e1 - e0);
  if (reset_total) {
    cudaError_t e = cudaMemsetAsync(total, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
  }
  if (blocks > 0) {
    count_done_kernel<<<blocks, kCompactBlock, 0, st>>>(term, trunc, e0, e1, blockcnt);
    gather_done_kernel<<<blocks, kCompactBlock, 0, st>>>(term, trunc, e0, e1, blockcnt, total, tobs, row_floats, cap, idx_out, rows_out);
  }
  compact_total_kernel<<<1, 32, 0, st>>>(blockcnt, blocks, total, idx_out, 0);
  return cudaGetLastError();
}

__global__ void set_epoch_kernel(int* tile_epoch, int tile, int value) { tile_epoch[tile] = value; }
__global__ void gate_kernel(const uint32_t* flag) {
  const long long t0 = clock64();
  while (*reinterpret_cast<const volatile uint32_t*>(flag) == 0u) {
    __nanosleep(500);
    if (clock64() - t0 > (1LL << 32)) break;
  }
}
cudaError_t launch_gate(const uint32_t* flag_mapped, cudaStream_t st) {
  gate_kernel<<<1, 1, 0, st>>>(flag_mapped);
  return cudaGetLastError();
}

cudaError_t launch_set_epoch(int* tile_epoch, int tile, int value, cudaStream_t st) {
  set_epoch_kernel<<<1, 1, 0, st>>>(tile_epoch, tile, value);
  return cudaGetLastError();
}

cudaError_t launch_get_targets(int precision, const void* p, void* targets, cudaStream_t st) {
  if (precision) {
    const auto& P = *static_cast<const Params<double>*>(p);
    get_targets_kernel<double><<<flat_grid(P), 256, 0, st>>>(P, (double*)targets);
  } else {
    const auto& P = *static_cast<const Params<float>*>(p);
    get_targets_kernel<float><<<flat_grid(P), 256, 0, st>>>(P, (float*)targets);
  }
  return cudaGetLastError();
}

}  // namespace bd
