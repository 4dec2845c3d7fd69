// Internal kernel-parameter block shared by bd_kernels.cu and bd_api.cu.
// Not part of the public ABI (that is include/batch_drones.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bd {

constexpr int kBlock = 128;        // threads per CTA; one thread per drone
constexpr int kMaxDrones = 128;    // M <= kBlock (an env never straddles CTAs)
constexpr int kMaxJitterTries = 64;
constexpr int kCtrlPlanesHost = 13;  // 9 DSL PID memory planes + 4 commanded-rpm planes (bd_device.cuh)

template <typename Real> struct V4;
template <> struct V4<float>  { using type = float4;  };
template <> struct V4<double> { using type = double4; };

// Device-resident SoA drone state (see DESIGN.md "HBM layout").
//   s0[g] = (px, py, pz, qx)   s1[g] = (qy, qz, qw, vx)
//   s2[g] = (vy, vz, wx, wy)   s3[g] = (wz, tx, ty, tz)      t = TARGET_POS
//   s4[g] = (avx, avy, avz, -) world angular velocity, only with keep_ang_vel
//   hist[slot][g][A]           float action ring, B slots (survives reset,
//                              BaseRLAviary.py:153-154,187)
//   stepc[e]                   step_counter since the env's last reset (BaseAviary.py:382,460)
//   gsteps[0] = total control steps taken (ring head = total % B, Philox stream), gsteps[1] = CTA ticket
template <typename Real>
struct Params {
  int N, M, S, A, B, D, E;
  int EW;                         // fast tile kernel: whole envs per warp (32 / M)
  long long n_total;
  typename V4<Real>::type *s0, *s1, *s2, *s3, *s4;
  float* hist;
  int* stepc;
  int* gsteps;
  float* ep_ret;                  // running episode return per env (VecRecordEpisodeStatistics, :144-171)
  double* ep_acc;                 // [3] sums over finished episodes: return, length, count
  Real* ctrl;                     // [13][n_total] DSL PID memory + commanded rpm (PID action types), else nullptr
  const Real* init_xyz;
  const Real* init_rpy;
  int init_env_stride;            // 0 (shared (M,3) table) or M*3
  const Real* jitter;             // (N,M,3) or nullptr
  // per-call I/O
  const void* actions;
  float* obs;
  Real* reward;
  uint8_t* terminated;
  uint8_t* truncated;
  float* terminal_obs;
  const uint8_t* reset_mask;
  // constants
  Real dt, hover_rpm, kf, km, arm, inv_m, gravity;
  Real jx, jy, jz, ijx, ijy, ijz;
  Real gnd_coeff, prop_radius, gnd_h_clip, drag_xy, drag_z, dw1, dw2, dw3;
  Real prop_x[4], prop_y[4];
  Real sp_R, sp_omega, sp_vz, sp_cx, sp_cy;
  double pyb_freq, episode_len;
  int trunc_counter;              // smallest step_counter with step_counter / pyb_freq > episode_len (fp64)
  int model, aero, integrator, auto_reset, reset_mode, action_is_f32, keep_angv;
  int task;                       // BD_TASK_* (the swarm tasks share one kernel instantiation and branch on this)
  int act_type, ctrl_reset;       // ACT_*; 1: env resets also zero the controller memory (reference: never)
  Real ctrl_dt, ctrl_gravity, ctrl_4kf, speed_limit;   // DSLPIDControl constants (CF2X), BaseRLAviary.py:95
  float speed_limit_f;
  int host_total;                 // >= 0: total control steps so far, tracked by the host (ring head with no
                                  // memory latency); -1: read gsteps[0] (CUDA-graph capture / replay)
  int host_head;                  // host_total % B when host_total >= 0
  int total_wrap;                 // step counters wrap at this multiple of B (ring head stays continuous)
  int* tile_epoch;                // [tiles] control steps completed per tile (tile-level step pipelining)
  unsigned long long* finished;   // tiles finished since creation, all steps (== total * step_tiles: previous step complete)
  long long step_tiles;           // tiles of one whole control step with this handle's kernel
  int pipeline;                   // 1: the handle pipelines steps tile by tile: every launch publishes tile epochs
  int pipe_wait;                  // 1: this launch waits for MY tile's previous step only (no grid-wide dependency wait)
  int early_prefetch;             // 1: ring planes may be prefetched before griddepcontrol.wait (grid >= resident capacity).
                                  // Host side 0 forbids it for one launch (the first step after bd_load_snapshot, whose
                                  // unpack kernel wrote those planes); launch_step_tile decides the value the kernel sees
  int block0, grid_blocks;        // sub-range launch: first tile and tile count (0 = all tiles)
  int advance;                    // 1: this launch advances the device-resident step count (last chunk of a step)
  int reset_epoch;                // >=1 for explicit bd_reset calls (Philox stream id), 0 in-step
  unsigned long long seed;
  int obs_aligned;                // 1: the caller's observation pointer is 16-byte aligned (bulk / 128-bit row stores allowed)
  uint32_t philox_base;           // added to the step count in the Philox counter (bd_set_rng_state: resumed runs continue the stream)
  // fast tile kernel's L2 residency budget (bd_l2_plan, DESIGN.md section 4): state planes, step counter and episode
  // return evict_last; ring slots younger than l2_keep_slots (0 .. B-1) evict_last, older ones evict_first
  int l2_keep_state;
  int l2_keep_slots;
};

// Simulator snapshot (bd_save_snapshot / bd_load_snapshot, include/batch_drones.h): a 256-byte header, then SoA planes,
// each starting on a 256-byte boundary, in this order: s0..s3, [s4], [13 controller planes], B ring planes by age,
// step counters, [episode returns].
constexpr uint32_t kSnapMagic = 0x4e534442u;   // "BDSN"
constexpr uint32_t kSnapVersion = 1;
constexpr long long kSnapAlign = 256;
struct SnapHeader {
  uint32_t magic, version;
  int32_t precision, n_envs, n_drones, act_dim, buf_slots;
  uint32_t flags;                 // BD_SNAP_* planes present
  uint64_t fingerprint;           // configuration that must match on restore (bd_api.cu: snap_fingerprint)
  int64_t bytes;                  // whole snapshot, header included
  uint64_t rng[4];                // bd_get_rng_state of the saving handle
  double ep_acc[3];               // episode accumulators (bd_episode_stats)
  int32_t task, act_type, drone_model, aero_flags, integrator, pyb_freq, ctrl_freq, reserved0;
  uint8_t reserved[120];
};
static_assert(sizeof(SnapHeader) == 256, "snapshot header is 256 bytes");
// byte offsets of the planes; -1 = not present
struct SnapLayout {
  long long kin[4], angv, ctrl, ctrl_stride, ring, ring_stride, stepc, ep_ret, bytes;
};
// host computation shared by bd_snapshot_layout and the handle calls (bd_api.cu)
SnapLayout snap_layout(long long n_envs, long long n_drones, int act_dim, int buf_slots, int real_bytes, int flags);

struct LaunchSpec {
  int task, act_a, precision, generic, device;
  int pdl;         // launch the fast kernel with programmatic stream serialization
  int impl;        // 0: two-role CTA kernel (any config), 1: fast tile kernel (bd_step_tile.cuh)
  int sm_count;    // SMs of the device (resident-CTA capacity of the fast kernel)
};

// implemented in bd_tile_launch.cu (fast tile kernel; task = template TASK value, act_a in {1, 4})
cudaError_t launch_step_tile(int task, int act_a, const Params<float>& P, const LaunchSpec& ls, cudaStream_t st);
// k control steps in one launch (step_kernel_tile_many); strides in elements between consecutive steps' slots
cudaError_t launch_step_tile_many(int task, int act_a, const Params<float>& P, int k, long long act_step, long long obs_step,
                                  long long out_step, const LaunchSpec& ls, cudaStream_t st);
// implemented in bd_kernels.cu
cudaError_t launch_step(const LaunchSpec& ls, const void* params, cudaStream_t st);
cudaError_t launch_reset(const LaunchSpec& ls, const void* params, cudaStream_t st);
cudaError_t launch_get_state(int precision, const void* params, void* state20, void* rates,
                             int32_t* step_counter, cudaStream_t st);
cudaError_t launch_set_state(int precision, const void* params, const void* kin13,
                             const void* targets, const int32_t* step_counter, cudaStream_t st);
cudaError_t launch_get_targets(int precision, const void* params, void* targets, cudaStream_t st);
cudaError_t launch_ctrl_state(int precision, const void* params, void* dst, const void* src, int write,
                              cudaStream_t st);
cudaError_t launch_episode_stats(double* ep_acc, double* out3, int reset, cudaStream_t st);
// save = 1: state -> snapshot (header written from `hdr`, ep_acc and the Philox counter filled in on the device);
// save = 0: snapshot -> state for the envs with mask[e] != 0 (all when NULL); full = 1 also restores ep_acc
cudaError_t launch_snapshot(int precision, const void* params, void* snap, const SnapLayout& L, const SnapHeader& hdr,
                            const uint8_t* mask, int save, int full, cudaStream_t st);
size_t step_smem_bytes(int precision, int A, int B, int D, int task);
int compact_blocks(int n);
cudaError_t launch_compact_done(const uint8_t* term, const uint8_t* trunc, int e0, int e1, int reset_total, int* blockcnt, int* total,
                                const float* tobs, int row_floats, int cap, int* idx_out, float* rows_out, cudaStream_t st);
cudaError_t launch_set_epoch(int* tile_epoch, int tile, int value, cudaStream_t st);
cudaError_t launch_gate(const uint32_t* flag_mapped, cudaStream_t st);

}  // namespace bd
