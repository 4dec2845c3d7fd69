/* batch_drones.h — C-ABI of the B200-native batched drone-step library.
 *
 * The reference (khuzema-h/marl-gym-pybullet-drones) is pure Python and has no
 * FFI for this path; the interface the path sits behind is
 *   - Gymnasium `reset/step` of the aviaries
 *       gym_pybullet_drones/envs/BaseAviary.py:220-255 (reset), :259-383 (step)
 *   - the VecEnv protocol the MAPPO rollout calls
 *       safe_control_gym/envs/env_wrappers/vectorized_env/subproc_vec_env.py:51-73,186-207
 * This header is what a ctypes binding placed under those two protocols binds
 * (see INTEGRATION.md for the stub).  Each entry point names the reference
 * code it replaces.
 *
 * Conventions
 *   - plain C, no torch types; every *_dev pointer is CALLER-OWNED DEVICE memory,
 *     every *_host pointer is host memory; the library owns only the drone state
 *     inside the handle.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *     All device entry points are stream-ordered, never synchronise, and are
 *     CUDA-graph capturable; bd_step_host() synchronises `stream` before returning.
 *   - "Real" = float when cfg.precision == BD_F32, double when BD_F64.
 *   - return 0 on success, a negative BD_E* code otherwise (never exit());
 *     bd_last_error() returns the message of the calling thread's last failure.
 *   - one handle per GPU; a handle is not thread-safe.
 *
 * Shapes: N = n_envs, M = n_drones, A = 4 (RPM, VEL), 3 (PID) or 1 (ONE_D_RPM, ONE_D_PID),
 *   B = ctrl_freq/2 (BaseRLAviary.py:66), D = 12 + B*A (+11 for the spiral task).
 */
#ifndef BATCH_DRONES_H_
#define BATCH_DRONES_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BD_VERSION 1

enum { BD_TASK_HOVER = 0, BD_TASK_MULTIHOVER = 1, BD_TASK_SPIRAL = 2,
       /* envs/MeetupAviary.py:74-154, FlockAviary.py:75-189, LeaderFollowerAviary.py:72-145 */
       BD_TASK_MEETUP = 3, BD_TASK_FLOCK = 4, BD_TASK_LEADERFOLLOWER = 5 };
/* ActionType (utils/enums.py:35-41).  PID / VEL / ONE_D_PID run the reference's DSLPIDControl
 * (control/DSLPIDControl.py:82-246) inside the step kernel, one controller per drone. */
enum { BD_ACT_RPM = 0, BD_ACT_ONE_D_RPM = 1, BD_ACT_PID = 2, BD_ACT_VEL = 3, BD_ACT_ONE_D_PID = 4 };
enum { BD_MODEL_CF2X = 0, BD_MODEL_CF2P = 1, BD_MODEL_RACE = 2 };
enum { BD_F32 = 0, BD_F64 = 1 };
enum { BD_AERO_GND = 1, BD_AERO_DRAG = 2, BD_AERO_DW = 4 };
enum { BD_INTEGRATOR_QUAT = 0, BD_INTEGRATOR_EULER = 1 };
enum { BD_RESET_FIXED = 0, BD_RESET_JITTER_PHILOX = 1, BD_RESET_JITTER_BUFFER = 2 };

enum {
  BD_OK = 0,
  BD_EINVAL = -1,   /* bad argument / unsupported configuration */
  BD_ECUDA = -2,    /* a CUDA runtime call failed                */
  BD_ENOMEM = -3    /* device or host allocation failed          */
};

/* Everything BaseAviary.__init__ / BaseRLAviary.__init__ / the task __init__
 * take or derive (BaseAviary.py:74-128, BaseRLAviary.py:66-67, HoverAviary.py:51-52,
 * MultiHoverAviary.py:58-72, SpiralAviary.py:39-56).  Airframe numbers are the
 * URDF <properties> (cf2x.urdf:5,11-12) parsed by the host language. */
typedef struct bd_config {
  int32_t struct_size;      /* = sizeof(bd_config), ABI guard                         */
  int32_t device;           /* CUDA device ordinal                                    */
  int32_t n_envs;           /* N                                                      */
  int32_t n_drones;         /* M (1..128); BD_TASK_HOVER requires 1                   */
  int32_t task;             /* BD_TASK_*                                              */
  int32_t act_type;         /* BD_ACT_*                                               */
  int32_t drone_model;      /* BD_MODEL_* (torque mixing, BaseAviary.py:846-854)      */
  int32_t precision;        /* BD_F32 fast mode | BD_F64 parity mode                  */
  int32_t aero_flags;       /* BD_AERO_* bits on top of DYN                           */
  int32_t integrator;       /* BD_INTEGRATOR_QUAT (BaseAviary.py:879-892) or _EULER
                               (safe_control_gym/.../base_aviary.py:499-508)          */
  int32_t pyb_freq;         /* BaseAviary.py:78                                       */
  int32_t ctrl_freq;        /* BaseAviary.py:77; pyb_freq % ctrl_freq must be 0       */
  int32_t auto_reset;       /* 1: SubprocVecEnv semantics (subproc_vec_env.py:195-206) */
  int32_t reset_mode;       /* BD_RESET_*; JITTER_* = MultiHoverAviary.py:83-102      */
  int32_t action_is_f32;    /* BD_F64 only: actions are float (numpy computes
                               1+0.05*a in float32 then), else double                 */
  int32_t keep_ang_vel;     /* 1: keep world angular velocity for bd_get_state        */
  int32_t track_episodes;   /* 1: accumulate episode returns/lengths (bd_episode_stats) */
  int32_t ctrl_reset_on_reset; /* PID action types: 1 = an env reset also clears its drones' controller
                               memory; 0 = reference behaviour, the controllers are built once in
                               BaseRLAviary.__init__ (:73-78) and never reset by env.reset()   */
  uint64_t seed;            /* Philox key for BD_RESET_JITTER_PHILOX                  */
  double episode_len_sec;   /* 12 (spiral) / 8 (every other task)                     */
  /* airframe */
  double mass, arm, kf, km, ixx, iyy, izz, g;
  double thrust2weight, gnd_eff_coeff, prop_radius, drag_coeff_xy, drag_coeff_z;
  double dw_coeff_1, dw_coeff_2, dw_coeff_3;
  double prop_xy[8];        /* x0,y0,...,x3,y3 body-frame propeller offsets            */
  /* spiral task (SpiralAviary.py:33-45) */
  double spiral_radius, spiral_period, height_rate, target_center[3];
  /* PID action types: the controller is always DSLPIDControl(DroneModel.CF2X)
   * (BaseRLAviary.py:76), so its mass / kf are CF2X's (BaseControl.py:35-37), not the env's */
  double ctrl_mass, ctrl_kf;
  double speed_limit;       /* VEL: 0.03 * MAX_SPEED_KMH * 1000/3600 (BaseRLAviary.py:95)     */
} bd_config;

typedef struct bd_handle bd_handle;

/* Replaces BaseAviary.__init__ + _housekeeping (BaseAviary.py:74-216, 451-505):
 * allocates the SoA drone state on cfg->device and puts every env in its
 * reset state with the default initial poses (BaseAviary.py:194-203; spiral
 * ring SpiralAviary.py:47-53). */
int bd_create(const bd_config* cfg, bd_handle** out);

/* Replaces BaseAviary.close / SubprocVecEnv.close. */
void bd_destroy(bd_handle* h);

/* INIT_XYZS / INIT_RPYS (BaseAviary.py:194-207).  Host arrays of doubles,
 * (M,3) when per_env == 0, (N,M,3) when per_env == 1; rpy_host may be NULL
 * (zeros).  Like the constructor (BaseAviary.py:212-214; MultiHoverAviary.py:72)
 * it also puts EVERY env into its reset state at exactly these poses (no
 * jitter, step counters zeroed, action history kept).  Synchronises. */
int bd_set_init_poses(bd_handle* h, const double* xyz_host, const double* rpy_host, int per_env);

/* Jitter draws for BD_RESET_JITTER_BUFFER: (N,M,3) Real in [-0.25,0.25), the
 * stand-in for np.random.uniform at MultiHoverAviary.py:83.  Copied (stream
 * ordered) into the handle; each env consumes its row at its next reset. */
int bd_set_jitter(bd_handle* h, const void* jitter_dev, void* stream);

/* Replaces env.reset() on every env with env_mask_dev[e] != 0 (all envs when
 * NULL): MultiHoverAviary.py:75-110 + BaseAviary.py:220-255.  Writes the reset
 * observation rows (float32, (N,M,D)) of those envs when obs_dev != NULL. */
int bd_reset(bd_handle* h, const uint8_t* env_mask_dev, float* obs_dev, void* stream);

/* Replaces one VecEnv.step(): BaseRLAviary._preprocessAction (BaseRLAviary.py:160-239),
 * BaseAviary.step's substep loop with _dynamics/_integrateQ (BaseAviary.py:343-374,
 * 815-892), _computeObs/_computeReward/_computeTerminated/_computeTruncated of the
 * task, the step-counter advance (:382) and, with auto_reset, the worker's
 * reset-on-done (subproc_vec_env.py:195-206).  ONE kernel launch.
 *   actions_dev      (N,M,A) float (double when BD_F64 && !action_is_f32)
 *   obs_dev          (N,M,D) float; for envs that were auto-reset this is the RESET obs
 *   reward_dev       (N) Real
 *   terminated_dev   (N) uint8, truncated_dev (N) uint8
 *   terminal_obs_dev (N,M,D) float or NULL; rows are written only for envs that
 *                    finished in this step (info['terminal_observation'])       */
int bd_step(bd_handle* h, const void* actions_dev, float* obs_dev, void* reward_dev,
            uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev,
            void* stream);

/* Same as bd_step with HOST buffers: copies the actions up, steps, copies
 * obs/reward/flags (and terminal obs when not NULL) back and synchronises
 * `stream`.  Buffers should be page-locked for full PCIe rate.  Above ~4 MB of
 * observations the step runs as a pipeline of up to 8 chunks of whole tiles on two
 * internal streams (actions up + sub-range launch of the step kernel | observations
 * down), so the device->host copy — the bound of this call — overlaps everything
 * else; results are identical to bd_step. */
int bd_step_host(bd_handle* h, const void* actions_host, float* obs_host, void* reward_host,
                 uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host,
                 void* stream);

/* bd_step_host with COMPACT terminal observations — what SubprocVecEnv's workers actually send
 * (subproc_vec_env.py:195-206: only an env that finished carries info['terminal_observation']).
 * Terminal rows stay on the device; after the step two small kernels gather the finished envs' (M,D)
 * rows, in ascending env order, into page-locked memory owned by the handle, so the device->host
 * traffic is obs + flags + n_done rows instead of a second full (N,M,D) buffer.
 *   *n_done        number of envs that finished in this step
 *   *done_idx      their env indices (ascending), n_done entries
 *   *terminal_rows (n_done, M, D) float, row k belongs to env (*done_idx)[k]
 * The two arrays are owned by the handle (two sets used alternately) and stay valid until the
 * next-but-one step call. */
int bd_step_host_compact(bd_handle* h, const void* actions_host, float* obs_host, void* reward_host,
                         uint8_t* terminated_host, uint8_t* truncated_host, int32_t* n_done,
                         const int32_t** done_idx, const float** terminal_rows, void* stream);

/* k control steps with ONE host call (the launch-bound regime: small batches, random-action sweeps —
 * BASELINE configs[3] as literally sharded is 8192 envs per GPU).  actions_dev (k,N,M,A), obs_dev
 * (k,N,M,D), reward_dev (k,N) Real, terminated_dev / truncated_dev (k,N) uint8; step i reads
 * action set i and writes output slot i.  Results identical to k bd_step calls (no terminal observations).
 * On the fast float kernel the k steps are ONE launch (a tile's states stay in registers and its action
 * history in shared memory from step to step; only actions come in and observations / rewards / flags go
 * out); other configurations run k launches.  bd_set_step_many_mode(h, 1) forces k launches. */
int bd_step_many(bd_handle* h, int k, const void* actions_dev, float* obs_dev, void* reward_dev,
                 uint8_t* terminated_dev, uint8_t* truncated_dev, void* stream);
int bd_set_step_many_mode(bd_handle* h, int mode);
/* Benchmark helper: holds `stream` until the host stores a non-zero value into *flag_mapped (page-locked host memory,
 * mapped device address); gives up after ~2 s.  A timed window enqueued behind it has no host-side gaps. */
int bd_stream_gate(const uint32_t* flag_mapped, void* stream);

/* RNG state of the on-device re-spawn draws — the counterpart of the workers' np.random states the
 * reference checkpoints and restores (mappo/mappo.py:203-229; subproc_vec_env.py:101-112
 * get_env_random_state / set_env_random_state).  state4 = {Philox key (seed), Philox step counter,
 * explicit-reset epoch, 0}.  After bd_set_rng_state a resumed run continues the random stream
 * instead of replaying it.  BD_EINVAL once a step has been captured into a CUDA graph. */
int bd_get_rng_state(const bd_handle* h, uint64_t* state4);
int bd_set_rng_state(bd_handle* h, const uint64_t* state4);

/* Test hook for the tile-epoch protocol (DESIGN.md section 4): overwrite one tile's epoch, stream
 * ordered.  A CTA that waits for an epoch nobody publishes traps after ~1 s instead of hanging. */
int bd_debug_set_tile_epoch(bd_handle* h, int tile, int value, void* stream);

/* Replaces BaseAviary._getDroneStateVector (BaseAviary.py:541-561) for every
 * drone: state20_dev (N,M,20) Real = [pos3 quat4 rpy3 vel3 ang_v3 last_rpm4];
 * ang_v is NaN unless cfg.keep_ang_vel.  Optional: body rates `self.rpy_rates`
 * (N,M,3) Real and the per-env step counter (N) int32. */
int bd_get_state(bd_handle* h, void* state20_dev, void* rates_dev, int32_t* step_counter_dev,
                 void* stream);

/* Inject a state (parity tests, curriculum starts): kin13_dev (N,M,13) Real =
 * [pos3 quat4(xyzw) vel3 body_rates3]; optional targets_dev (N,M,3) Real
 * (TARGET_POS) and step_counter_dev (N) int32.  Quaternions are taken as given. */
int bd_set_state(bd_handle* h, const void* kin13_dev, const void* targets_dev,
                 const int32_t* step_counter_dev, void* stream);

/* TARGET_POS of every drone, (N,M,3) Real (MultiHoverAviary.py:72,106). */
int bd_get_targets(bd_handle* h, void* targets_dev, void* stream);

/* Replaces VecRecordEpisodeStatistics (record_episode_statistics.py:144-171) for envs that live
 * on the device: stats3_dev[0..2] = sum of returns, sum of lengths and number of the episodes that
 * finished since the last reset of the accumulators (per-step return = the env's scalar reward).
 * stats3_dev may be NULL (reset only).  Stream ordered.  Needs cfg.track_episodes = 1. */
int bd_episode_stats(bd_handle* h, double* stats3_dev, int reset, void* stream);

/* DSL PID controller memory of every drone, (N,M,9) Real =
 * [integral_pos_e(3), integral_rpy_e(3), last_rpy(3)] (DSLPIDControl.py:64-79).
 * bd_set_controller_state(NULL) zeroes it = `ctrl[k].reset()` on every drone.
 * BD_EINVAL for the RPM action types. */
int bd_get_controller_state(bd_handle* h, void* ctrl9_dev, void* stream);
int bd_set_controller_state(bd_handle* h, const void* ctrl9_dev, void* stream);

/* BD_F64 handles only: switch between float32 and float64 action input (see
 * bd_config.action_is_f32).  numpy evaluates HOVER_RPM*(1+0.05*a) partly in float32
 * when the policy hands float32 actions to the reference (BaseRLAviary.py:192). */
int bd_set_action_f32(bd_handle* h, int is_f32);

/* L2 residency plan of the fast step kernel (DESIGN.md section 4).  Between two steps of a tile the
 * state planes, step counters and episode returns (*keep_state = 1) and the keep_slots newest action-ring
 * slots (*keep_slots, 0 .. buf_slots-1) are marked evict_last; everything read for the last time is marked
 * evict_first.  The budget rule keeps the state first, then as many slots as fit, in what the device's L2
 * (l2_bytes) can hold; *keep_state = 0 when the state alone does not fit.  `force` is the BD_L2_KEEP
 * override ("off", "state", or a slot count k: the state plus k slots) or NULL.  Host computation only;
 * BD_EINVAL for a malformed override or shape.  bd_create runs it with the device's L2 size and BD_L2_KEEP. */
int bd_l2_plan(int n_envs, int n_drones, int act_dim, int buf_slots, int track_episodes, int64_t l2_bytes,
               const char* force, int* keep_state, int* keep_slots);
/* The plan a handle's step kernel runs with (both 0 when the handle does not use the fast tile kernel). */
int bd_l2_policy(const bd_handle* h, int* keep_state, int* keep_slots);

/* Snapshot of the complete simulator state, for checkpoints that resume mid-episode and for branching / replay from a
 * state.  An opaque, versioned byte buffer in CALLER-OWNED device memory (256-byte aligned): a 256-byte header (magic,
 * format version 1, precision, N, M, A, B, plane flags, configuration fingerprint, the bd_get_rng_state 4-tuple, the
 * bd_episode_stats accumulators), then SoA planes, each starting on a 256-byte boundary, in this order:
 *   kinematics      4 x Real4[n_total]   (pos, quat, vel, body rates, TARGET_POS)       always
 *   world ang. vel. Real4[n_total]                                                       BD_SNAP_ANGV (keep_ang_vel)
 *   controller      13 x Real[n_total]   (9 DSL PID memory + 4 commanded-rpm planes)    BD_SNAP_CTRL (PID / VEL / ONE_D_PID)
 *   action ring     B x float[n_total][A], by AGE: plane a = the action of a steps ago   always
 *   step counters   int32[N]                                                             always
 *   episode returns float[N]                                                             BD_SNAP_EPISODES (track_episodes)
 * Because the ring is stored by age, a snapshot does not depend on the saving handle's step count.
 * Restoring needs a handle with the same N, M, task, act_type, drone model, precision, aero flags, integrator,
 * pyb_freq, ctrl_freq, airframe / controller / spiral constants and episode length (checked against the fingerprint).
 * Device, seed, auto_reset, reset_mode, action_is_f32, ctrl_reset_on_reset, the L2 plan and BD_PIPELINE may differ, and
 * so may keep_ang_vel and track_episodes as long as the snapshot carries every plane the target needs (planes the
 * target has no use for are ignored).  Initial poses and the jitter buffer are configuration, not state: set them with
 * bd_set_init_poses / bd_set_jitter.  Observations are not part of the snapshot either: the observation of a saved
 * state is the one the step returned then, and the caller keeps it.
 * Neither call is capturable (BD_EINVAL while `stream` is capturing); both BD_EINVAL on a poisoned handle. */
enum { BD_SNAP_ANGV = 1, BD_SNAP_CTRL = 2, BD_SNAP_EPISODES = 4 };
/* Size in bytes of a snapshot of this shape (host computation only); BD_EINVAL for a malformed shape or flag. */
int bd_snapshot_layout(int n_envs, int n_drones, int act_dim, int buf_slots, int precision, int flags, int64_t* bytes);
/* Size of this handle's snapshots (BD_EINVAL for a NULL handle). */
int64_t bd_snapshot_bytes(const bd_handle* h);
/* Write the handle's state into snap_dev (bd_snapshot_bytes bytes).  Stream ordered, does not synchronise; a plain
 * launch, so it runs after the previous step has completed. */
int bd_save_snapshot(bd_handle* h, void* snap_dev, void* stream);
/* Restore a snapshot.  Copies the header back, synchronises `stream`, validates it (BD_EINVAL with a message for a bad
 * magic, version or size, a configuration mismatch or a missing plane), then launches the unpack kernel.
 *   env_mask_dev == NULL: full restore — every per-env plane, the episode accumulators, and the Philox counter and
 *     explicit-reset epoch exactly as bd_set_rng_state sets them.  BD_EINVAL once a step was captured into a CUDA graph.
 *   env_mask_dev (N) uint8: masked restore — only the envs with a non-zero entry; the handle's step count, episode
 *     accumulators and RNG state are left alone, and the ring is rewritten by age relative to this handle's head.
 * The next step launch of the handle reads nothing before its dependency wait (DESIGN.md section 4). */
int bd_load_snapshot(bd_handle* h, const void* snap_dev, const uint8_t* env_mask_dev, void* stream);

int bd_obs_dim(const bd_handle* h);              /* D                                 */
int bd_act_dim(const bd_handle* h);              /* A                                 */
int bd_action_buffer_size(const bd_handle* h);   /* B                                 */
int bd_substeps(const bd_handle* h);             /* PYB_STEPS_PER_CTRL                */
int64_t bd_launch_count(const bd_handle* h);     /* kernels launched by this handle   */
const char* bd_last_error(void);
int bd_version(void);

/* ------------------------------------------------------------------------------------------
 * Fused actor forward on the tensor cores (SURVEY.md 8f-1, the caller of the step).
 * Replaces the batched branch of MAPPOActorCritic.step (mappo/agent.py:389-415): shared actor
 * MLP obs_dim -> hidden -> hidden -> act_dim with tanh (safe_control_gym/math_and_models/
 * neural_networks.py:18-53), Gaussian sample with state-independent logstd and its summed
 * log-probability (distributions.py:9-21), in one tcgen05/TMEM kernel (bf16 operands, fp32
 * accumulation).  hidden in {64,128,256}, act_dim <= 4.
 * ------------------------------------------------------------------------------------------ */
typedef struct bd_actor bd_actor;
int bd_actor_create(int obs_dim, int hidden, int act_dim, int device, bd_actor** out);
void bd_actor_destroy(bd_actor* a);
/* fp32 device pointers in torch.nn.Linear layout: w1 (hidden,obs_dim), w2 (hidden,hidden),
 * w3 (act_dim,hidden), biases, logstd (act_dim).  Repacked (stream ordered) to bf16 UMMA tiles. */
int bd_actor_set_weights(bd_actor* a, const float* w1, const float* b1, const float* w2, const float* b2,
                         const float* w3, const float* b3, const float* logstd, void* stream);
/* obs_dev (rows,obs_dim) float -> act_dev (rows,act_dim), logp_dev (rows), optional mean_dev.
 * noise_dev (rows,act_dim) standard normals, or NULL: Philox4x32-10(seed; row, offset). */
int bd_actor_forward(bd_actor* a, const float* obs_dev, int64_t rows, const float* noise_dev, uint64_t seed,
                     uint64_t offset, float* act_dev, float* logp_dev, float* mean_dev, void* stream);
/* Diagnostics: when trace_dev != NULL, CTA 0 of the next forward launches writes 16 SM-clock stamps
 * per tile it processes ([tiles_of_cta0][16] int64) marking the pipeline phases (see bd_actor.cu);
 * NULL switches tracing off. */
int bd_actor_set_trace(bd_actor* a, long long* trace_dev);
/* Normalise the input rows on load: x <- clip((x - mean[(row % period) * obs_dim + k]) * rstd[...], +-clip)
 * with float vectors of period*obs_dim entries (bd_rms_get's mean_f / rstd_f); mean_dev == NULL
 * switches it off.  `period` = agents per env (the reference's normaliser has the observation
 * space's shape (M, D), mappo/mappo.py:132). */
int bd_actor_set_input_norm(bd_actor* a, const float* mean_dev, const float* rstd_dev, int period, float clip);
int64_t bd_actor_launch_count(const bd_actor* a);
const char* bd_actor_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Running observation statistics on the device: RunningMeanStd / MeanStdNormalizer of
 * safe_control_gym/math_and_models/normalization.py:13-96 as MAPPO uses them on every
 * observation batch (mappo/mappo.py:132,165,804).  cols = prod(observation_space.shape).
 * ------------------------------------------------------------------------------------------ */
typedef struct bd_rms bd_rms;
/* mean = 0, var = 1, count = count0 (the reference's epsilon = 1e-4, :24-32); eps = the normaliser's
 * divide-by-zero offset (1e-8, :71). */
int bd_rms_create(int cols, int device, double count0, double eps, bd_rms** out);
void bd_rms_destroy(bd_rms* r);
/* RunningMeanStd.update (:34-58): batch mean / population variance over the `rows` axis of
 * x_dev (rows, cols) float, merged into the running statistics.  One launch, stream ordered. */
int bd_rms_update(bd_rms* r, const float* x_dev, int64_t rows, void* stream);
/* The two halves of bd_rms_update, for envs sharded over ranks: batch moments of the local rows into
 * moments_dev = [mean(cols) | var(cols) | count] doubles (:37-39), then — after the caller has
 * all-gathered every rank's moments into (parts, 2*cols+1) — update_from_moments (:44-58) with the
 * moments of the union of the parts (combined in order, so every rank gets identical statistics). */
int bd_rms_batch_moments(bd_rms* r, const float* x_dev, int64_t rows, double* moments_dev, void* stream);
int bd_rms_merge_moments(bd_rms* r, const double* moments_dev, int parts, void* stream);
/* y = clip((x - mean) / sqrt(var + eps), -clip, clip) (:84-88), y_dev may equal x_dev. */
int bd_rms_normalize(bd_rms* r, const float* x_dev, float* y_dev, int64_t rows, float clip, void* stream);
/* state_dict / load_state_dict (:90-96): any pointer may be NULL.  mean_f / rstd_f are the float
 * vectors (mean, 1/sqrt(var+eps)) fused consumers read (bd_actor_set_input_norm). */
int bd_rms_get(bd_rms* r, double* mean_dev, double* var_dev, double* count_dev, float* mean_f_dev, float* rstd_f_dev,
               void* stream);
int bd_rms_set(bd_rms* r, const double* mean_dev, const double* var_dev, const double* count_dev, void* stream);
int64_t bd_rms_launch_count(const bd_rms* r);
const char* bd_rms_last_error(void);

/* ------------------------------------------------------------------------------------------
 * PPO update of the MAPPO trainer as hand-written tensor-core kernels (csrc/bd_ppo.cu).
 * Replaces MAPPOAgent.update / compute_policy_loss / compute_value_loss (mappo/agent.py:602-772)
 * and _compute_single_agent_returns + normalize_advantages (mappo/buffer.py:561-614, 666-695).
 * A bd_ppo_net is one MLP in -> 256 -> 256 -> out with tanh (neural_networks.py:18-53):
 *   actor : in_dim = obs_dim, chunks = 1, out_dim = act_dim, has_logstd = 1; row = (sample, agent)
 *   critic: in_dim = obs_dim, chunks = M, out_dim = 1 (centralised: the M agents' observations of an
 *           env-step, agent.py:164-223); row = sample
 * Master parameters are fp32 in ONE flat caller-owned buffer in torch's parameter order
 * ([logstd] W1 b1 W2 b2 W3 b3, nn.Linear layout); the library keeps bf16 copies for the tensor cores.
 * "sample" = env-step index t * n_envs + n into the rollout arrays; obs_dev is (slots, N, M, D).
 * ------------------------------------------------------------------------------------------ */
typedef struct bd_ppo_net bd_ppo_net;
int bd_ppo_net_create(int in_dim, int chunks, int out_dim, int has_logstd, int64_t max_rows, int device,
                      bd_ppo_net** out);
void bd_ppo_net_destroy(bd_ppo_net* n);
int64_t bd_ppo_net_param_count(const bd_ppo_net* n);
/* device doubles [16] of the last bd_ppo_grad: [0] sum of per-row losses, [1] sum of (logp_old - logp), [2] rows,
 * [3..6] d loss / d logstd sums, [7..10] output-bias gradient sums */
double* bd_ppo_net_stats(bd_ppo_net* n);
/* flat fp32 parameters -> bf16 K-step slabs (stream ordered; bd_ppo_adam_step does it itself) */
int bd_ppo_net_pack(bd_ppo_net* n, const float* flat_params_dev, void* stream);
/* out (rows, out_dim) = MLP(rows); idx_dev (samples) int64 or NULL = identity; nmean / nrstd: optional
 * per-slot observation statistics ((slots, M*D) floats, MeanStdNormalizer on load) */
int bd_ppo_forward(bd_ppo_net* n, const float* obs_dev, int n_envs, int n_agents, const int64_t* idx_dev,
                   int64_t rows, const float* nmean_dev, const float* nrstd_dev, float nclip, float* out_dev,
                   void* stream);
/* rollout-time policy step of an actor net (MAPPOActorCritic.step, mappo/agent.py:389-415) in ONE launch:
 * obs_dev (n_envs, n_agents, D) = one slot -> act_dev (rows, out_dim) = mean + exp(logstd) eps, logp_dev (rows) = summed
 * Gaussian log-density, optional mean_dev; rows = n_envs * n_agents.  eps = noise_dev (rows, out_dim) standard normals, or
 * NULL: Philox4x32-10(seed; row, offset).  nmean / nrstd: that slot's (n_agents * D) statistics or NULL. */
int bd_ppo_sample(bd_ppo_net* n, const float* obs_dev, int n_envs, int n_agents, const float* nmean_dev,
                  const float* nrstd_dev, float nclip, const float* noise_dev, uint64_t seed, uint64_t offset,
                  float* act_dev, float* logp_dev, float* mean_dev, void* stream);
/* one minibatch: forward, PPO clipped-ratio loss (actor: act, logp_old (slots,N,M[,A]), adv (slots,N) with
 * adv_stats = (mean, scale)) or value loss (critic: ret, optional v_old (slots,N)), backward, weight
 * gradients -> grad_dev (flat, parameter order) = mean over rows_global rows (0 = this call's rows);
 * run_acc_dev (optional, 4 doubles) += per-minibatch (mean loss, approx_kl, 1, entropy loss) */
int bd_ppo_grad(bd_ppo_net* n, int critic, const float* obs_dev, int n_envs, int n_agents, const int64_t* idx_dev,
                int64_t samples, const float* act_dev, const float* logp_old_dev, const float* adv_dev,
                const float* adv_stats_dev, const float* ret_dev, const float* v_old_dev, float clip,
                int use_clipped_value, float entropy_coef, const float* nmean_dev, const float* nrstd_dev,
                float nclip, int64_t rows_global, float* grad_dev, double* run_acc_dev, void* stream);
/* torch.optim.Adam step on flat buffers, skipped entirely (moments and step count too) when
 * kl_sum / kl_rows > 1.5 target_kl (agent.py:731; NULL or target_kl <= 0: unconditional); then repack */
int bd_ppo_adam_step(bd_ppo_net* n, float* param_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                     const float* grad_dev, double* step_dev, float lr, float beta1, float beta2, float eps,
                     const double* kl_sum_dev, const double* kl_rows_dev, float target_kl, double* gate_count_dev,
                     void* stream);
/* returns / advantages of a rollout in one launch: rew (T,N), term / trunc (T,N) uint8, vals (T+1,N) with the
 * bootstrap value in row T; acc3_dev += (sum adv, sum adv^2, count) */
int bd_ppo_gae(const float* rew_dev, const uint8_t* term_dev, const uint8_t* trunc_dev, const float* vals_dev, int T,
               int N, float gamma, float lam, int use_gae, float* ret_dev, float* adv_dev, double* acc3_dev,
               void* stream);
int bd_ppo_adv_stats(const double* acc3_dev, float* stats2_dev, void* stream);
/* diagnostics: CTA 0 of the following forward / sample launches writes SM-clock stamps of its pipeline phases
 * ([tile pair][64] int64, see csrc/bd_ppo.cu); NULL switches tracing off */
int bd_ppo_set_trace(bd_ppo_net* n, long long* trace_dev);
/* which forward / loss / backward kernel bd_ppo_grad launches: 0 (default) one 128-row tile in flight per CTA, 1 two tiles in
 * flight (one in-place activation buffer per tile, every weight slab serving both tiles); same results */
int bd_ppo_set_train_mode(bd_ppo_net* n, int mode);
/* which kernel bd_ppo_forward / bd_ppo_sample launch for an actor net: 0 (default) two tiles in flight per CTA, weights
 * streamed from L2; 1 the CTA-pair kernel (cta_group::2: M = 256 MMAs, half of every weight matrix resident per CTA) */
int bd_ppo_set_forward_mode(bd_ppo_net* n, int mode);
int64_t bd_ppo_launch_count(const bd_ppo_net* n);
const char* bd_ppo_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Gradient all-reduce of the data-parallel trainer over NVLink peer memory (csrc/bd_peer.cu).
 * The reference's MAPPOAgent.update (mappo/agent.py:702-772) runs in one process; with the envs sharded
 * over one process per GPU every minibatch needs the sum of the ranks' flat gradients and of the KL pair
 * of the gate (agent.py:731) before the optimiser step.  A bd_peer is one rank's block of device memory,
 * mapped by all ranks of the node through CUDA IPC; bd_peer_allreduce is ONE kernel launch per rank that
 * sums the first `floats` floats of every rank's data region IN PLACE (rank r reduces slice r from all
 * peers and writes it back to all of them: identical bits on every rank) and `n_extra` doubles that live
 * outside the block.  Stream ordered, no host synchronisation, capturable in a CUDA graph; all ranks
 * must make the same sequence of calls.
 * ------------------------------------------------------------------------------------------ */
typedef struct bd_peer bd_peer;
int bd_peer_create(int device, int rank, int world, int64_t floats, bd_peer** out);   /* 2 <= world <= 16, one node */
void bd_peer_destroy(bd_peer* p);
int bd_peer_handle_size(void);                           /* bytes of an exported handle (cudaIpcMemHandle_t) */
int bd_peer_get_handle(bd_peer* p, void* handle_out);    /* to be all-gathered by the caller (any transport) */
int bd_peer_open(bd_peer* p, const void* handles, int count);   /* count = world handles in rank order */
float* bd_peer_data(bd_peer* p);                         /* the rank's data region: gradient kernels write here */
int bd_peer_allreduce(bd_peer* p, int64_t floats, double* extra_dev, int n_extra, void* stream);
/* shutdown: every rank bd_peer_unmap, barrier (caller's transport), every rank bd_peer_destroy */
int bd_peer_unmap(bd_peer* p);
int64_t bd_peer_launch_count(const bd_peer* p);
const char* bd_peer_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* BATCH_DRONES_H_ */
