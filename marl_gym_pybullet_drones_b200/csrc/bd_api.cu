// C-ABI of the batched drone-step library (include/batch_drones.h).
// Host-side only: argument checking, device allocations, kernel-parameter
// blocks and stream-ordered launches.  No CPU compute path exists here; if CUDA
// is unavailable every call fails with BD_ECUDA.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "../../include/batch_drones.h"
#include "bd_params.h"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define BD_CUDA(expr)                                                                 \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess)                                                            \
      return fail(BD_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),   \
                  __FILE__, __LINE__);                                                \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    target = dev;
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != target) cudaSetDevice(prev);
  }
  int target = -1;
};

}  // namespace

struct bd_handle {
  bd_config cfg;
  int S = 0, A = 0, B = 0, D = 0, E = 0;
  int EW = 1;                  // fast tile kernel: whole envs per warp (32 / M); a tile = 4 EW envs
  long long n_total = 0;
  size_t real = 4;
  bd::LaunchSpec spec{};
  // device allocations
  void *s0 = nullptr, *s1 = nullptr, *s2 = nullptr, *s3 = nullptr, *s4 = nullptr;
  float* hist = nullptr;
  int* stepc = nullptr;
  int* gsteps = nullptr;
  int* tile_epoch = nullptr;
  unsigned long long* finished = nullptr;
  int pipeline = 0;
  int l2_keep_state = 0, l2_keep_slots = 0;   // fast tile kernel's L2 residency plan (bd_l2_plan)
  float* ep_ret = nullptr;
  double* ep_acc = nullptr;
  void* ctrl = nullptr;        // DSL PID memory + commanded rpm, PID action types only
  void* init_xyz = nullptr;
  void* init_rpy = nullptr;
  int init_env_stride = 0;
  void* jitter = nullptr;
  // staging for bd_step_host
  void* h_actions = nullptr;
  float* h_obs = nullptr;
  void* h_reward = nullptr;
  uint8_t *h_term = nullptr, *h_trunc = nullptr;
  float* h_tobs = nullptr;
  cudaStream_t hs_a = nullptr, hs_b = nullptr;   // bd_step_host pipeline: (H2D, kernel) chunks / D2H chunks
  cudaEvent_t hs_start = nullptr, hs_done = nullptr, hs_chunk[8] = {};
  int64_t launches = 0;
  long long total_steps = 0;   // host mirror of gsteps[0]
  bool graph_mode = false;     // a step was captured into a CUDA graph: the device counter is authoritative
  int reset_epoch = 0;
  uint32_t philox_base = 0;    // bd_set_rng_state: offset of the Philox step counter
  int many_mode = 0;           // bd_step_many: 0 = one launch when possible, 1 = always k launches (bd_set_step_many_mode)
  bool poisoned = false;       // a launch failed half-way through a chunked host step: the tile epochs are inconsistent
  bool restored = false;       // bd_load_snapshot ran since the last step launch: that launch must not prefetch early
  // compact terminal observations (bd_step_host_compact): pinned, device-mapped staging owned by the handle
  int* c_blockcnt = nullptr;   // [blocks of 1024 envs] done envs per block
  int* c_total = nullptr;      // running count of finished envs over the chunks of one step
  int* c_idx_dev = nullptr;    // device: [0] = count, [1..N] = done env indices (ascending)
  float* c_rows_dev = nullptr; // device: [cap][M][D] terminal observation rows, same order
  int c_cap_dev = 0;
  cudaEvent_t hs_compact = nullptr;
  // host side: two page-locked sets, used alternately: what a call returns stays valid until the next-but-one step
  int* c_host[2] = {nullptr, nullptr};
  float* c_rows_host[2] = {nullptr, nullptr};
  int c_cap[2] = {0, 0};
  int c_flip = 0;
  bd::Params<float> pf{};
  bd::Params<double> pd{};
};

namespace {

template <typename R>
void fill_params(const bd_handle* h, bd::Params<R>& P) {
  const bd_config& c = h->cfg;
  using R4 = typename bd::V4<R>::type;
  P.N = c.n_envs; P.M = c.n_drones; P.S = h->S; P.A = h->A; P.B = h->B; P.D = h->D;
  P.E = h->E; P.EW = h->EW; P.n_total = h->n_total;
  P.s0 = (R4*)h->s0; P.s1 = (R4*)h->s1; P.s2 = (R4*)h->s2; P.s3 = (R4*)h->s3; P.s4 = (R4*)h->s4;
  P.hist = h->hist; P.stepc = h->stepc; P.gsteps = h->gsteps; P.tile_epoch = h->tile_epoch; P.finished = h->finished;
  P.step_tiles = h->spec.impl == 1 ? (h->cfg.n_envs + 4 * h->EW - 1) / (4 * h->EW) : (h->cfg.n_envs + h->E - 1) / h->E;
  P.pipeline = h->pipeline; P.pipe_wait = 0; P.early_prefetch = 1; P.ep_ret = h->ep_ret; P.ep_acc = h->ep_acc;
  P.l2_keep_state = h->l2_keep_state; P.l2_keep_slots = h->l2_keep_slots;
  P.ctrl = (R*)h->ctrl;
  P.act_type = c.act_type; P.ctrl_reset = c.ctrl_reset_on_reset;
  P.ctrl_dt = (R)(1.0 / c.ctrl_freq);                      // CTRL_TIMESTEP (BaseAviary.py:83)
  P.ctrl_gravity = (R)(c.g * c.ctrl_mass);                 // BaseControl.py:35
  P.ctrl_4kf = (R)(4 * c.ctrl_kf);                         // DSLPIDControl.py:187
  P.speed_limit = (R)c.speed_limit; P.speed_limit_f = (float)c.speed_limit;
  P.init_xyz = (const R*)h->init_xyz; P.init_rpy = (const R*)h->init_rpy;
  P.init_env_stride = h->init_env_stride;
  P.jitter = (const R*)h->jitter;
  P.actions = nullptr; P.obs = nullptr; P.reward = nullptr; P.terminated = nullptr;
  P.truncated = nullptr; P.terminal_obs = nullptr; P.reset_mask = nullptr;
  // derived constants exactly as BaseAviary.py:117-118 computes them, in double,
  // then narrowed once to the kernel's precision
  const double gravity = c.g * c.mass;
  const double hover_rpm = sqrt(gravity / (4 * c.kf));
  const double max_rpm = sqrt((c.thrust2weight * gravity) / (4 * c.kf));
  const double max_thrust = 4 * c.kf * max_rpm * max_rpm;
  const double gnd_h_clip =
      0.25 * c.prop_radius * sqrt((15 * max_rpm * max_rpm * c.kf * c.gnd_eff_coeff) / max_thrust);
  P.dt = (R)(1.0 / c.pyb_freq);
  P.hover_rpm = (R)hover_rpm;
  P.kf = (R)c.kf; P.km = (R)c.km;
  P.arm = (R)(c.drone_model == BD_MODEL_CF2P ? c.arm : c.arm / sqrt(2.0));
  P.inv_m = (R)(1.0 / c.mass);
  P.gravity = (R)gravity;
  P.jx = (R)c.ixx; P.jy = (R)c.iyy; P.jz = (R)c.izz;
  P.ijx = (R)(1.0 / c.ixx); P.ijy = (R)(1.0 / c.iyy); P.ijz = (R)(1.0 / c.izz);
  P.gnd_coeff = (R)c.gnd_eff_coeff; P.prop_radius = (R)c.prop_radius; P.gnd_h_clip = (R)gnd_h_clip;
  P.drag_xy = (R)c.drag_coeff_xy; P.drag_z = (R)c.drag_coeff_z;
  P.dw1 = (R)c.dw_coeff_1; P.dw2 = (R)c.dw_coeff_2; P.dw3 = (R)c.dw_coeff_3;
  for (int k = 0; k < 4; ++k) { P.prop_x[k] = (R)c.prop_xy[2 * k]; P.prop_y[k] = (R)c.prop_xy[2 * k + 1]; }
  P.sp_R = (R)c.spiral_radius;
  P.sp_omega = (R)(c.spiral_period != 0.0 ? 2 * 3.14159265358979323846 / c.spiral_period : 0.0);
  P.sp_vz = (R)c.height_rate; P.sp_cx = (R)c.target_center[0]; P.sp_cy = (R)c.target_center[1];
  P.pyb_freq = (double)c.pyb_freq; P.episode_len = c.episode_len_sec;
  P.task = c.task;
  {  // integer form of `step_counter / PYB_FREQ > EPISODE_LEN_SEC` (MultiHoverAviary.py:268), same fp64 division
    long long k = (long long)(c.episode_len_sec * c.pyb_freq) - 2;
    if (k < 0) k = 0;
    while (!((double)k / (double)c.pyb_freq > c.episode_len_sec)) ++k;
    P.trunc_counter = (int)k;
  }
  P.model = c.drone_model; P.aero = c.aero_flags; P.integrator = c.integrator;
  P.auto_reset = c.auto_reset; P.reset_mode = c.reset_mode; P.action_is_f32 = c.action_is_f32;
  P.keep_angv = c.keep_ang_vel;
  P.seed = c.seed;
  P.philox_base = h->philox_base;
  P.obs_aligned = 1;
  P.reset_epoch = 0;
  P.block0 = 0; P.grid_blocks = 0; P.advance = 1;
  P.total_wrap = h->B * ((1 << 30) / h->B);
  P.host_total = h->graph_mode ? -1 : (int)h->total_steps;
  P.host_head = (int)(h->total_steps % h->B);
}

// tiles of either step kernel (128 drones for the fast kernel, E whole envs for the generic one)
long long epoch_tiles(const bd_handle* h) {
  const long long ept = 4 * h->EW;
  const long long a = (h->cfg.n_envs + ept - 1) / ept, b = (h->cfg.n_envs + h->E - 1) / h->E;
  return a > b ? a : b;
}

void refresh_params(bd_handle* h) {
  if (h->cfg.precision == BD_F64) fill_params<double>(h, h->pd);
  else fill_params<float>(h, h->pf);
}

void* params_ptr(bd_handle* h) {
  const int ht = h->graph_mode ? -1 : (int)h->total_steps;
  h->pd.host_total = ht;
  h->pf.host_total = ht;
  h->pd.host_head = h->pf.host_head = (int)(h->total_steps % h->B);
  return h->cfg.precision == BD_F64 ? (void*)&h->pd : (void*)&h->pf;
}

template <typename F>
void with_params(bd_handle* h, F&& f) {
  if (h->cfg.precision == BD_F64) f(h->pd); else f(h->pf);
}

int upload_table(bd_handle* h, const double* src, size_t count, void** dst) {
  std::vector<unsigned char> tmp(count * h->real);
  if (h->real == 8) {
    memcpy(tmp.data(), src, count * 8);
  } else {
    float* f = reinterpret_cast<float*>(tmp.data());
    for (size_t i = 0; i < count; ++i) f[i] = (float)src[i];
  }
  if (*dst) { cudaFree(*dst); *dst = nullptr; }
  BD_CUDA(cudaMalloc(dst, count * h->real));
  BD_CUDA(cudaMemcpy(*dst, tmp.data(), count * h->real, cudaMemcpyHostToDevice));
  return BD_OK;
}

int default_init_tables(bd_handle* h) {
  const bd_config& c = h->cfg;
  const int M = c.n_drones;
  std::vector<double> xyz(M * 3), rpy(M * 3, 0.0);
  for (int i = 0; i < M; ++i) {
    if (c.task == BD_TASK_SPIRAL) {            // SpiralAviary.py:47-53
      const double ang = 2 * 3.14159265358979323846 * i / M;
      xyz[i * 3 + 0] = c.spiral_radius * cos(ang);
      xyz[i * 3 + 1] = c.spiral_radius * sin(ang);
      xyz[i * 3 + 2] = 0.3;
    } else {                                   // BaseAviary.py:194-197 (collision cyl h=.025, offset 0)
      xyz[i * 3 + 0] = i * 4 * c.arm;
      xyz[i * 3 + 1] = i * 4 * c.arm;
      xyz[i * 3 + 2] = 0.025 / 2 - 0.0 + .1;
    }
  }
  h->init_env_stride = 0;
  int rc = upload_table(h, xyz.data(), xyz.size(), &h->init_xyz);
  if (rc) return rc;
  return upload_table(h, rpy.data(), rpy.size(), &h->init_rpy);
}

int do_reset(bd_handle* h, const uint8_t* mask, float* obs, int force_fixed, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  with_params(h, [&](auto& P) {
    auto Q = P;
    Q.host_total = h->graph_mode ? -1 : (int)h->total_steps;
    Q.reset_mask = mask;
    Q.obs = obs;
    if (force_fixed) Q.reset_mode = BD_RESET_FIXED;
    Q.reset_epoch = ++h->reset_epoch;
    e = bd::launch_reset(h->spec, &Q, st);
  });
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "reset kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

void free_all(bd_handle* h) {
  cudaFree(h->s0); cudaFree(h->s1); cudaFree(h->s2); cudaFree(h->s3); cudaFree(h->s4);
  cudaFree(h->hist); cudaFree(h->stepc); cudaFree(h->gsteps); cudaFree(h->tile_epoch); cudaFree(h->finished); cudaFree(h->ep_ret); cudaFree(h->ep_acc); cudaFree(h->ctrl);
  cudaFree(h->init_xyz); cudaFree(h->init_rpy);
  cudaFree(h->jitter);
  cudaFree(h->c_blockcnt);
  cudaFree(h->c_total);
  cudaFree(h->c_idx_dev);
  cudaFree(h->c_rows_dev);
  if (h->hs_compact) cudaEventDestroy(h->hs_compact);
  for (int i = 0; i < 2; ++i) { if (h->c_host[i]) cudaFreeHost(h->c_host[i]); if (h->c_rows_host[i]) cudaFreeHost(h->c_rows_host[i]); }
  cudaFree(h->h_actions); cudaFree(h->h_obs); cudaFree(h->h_reward); cudaFree(h->h_term);
  cudaFree(h->h_trunc); cudaFree(h->h_tobs);
  if (h->hs_a) {
    cudaStreamDestroy(h->hs_a); cudaStreamDestroy(h->hs_b);
    cudaEventDestroy(h->hs_start); cudaEventDestroy(h->hs_done);
    for (auto ev : h->hs_chunk) cudaEventDestroy(ev);
  }
}

}  // namespace

extern "C" {

int bd_version(void) { return BD_VERSION; }
const char* bd_last_error(void) { return g_err; }

int bd_create(const bd_config* cfg, bd_handle** out) {
  if (!cfg || !out) return fail(BD_EINVAL, "bd_create: null argument");
  *out = nullptr;
  if (cfg->struct_size != (int32_t)sizeof(bd_config))
    return fail(BD_EINVAL, "bd_create: struct_size %d != %zu (ABI mismatch)", cfg->struct_size, sizeof(bd_config));
  if (cfg->n_envs < 1) return fail(BD_EINVAL, "bd_create: n_envs must be >= 1");
  if (cfg->n_drones < 1 || cfg->n_drones > bd::kMaxDrones)
    return fail(BD_EINVAL, "bd_create: n_drones must be in [1,%d]", bd::kMaxDrones);
  if (cfg->task < 0 || cfg->task > BD_TASK_LEADERFOLLOWER) return fail(BD_EINVAL, "bd_create: unknown task %d", cfg->task);
  if (cfg->task == BD_TASK_HOVER && cfg->n_drones != 1)
    return fail(BD_EINVAL, "bd_create: the hover task is single-drone (HoverAviary.py:54)");
  if (cfg->act_type < BD_ACT_RPM || cfg->act_type > BD_ACT_ONE_D_PID)
    return fail(BD_EINVAL, "bd_create: unknown act_type %d", cfg->act_type);
  const bool pid_act = cfg->act_type >= BD_ACT_PID;
  if (pid_act && cfg->drone_model == BD_MODEL_RACE)
    return fail(BD_EINVAL, "[ERROR] in BaseRLAviary.__init()__, no controller is available for the specified drone_model");
  if (pid_act && (!(cfg->ctrl_mass > 0) || !(cfg->ctrl_kf > 0) || cfg->speed_limit < 0))
    return fail(BD_EINVAL, "bd_create: PID action types need ctrl_mass > 0, ctrl_kf > 0, speed_limit >= 0");
  if (cfg->drone_model < 0 || cfg->drone_model > 2) return fail(BD_EINVAL, "bd_create: unknown drone_model");
  if (cfg->precision != BD_F32 && cfg->precision != BD_F64) return fail(BD_EINVAL, "bd_create: unknown precision");
  if (cfg->pyb_freq <= 0 || cfg->ctrl_freq <= 0 || cfg->pyb_freq % cfg->ctrl_freq != 0)
    return fail(BD_EINVAL, "[ERROR] in BaseAviary.__init__(), pyb_freq is not divisible by env_freq.");
  if (cfg->ctrl_freq / 2 < 1) return fail(BD_EINVAL, "bd_create: ctrl_freq must be >= 2 (action buffer)");
  if (cfg->aero_flags & ~7) return fail(BD_EINVAL, "bd_create: unknown aero flag");
  if (cfg->integrator != BD_INTEGRATOR_QUAT && cfg->integrator != BD_INTEGRATOR_EULER)
    return fail(BD_EINVAL, "bd_create: unknown integrator");
  if (cfg->reset_mode < 0 || cfg->reset_mode > 2) return fail(BD_EINVAL, "bd_create: unknown reset_mode");
  if (!(cfg->mass > 0) || !(cfg->kf > 0) || !(cfg->ixx > 0) || !(cfg->iyy > 0) || !(cfg->izz > 0))
    return fail(BD_EINVAL, "bd_create: airframe constants must be positive");

  int ndev = 0;
  BD_CUDA(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev)
    return fail(BD_EINVAL, "bd_create: device %d out of range (%d visible)", cfg->device, ndev);
  DeviceGuard guard(cfg->device);
  if (!guard.ok) return fail(BD_ECUDA, "bd_create: cannot select device %d", cfg->device);

  bd_handle* h = new (std::nothrow) bd_handle();
  if (!h) return fail(BD_ENOMEM, "bd_create: out of host memory");
  h->cfg = *cfg;
  h->S = cfg->pyb_freq / cfg->ctrl_freq;
  h->A = (cfg->act_type == BD_ACT_RPM || cfg->act_type == BD_ACT_VEL) ? 4 : (cfg->act_type == BD_ACT_PID ? 3 : 1);
  h->B = cfg->ctrl_freq / 2;
  h->D = 12 + h->B * h->A + (cfg->task == BD_TASK_SPIRAL ? 11 : 0);
  h->E = bd::kBlock / cfg->n_drones;
  h->n_total = (long long)cfg->n_envs * cfg->n_drones;
  h->real = cfg->precision == BD_F64 ? 8 : 4;
  h->spec.task = cfg->task;
  h->spec.act_a = h->A;
  h->spec.precision = cfg->precision;
  h->spec.device = cfg->device;
  const bool swarm = cfg->task >= BD_TASK_MEETUP;   // coupled rewards: fast tile kernel or generic kernel, never the non-generic CTA kernel
  h->spec.generic = (cfg->aero_flags != 0 || cfg->integrator != BD_INTEGRATOR_QUAT || cfg->keep_ang_vel || pid_act || swarm) ? 1 : 0;
  {
    // kernel selection: the fast tile kernel covers the throughput configurations
    // (float, plain DYN, M a power of two <= 32); everything else runs the two-role CTA
    // kernel.  BD_STEP_IMPL=cta forces the latter (A/B measurements, tests).
    const int m = cfg->n_drones;
    const bool pow2 = (m & (m - 1)) == 0 && m <= 32;
    h->EW = m <= 32 ? 32 / m : 1;   // whole envs per warp on the fast kernel
    const char* force = getenv("BD_STEP_IMPL");
    // the fast kernel carries ground effect, drag and downwash (shuffle exchange inside the env's lane group); the
    // swarm tasks' shuffle rewards need M == G
    const bool plain = cfg->integrator == BD_INTEGRATOR_QUAT && !cfg->keep_ang_vel;
    h->spec.impl = (cfg->precision == BD_F32 && plain && m <= 32 && (pow2 || !swarm) && !pid_act) ? 1 : 0;
    if (force && strcmp(force, "cta") == 0) h->spec.impl = 0;
    const char* pdl = getenv("BD_PDL");
    h->spec.pdl = (pdl && strcmp(pdl, "0") == 0) ? 0 : 1;
    const char* pl = getenv("BD_PIPELINE");
    h->pipeline = (h->spec.pdl && !(pl && strcmp(pl, "0") == 0)) ? 1 : 0;   // BD_PIPELINE=0 switches it off
  }

  const size_t smem = bd::step_smem_bytes(cfg->precision, h->A, h->B, h->D, cfg->task);
  cudaDeviceProp prop;
  cudaError_t pe = cudaGetDeviceProperties(&prop, cfg->device);
  if (pe != cudaSuccess) { delete h; return fail(BD_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(pe)); }
  if (h->spec.impl == 1 && (size_t)(4 * h->EW) * cfg->n_drones * h->D * 4 > prop.sharedMemPerBlockOptin) h->spec.impl = 0;
  h->spec.sm_count = prop.multiProcessorCount;
  if (h->spec.impl == 1) {
    const int rc = bd_l2_plan(cfg->n_envs, cfg->n_drones, h->A, h->B, cfg->track_episodes, prop.l2CacheSize,
                              getenv("BD_L2_KEEP"), &h->l2_keep_state, &h->l2_keep_slots);
    if (rc) { delete h; return rc; }
  }
  if (smem > prop.sharedMemPerBlockOptin) {
    delete h;
    return fail(BD_EINVAL, "bd_create: the history staging tile needs %zu B of shared memory (> %zu)", smem,
                (size_t)prop.sharedMemPerBlockOptin);
  }

  const size_t plane = (size_t)h->n_total * 4 * h->real;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(p, bytes);
    if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes);
  };
  alloc(&h->s0, plane); alloc(&h->s1, plane); alloc(&h->s2, plane); alloc(&h->s3, plane);
  if (cfg->keep_ang_vel) alloc(&h->s4, plane);
  alloc((void**)&h->hist, (size_t)h->B * h->n_total * h->A * sizeof(float));   // zeros: BaseRLAviary.py:153-154
  alloc((void**)&h->stepc, (size_t)cfg->n_envs * sizeof(int));
  alloc((void**)&h->gsteps, 16 * sizeof(int));   // [0] total steps, [1] CTA ticket, [8..15] per-launch wait decisions
  alloc((void**)&h->tile_epoch, (size_t)epoch_tiles(h) * sizeof(int));
  alloc((void**)&h->finished, sizeof(unsigned long long));
  if (cfg->track_episodes) alloc((void**)&h->ep_ret, (size_t)cfg->n_envs * sizeof(float));
  alloc((void**)&h->ep_acc, 3 * sizeof(double));
  if (pid_act) alloc(&h->ctrl, (size_t)bd::kCtrlPlanesHost * h->n_total * h->real);   // zeros: DSLPIDControl.reset()
  if (e != cudaSuccess) {
    free_all(h); delete h;
    return fail(e == cudaErrorMemoryAllocation ? BD_ENOMEM : BD_ECUDA, "bd_create: device allocation failed: %s",
                cudaGetErrorString(e));
  }
  int rc = default_init_tables(h);
  if (rc) { free_all(h); delete h; return rc; }
  refresh_params(h);
  rc = do_reset(h, nullptr, nullptr, /*force_fixed=*/1, nullptr);   // __init__: no jitter (MultiHoverAviary.py:72)
  if (rc == BD_OK) {
    cudaError_t se = cudaDeviceSynchronize();
    if (se != cudaSuccess) rc = fail(BD_ECUDA, "bd_create: initial reset failed: %s", cudaGetErrorString(se));
  }
  if (rc) { free_all(h); delete h; return rc; }
  *out = h;
  return BD_OK;
}

void bd_destroy(bd_handle* h) {
  if (!h) return;
  DeviceGuard guard(h->cfg.device);
  free_all(h);
  delete h;
}

int bd_set_init_poses(bd_handle* h, const double* xyz_host, const double* rpy_host, int per_env) {
  if (!h || !xyz_host) return fail(BD_EINVAL, "bd_set_init_poses: null argument");
  DeviceGuard guard(h->cfg.device);
  BD_CUDA(cudaDeviceSynchronize());
  const size_t count = (size_t)(per_env ? h->cfg.n_envs : 1) * h->cfg.n_drones * 3;
  int rc = upload_table(h, xyz_host, count, &h->init_xyz);
  if (rc) return rc;
  if (rpy_host) {
    rc = upload_table(h, rpy_host, count, &h->init_rpy);
  } else {
    std::vector<double> z(count, 0.0);
    rc = upload_table(h, z.data(), count, &h->init_rpy);
  }
  if (rc) return rc;
  h->init_env_stride = per_env ? h->cfg.n_drones * 3 : 0;
  refresh_params(h);
  // like BaseAviary.__init__ -> _housekeeping: every env starts at the given poses, un-jittered
  rc = do_reset(h, nullptr, nullptr, /*force_fixed=*/1, nullptr);
  if (rc) return rc;
  BD_CUDA(cudaDeviceSynchronize());
  return BD_OK;
}

int bd_set_jitter(bd_handle* h, const void* jitter_dev, void* stream) {
  if (!h || !jitter_dev) return fail(BD_EINVAL, "bd_set_jitter: null argument");
  DeviceGuard guard(h->cfg.device);
  const size_t bytes = (size_t)h->n_total * 3 * h->real;
  if (!h->jitter) {
    BD_CUDA(cudaMalloc(&h->jitter, bytes));
    refresh_params(h);
  }
  BD_CUDA(cudaMemcpyAsync(h->jitter, jitter_dev, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return BD_OK;
}

int bd_reset(bd_handle* h, const uint8_t* env_mask_dev, float* obs_dev, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_reset: null handle");
  if (h->cfg.reset_mode == BD_RESET_JITTER_BUFFER && h->cfg.task == BD_TASK_MULTIHOVER && !h->jitter)
    return fail(BD_EINVAL, "bd_reset: BD_RESET_JITTER_BUFFER needs bd_set_jitter() first");
  DeviceGuard guard(h->cfg.device);
  return do_reset(h, env_mask_dev, obs_dev, 0, (cudaStream_t)stream);
}

int bd_step(bd_handle* h, const void* actions_dev, float* obs_dev, void* reward_dev,
            uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_step: null handle");
  if (!actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev)
    return fail(BD_EINVAL, "bd_step: actions, obs, reward, terminated and truncated are required");
  // 128-bit accesses: action rows when A == 4 (float4 loads), observation rows when D % 4 == 0 on the fast
  // kernel.  Other shapes (ONE_D_RPM: A = 1, D = 27; PID: A = 3, D = 57) take scalar paths and any 4-byte
  // aligned pointer — a rollout buffer slot obs[t+1] is 16-byte aligned only when N*M*D % 4 == 0.
  const size_t act_elem_sz = (h->cfg.precision == BD_F64 && !h->cfg.action_is_f32) ? 8 : 4;
  if ((h->A == 4 && ((uintptr_t)actions_dev & 15)) || ((uintptr_t)actions_dev & (act_elem_sz - 1)))
    return fail(BD_EINVAL, "bd_step: actions must be 16-byte aligned (A = 4) / element aligned");
  const bool obs_vec = h->spec.impl == 1 && h->A == 4 && (h->D & 3) == 0;
  if ((obs_vec && ((uintptr_t)obs_dev & 15)) || ((uintptr_t)obs_dev & 3))
    return fail(BD_EINVAL, "bd_step: obs must be 16-byte aligned (A = 4, D %% 4 == 0) / 4-byte aligned");
  if (h->poisoned)
    return fail(BD_ECUDA, "bd_step: an earlier launch of this handle failed half-way through a step; destroy the handle");
  if (h->cfg.auto_reset && h->cfg.reset_mode == BD_RESET_JITTER_BUFFER &&
      h->cfg.task == BD_TASK_MULTIHOVER && !h->jitter)
    return fail(BD_EINVAL, "bd_step: BD_RESET_JITTER_BUFFER needs bd_set_jitter() first");
  DeviceGuard guard(h->cfg.device);
  if (!h->graph_mode) {
    // Captured launches are replayed with frozen parameters, so from the first capture on
    // the ring head comes from the device-resident counter (kept current by every launch).
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing((cudaStream_t)stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone)
      h->graph_mode = true;
  }
  cudaError_t e = cudaSuccess;
  with_params(h, [&](auto& P) {
    P.host_total = h->graph_mode ? -1 : (int)h->total_steps;
    P.host_head = (int)(h->total_steps % h->B);
    P.actions = actions_dev;
    P.obs = obs_dev;
    P.reward = (decltype(P.reward))reward_dev;
    P.terminated = terminated_dev;
    P.truncated = truncated_dev;
    P.terminal_obs = terminal_obs_dev;
    P.obs_aligned = (((uintptr_t)obs_dev & 15) == 0) ? 1 : 0;
    P.early_prefetch = h->restored ? 0 : 1;
    e = bd::launch_step(h->spec, &P, (cudaStream_t)stream);
    P.obs_aligned = 1;
    P.early_prefetch = 1;
  });
  // the host step count follows the tile epochs the launch will publish: only a launch that was accepted counts
  if (e != cudaSuccess) return fail(BD_ECUDA, "step kernel launch failed: %s", cudaGetErrorString(e));
  h->restored = false;
  h->launches++;
  h->total_steps++;
  if (h->total_steps >= (long long)h->B * ((1 << 30) / h->B)) {
    h->total_steps = 0;
    if (h->pipeline) {   // tile epochs restart with the step count (once per ~1e9 steps)
      cudaStreamSynchronize((cudaStream_t)stream);
      cudaMemset(h->tile_epoch, 0, (size_t)epoch_tiles(h) * sizeof(int));
      cudaMemset(h->finished, 0, sizeof(unsigned long long));
      cudaMemset(h->gsteps + 8, 0, 8 * sizeof(int));
    }
  }
  return BD_OK;
}

}  // extern "C"

namespace {
int ensure_compact_buffers(bd_handle* h, int set, int cap) {
  const size_t row_bytes = (size_t)h->cfg.n_drones * h->D * sizeof(float);
  if (!h->c_blockcnt) BD_CUDA(cudaMalloc((void**)&h->c_blockcnt, (size_t)bd::compact_blocks(h->cfg.n_envs) * sizeof(int)));
  if (!h->c_total) BD_CUDA(cudaMalloc((void**)&h->c_total, sizeof(int)));
  if (!h->c_idx_dev) BD_CUDA(cudaMalloc((void**)&h->c_idx_dev, ((size_t)h->cfg.n_envs + 1) * sizeof(int)));
  if (!h->hs_compact) BD_CUDA(cudaEventCreateWithFlags(&h->hs_compact, cudaEventDisableTiming));
  if (cap > h->c_cap_dev) {
    if (h->c_rows_dev) { BD_CUDA(cudaDeviceSynchronize()); cudaFree(h->c_rows_dev); h->c_rows_dev = nullptr; h->c_cap_dev = 0; }
    BD_CUDA(cudaMalloc((void**)&h->c_rows_dev, (size_t)cap * row_bytes));
    h->c_cap_dev = cap;
  }
  if (!h->c_host[set])
    BD_CUDA(cudaHostAlloc((void**)&h->c_host[set], ((size_t)h->cfg.n_envs + 1) * sizeof(int), cudaHostAllocDefault));
  if (cap > h->c_cap[set]) {
    if (h->c_rows_host[set]) { cudaFreeHost(h->c_rows_host[set]); h->c_rows_host[set] = nullptr; h->c_cap[set] = 0; }
    BD_CUDA(cudaHostAlloc((void**)&h->c_rows_host[set], (size_t)cap * row_bytes, cudaHostAllocDefault));
    h->c_cap[set] = cap;
  }
  return BD_OK;
}
// compact = true: terminal observations stay in the device-side (N,M,D) buffer; after the step the finished envs'
// rows are gathered (ascending env order) into a compact device buffer by small kernels that run inside the chunk
// pipeline; after the flags have arrived the host copies exactly n_done rows (GPU stores straight into mapped host
// memory were tried first: 16-byte PCIe writes, 2 ms for 3 MB).
int step_host_impl(bd_handle* h, const void* actions_host, float* obs_host, void* reward_host,
                   uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host, bool compact,
                   void* stream);
}  // namespace

extern "C" {

int bd_step_host(bd_handle* h, const void* actions_host, float* obs_host, void* reward_host,
                 uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host,
                 void* stream) {
  return step_host_impl(h, actions_host, obs_host, reward_host, terminated_host, truncated_host, terminal_obs_host, false,
                        stream);
}

int bd_step_host_compact(bd_handle* h, const void* actions_host, float* obs_host, void* reward_host,
                         uint8_t* terminated_host, uint8_t* truncated_host, int32_t* n_done,
                         const int32_t** done_idx, const float** terminal_rows, void* stream) {
  if (!n_done || !done_idx || !terminal_rows) return fail(BD_EINVAL, "bd_step_host_compact: null output argument");
  *n_done = 0; *done_idx = nullptr; *terminal_rows = nullptr;
  int rc = step_host_impl(h, actions_host, obs_host, reward_host, terminated_host, truncated_host, nullptr, true, stream);
  if (rc) return rc;
  const int set = h->c_flip;       // the set this call filled
  *n_done = h->c_host[set][0];
  *done_idx = h->c_host[set] + 1;
  *terminal_rows = h->c_rows_host[set];
  return BD_OK;
}

}  // extern "C"

namespace {
int step_host_impl(bd_handle* h, const void* actions_host, float* obs_host, void* reward_host,
                   uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host, bool compact,
                   void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_step_host: null handle");
  if (!actions_host || !obs_host || !reward_host || !terminated_host || !truncated_host)
    return fail(BD_EINVAL, "bd_step_host: actions, obs, reward, terminated and truncated are required");
  if (h->poisoned)
    return fail(BD_ECUDA, "bd_step_host: an earlier launch of this handle failed half-way through a step; destroy the handle");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t act_elem = (h->cfg.precision == BD_F64 && !h->cfg.action_is_f32) ? 8 : 4;
  const size_t act_bytes = (size_t)h->n_total * h->A * act_elem;
  const size_t obs_bytes = (size_t)h->n_total * h->D * sizeof(float);
  const size_t n = (size_t)h->cfg.n_envs;
  if (!h->h_actions) {
    BD_CUDA(cudaMalloc(&h->h_actions, act_bytes));
    BD_CUDA(cudaMalloc((void**)&h->h_obs, obs_bytes));
    BD_CUDA(cudaMalloc(&h->h_reward, n * h->real));
    BD_CUDA(cudaMalloc((void**)&h->h_term, n));
    BD_CUDA(cudaMalloc((void**)&h->h_trunc, n));
  }
  const bool want_tobs = terminal_obs_host != nullptr || compact;
  if (want_tobs && !h->h_tobs) {
    BD_CUDA(cudaMalloc((void**)&h->h_tobs, obs_bytes));
    BD_CUDA(cudaMemsetAsync(h->h_tobs, 0, obs_bytes, st));
  }
  if (compact) {
    h->c_flip ^= 1;
    const int set = h->c_flip;
    // worst case up front (every env finished): growing the page-locked staging later costs 0.2 - 0.5 s per
    // cudaFreeHost + cudaHostAlloc (measured: two such calls inside a 20-step window tripled its mean), and the share of
    // finished envs climbs for many steps after a reset, so any smaller start would grow several times
    int want = h->cfg.n_envs;
    int rc = ensure_compact_buffers(h, set, want);
    if (rc) return rc;
  }
  // Pipeline over chunks of whole tiles: while the copy engine drains chunk k's observations to the host,
  // chunk k+1's actions go up and its tiles are stepped.  One control step = `chunks` sub-range launches of the
  // same kernel with the same step count; only the last one advances the device-resident counter.
  const int block_rows = h->spec.impl == 1 ? (4 * h->EW) * h->cfg.n_drones : h->E * h->cfg.n_drones;   // drones per tile
  const int n_blocks = (int)((h->n_total + block_rows - 1) / block_rows);
  int chunks = (int)(obs_bytes >> 21);   // at least 2 MB of observations per chunk, at most 8 chunks
  if (chunks > 8) chunks = 8;
  if (chunks > n_blocks) chunks = n_blocks;
  if (chunks <= 1 || h->graph_mode) {
    BD_CUDA(cudaMemcpyAsync(h->h_actions, actions_host, act_bytes, cudaMemcpyHostToDevice, st));
    int rc = bd_step(h, h->h_actions, h->h_obs, h->h_reward, h->h_term, h->h_trunc,
                     want_tobs ? h->h_tobs : nullptr, stream);
    if (rc) return rc;
    if (compact) {
      const int set = h->c_flip;
      cudaError_t ce = bd::launch_compact_done(h->h_term, h->h_trunc, 0, h->cfg.n_envs, 1, h->c_blockcnt, h->c_total, h->h_tobs,
                                               h->cfg.n_drones * h->D, h->c_cap_dev, h->c_idx_dev, h->c_rows_dev, st);
      h->launches += 3;
      (void)set;
      if (ce != cudaSuccess) return fail(BD_ECUDA, "compaction kernels failed to launch: %s", cudaGetErrorString(ce));
    }
    BD_CUDA(cudaMemcpyAsync(obs_host, h->h_obs, obs_bytes, cudaMemcpyDeviceToHost, st));
    if (terminal_obs_host)
      BD_CUDA(cudaMemcpyAsync(terminal_obs_host, h->h_tobs, obs_bytes, cudaMemcpyDeviceToHost, st));
  } else {
    if (h->cfg.auto_reset && h->cfg.reset_mode == BD_RESET_JITTER_BUFFER && h->cfg.task == BD_TASK_MULTIHOVER && !h->jitter)
      return fail(BD_EINVAL, "bd_step: BD_RESET_JITTER_BUFFER needs bd_set_jitter() first");
    if (!h->hs_a) {
      BD_CUDA(cudaStreamCreateWithFlags(&h->hs_a, cudaStreamNonBlocking));
      BD_CUDA(cudaStreamCreateWithFlags(&h->hs_b, cudaStreamNonBlocking));
      BD_CUDA(cudaEventCreateWithFlags(&h->hs_start, cudaEventDisableTiming));
      BD_CUDA(cudaEventCreateWithFlags(&h->hs_done, cudaEventDisableTiming));
      for (auto& ev : h->hs_chunk) BD_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    BD_CUDA(cudaEventRecord(h->hs_start, st));
    BD_CUDA(cudaStreamWaitEvent(h->hs_a, h->hs_start, 0));
    BD_CUDA(cudaStreamWaitEvent(h->hs_b, h->hs_start, 0));
    const size_t act_row = (size_t)h->A * act_elem, obs_row = (size_t)h->D * sizeof(float);
    cudaError_t e = cudaSuccess;
    for (int c = 0; c < chunks && e == cudaSuccess; ++c) {
      const int b0 = (int)((long long)n_blocks * c / chunks), b1 = (int)((long long)n_blocks * (c + 1) / chunks);
      const long long g0 = (long long)b0 * block_rows;
      long long g1 = (long long)b1 * block_rows;
      if (g1 > h->n_total) g1 = h->n_total;
      const size_t rows = (size_t)(g1 - g0);
      BD_CUDA(cudaMemcpyAsync((char*)h->h_actions + g0 * act_row, (const char*)actions_host + g0 * act_row, rows * act_row,
                              cudaMemcpyHostToDevice, h->hs_a));
      with_params(h, [&](auto& P) {
        P.host_total = (int)h->total_steps;
        P.host_head = (int)(h->total_steps % h->B);
        P.actions = h->h_actions;
        P.obs = h->h_obs;
        P.reward = (decltype(P.reward))h->h_reward;
        P.terminated = h->h_term;
        P.truncated = h->h_trunc;
        P.terminal_obs = want_tobs ? h->h_tobs : nullptr;
        P.block0 = b0; P.grid_blocks = b1 - b0; P.advance = (c == chunks - 1) ? 1 : 0;
        P.early_prefetch = h->restored ? 0 : 1;
        e = bd::launch_step(h->spec, &P, h->hs_a);
        P.block0 = 0; P.grid_blocks = 0; P.advance = 1; P.early_prefetch = 1;
      });
      if (e != cudaSuccess) {
        // chunks 0..c-1 have stepped their tiles and will publish epochs for a step that never completed
        if (c > 0) h->poisoned = true;
        break;
      }
      h->launches++;
      BD_CUDA(cudaEventRecord(h->hs_chunk[c], h->hs_a));
      BD_CUDA(cudaStreamWaitEvent(h->hs_b, h->hs_chunk[c], 0));
      if (compact) {   // this chunk's finished envs are gathered (device to device) while its observations travel
        const int env_per_block = block_rows / h->cfg.n_drones;
        const int e0 = b0 * env_per_block;
        int e1 = b1 * env_per_block;
        if (e1 > h->cfg.n_envs) e1 = h->cfg.n_envs;
        cudaError_t ce = bd::launch_compact_done(h->h_term, h->h_trunc, e0, e1, c == 0 ? 1 : 0, h->c_blockcnt, h->c_total, h->h_tobs,
                                                 h->cfg.n_drones * h->D, h->c_cap_dev, h->c_idx_dev, h->c_rows_dev, h->hs_a);
        h->launches += 3;
        if (ce != cudaSuccess) return fail(BD_ECUDA, "compaction kernels failed to launch: %s", cudaGetErrorString(ce));
      }
      BD_CUDA(cudaMemcpyAsync((char*)obs_host + g0 * obs_row, (const char*)h->h_obs + g0 * obs_row, rows * obs_row,
                              cudaMemcpyDeviceToHost, h->hs_b));
      if (terminal_obs_host)
        BD_CUDA(cudaMemcpyAsync((char*)terminal_obs_host + g0 * obs_row, (const char*)h->h_tobs + g0 * obs_row,
                                rows * obs_row, cudaMemcpyDeviceToHost, h->hs_b));
    }
    if (e != cudaSuccess) return fail(BD_ECUDA, "step kernel launch failed: %s", cudaGetErrorString(e));
    h->restored = false;
    h->total_steps++;
    if (h->total_steps >= (long long)h->B * ((1 << 30) / h->B)) {
      h->total_steps = 0;
      if (h->pipeline) {
        cudaDeviceSynchronize();
        cudaMemset(h->tile_epoch, 0, (size_t)epoch_tiles(h) * sizeof(int));
        cudaMemset(h->finished, 0, sizeof(unsigned long long));
        cudaMemset(h->gsteps + 8, 0, 8 * sizeof(int));
      }
    }
    BD_CUDA(cudaEventRecord(h->hs_done, h->hs_b));   // hs_b has waited for every chunk of hs_a
    BD_CUDA(cudaStreamWaitEvent(st, h->hs_done, 0));
    if (compact) {                                   // ... but not for the compaction kernels behind the last chunk
      BD_CUDA(cudaEventRecord(h->hs_compact, h->hs_a));
      BD_CUDA(cudaStreamWaitEvent(st, h->hs_compact, 0));
    }
  }
  BD_CUDA(cudaMemcpyAsync(reward_host, h->h_reward, n * h->real, cudaMemcpyDeviceToHost, st));
  BD_CUDA(cudaMemcpyAsync(terminated_host, h->h_term, n, cudaMemcpyDeviceToHost, st));
  BD_CUDA(cudaMemcpyAsync(truncated_host, h->h_trunc, n, cudaMemcpyDeviceToHost, st));
  if (compact) {
    const int row_floats = h->cfg.n_drones * h->D;
    const int set = h->c_flip;
    // the count travels with the flags; then exactly n_done indices and rows
    BD_CUDA(cudaMemcpyAsync(h->c_host[set], h->c_idx_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
    BD_CUDA(cudaStreamSynchronize(st));
    int cnt = h->c_host[set][0];
    if (cnt > h->c_cap_dev) {   // more finished envs than the staging holds: grow it and gather again (rare)
      int rc = ensure_compact_buffers(h, set, cnt + cnt / 4);
      if (rc) return rc;
      cudaError_t e = bd::launch_compact_done(h->h_term, h->h_trunc, 0, h->cfg.n_envs, 1, h->c_blockcnt, h->c_total, h->h_tobs,
                                              row_floats, h->c_cap_dev, h->c_idx_dev, h->c_rows_dev, st);
      h->launches += 3;
      if (e != cudaSuccess) return fail(BD_ECUDA, "compaction kernels failed to launch: %s", cudaGetErrorString(e));
    }
    if (cnt > h->c_cap[set]) {
      int rc = ensure_compact_buffers(h, set, cnt + cnt / 4);
      if (rc) return rc;
    }
    if (cnt > 0) {
      BD_CUDA(cudaMemcpyAsync(h->c_host[set] + 1, h->c_idx_dev + 1, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, st));
      BD_CUDA(cudaMemcpyAsync(h->c_rows_host[set], h->c_rows_dev, (size_t)cnt * row_floats * sizeof(float), cudaMemcpyDeviceToHost, st));
      BD_CUDA(cudaStreamSynchronize(st));
    }
    return BD_OK;
  }
  BD_CUDA(cudaStreamSynchronize(st));
  return BD_OK;
}
}  // namespace

extern "C" {

// K control steps with one host call (launch-bound regimes: small batches, random-action sweeps).  The K action
// sets and K output slots are contiguous arrays; identical to K bd_step calls.
int bd_step_many(bd_handle* h, int k, const void* actions_dev, float* obs_dev, void* reward_dev, uint8_t* terminated_dev,
                 uint8_t* truncated_dev, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_step_many: null handle");
  if (k < 0) return fail(BD_EINVAL, "bd_step_many: k must be >= 0");
  const size_t act_elem = (h->cfg.precision == BD_F64 && !h->cfg.action_is_f32) ? 8 : 4;
  const size_t act_step = (size_t)h->n_total * h->A * act_elem, obs_step = (size_t)h->n_total * h->D;
  const size_t n = (size_t)h->cfg.n_envs;
  // The fast tile kernel takes a tile through all k steps in ONE launch (states in registers, history in shared memory):
  // a small batch is bound by the latency of a step's launch -> load -> compute -> store chain, not by bandwidth.
  // BD_STEP_MANY=loop keeps k launches (A/B runs, tests).  Needs rows that leave as TMA bulk stores.
  static const bool force_loop = [] { const char* e = getenv("BD_STEP_MANY"); return e && strcmp(e, "loop") == 0; }();
  const long long wrap = (long long)h->B * ((1 << 30) / h->B);
  const size_t tile_bytes = (size_t)(4 * h->EW) * h->cfg.n_drones * h->D * 4;
  const size_t last_rows = (size_t)(h->n_total % ((long long)(4 * h->EW) * h->cfg.n_drones));
  const bool one_launch = !force_loop && h->many_mode == 0 && k >= 2 && h->spec.impl == 1 && h->cfg.precision == BD_F32 && !h->poisoned &&
                          actions_dev && obs_dev && reward_dev && terminated_dev && truncated_dev &&
                          ((uintptr_t)obs_dev & 15) == 0 && ((obs_step * 4) & 15) == 0 && (tile_bytes & 15) == 0 &&
                          ((last_rows * h->D * 4) & 15) == 0 && (h->A != 4 || (((uintptr_t)actions_dev & 15) == 0 && (act_step & 15) == 0)) &&
                          2 * tile_bytes <= 200 * 1024 && h->total_steps + k < wrap &&
                          !(h->cfg.auto_reset && h->cfg.reset_mode == BD_RESET_JITTER_BUFFER && h->cfg.task == BD_TASK_MULTIHOVER && !h->jitter);
  if (one_launch) {
    DeviceGuard guard(h->cfg.device);
    if (!h->graph_mode) {
      cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
      if (cudaStreamIsCapturing((cudaStream_t)stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) h->graph_mode = true;
    }
    cudaError_t e = cudaSuccess;
    bd::Params<float>& P = h->pf;
    P.host_total = h->graph_mode ? -1 : (int)h->total_steps;
    P.host_head = (int)(h->total_steps % h->B);
    P.actions = actions_dev;
    P.obs = obs_dev;
    P.reward = (float*)reward_dev;
    P.terminated = terminated_dev;
    P.truncated = truncated_dev;
    P.terminal_obs = nullptr;
    e = bd::launch_step_tile_many(h->spec.task, h->spec.act_a, P, k, (long long)(act_step / act_elem), (long long)obs_step, (long long)n,
                                  h->spec, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(BD_ECUDA, "bd_step_many: kernel launch failed: %s", cudaGetErrorString(e));
    h->restored = false;   // a plain launch: it started after the unpack kernel had completed
    h->launches++;
    h->total_steps += k;
    return BD_OK;
  }
  for (int i = 0; i < k; ++i) {
    int rc = bd_step(h, (const char*)actions_dev + i * act_step, obs_dev + i * obs_step, (char*)reward_dev + i * n * h->real,
                     terminated_dev + i * n, truncated_dev + i * n, nullptr, stream);
    if (rc) return rc;
  }
  return BD_OK;
}

// Benchmark helper: a one-thread kernel that holds `stream` until the host stores a non-zero value into *flag (page-locked
// host memory, read by the GPU through its mapped address) — so that a caller can enqueue a whole timed window behind it
// and the device timeline of the window has no host-side gaps.  Bounded: gives up after ~2^32 SM clocks (2 s).
int bd_stream_gate(const uint32_t* flag_mapped, void* stream) {
  if (!flag_mapped) return fail(BD_EINVAL, "bd_stream_gate: null flag");
  cudaError_t e = bd::launch_gate(flag_mapped, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(BD_ECUDA, "bd_stream_gate: %s", cudaGetErrorString(e));
  return BD_OK;
}

// bd_step_many: mode 0 (default) = one launch for the k steps where the configuration allows it, 1 = always k launches
// (what a closed-loop caller's steps cost; benchmarks of the per-step kernel).
int bd_set_step_many_mode(bd_handle* h, int mode) {
  if (!h || mode < 0 || mode > 1) return fail(BD_EINVAL, "bd_set_step_many_mode: mode must be 0 or 1");
  h->many_mode = mode;
  return BD_OK;
}

// RNG state of the on-device re-spawn draws (the counterpart of the workers' np.random states the reference
// checkpoints, mappo/mappo.py:203-229, subproc_vec_env.py:101-112): state4 = {seed, Philox step counter
// (= philox_base + control steps so far), explicit-reset epoch, 0}.  Setting it makes a resumed run continue
// the stream instead of replaying it; the action ring and the drone states are not part of it.
int bd_get_rng_state(const bd_handle* h, uint64_t* state4) {
  if (!h || !state4) return fail(BD_EINVAL, "bd_get_rng_state: null argument");
  state4[0] = h->cfg.seed;
  state4[1] = (uint64_t)(uint32_t)(h->philox_base + (uint32_t)h->total_steps);
  state4[2] = (uint64_t)h->reset_epoch;
  state4[3] = 0;
  return BD_OK;
}
int bd_set_rng_state(bd_handle* h, const uint64_t* state4) {
  if (!h || !state4) return fail(BD_EINVAL, "bd_set_rng_state: null argument");
  if (h->graph_mode) return fail(BD_EINVAL, "bd_set_rng_state: not available after a step was captured into a CUDA graph");
  h->cfg.seed = state4[0];
  h->philox_base = (uint32_t)state4[1] - (uint32_t)h->total_steps;
  h->reset_epoch = (int)state4[2];
  refresh_params(h);
  return BD_OK;
}

// Test hook: overwrite one tile's epoch (stream ordered).  A value below the step count makes the next pipelined
// launch wait for an epoch nobody will publish; the bounded spin must then trap instead of hanging the GPU.
int bd_debug_set_tile_epoch(bd_handle* h, int tile, int value, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_debug_set_tile_epoch: null handle");
  if (tile < 0 || tile >= (int)epoch_tiles(h)) return fail(BD_EINVAL, "bd_debug_set_tile_epoch: tile out of range");
  DeviceGuard guard(h->cfg.device);
  cudaError_t e = bd::launch_set_epoch(h->tile_epoch, tile, value, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(BD_ECUDA, "bd_debug_set_tile_epoch: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_get_state(bd_handle* h, void* state20_dev, void* rates_dev, int32_t* step_counter_dev, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_get_state: null handle");
  DeviceGuard guard(h->cfg.device);
  cudaError_t e = bd::launch_get_state(h->cfg.precision, params_ptr(h), state20_dev, rates_dev,
                                       step_counter_dev, (cudaStream_t)stream);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "get_state kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_set_state(bd_handle* h, const void* kin13_dev, const void* targets_dev,
                 const int32_t* step_counter_dev, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_set_state: null handle");
  DeviceGuard guard(h->cfg.device);
  cudaError_t e = bd::launch_set_state(h->cfg.precision, params_ptr(h), kin13_dev, targets_dev,
                                       step_counter_dev, (cudaStream_t)stream);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "set_state kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_get_targets(bd_handle* h, void* targets_dev, void* stream) {
  if (!h || !targets_dev) return fail(BD_EINVAL, "bd_get_targets: null argument");
  DeviceGuard guard(h->cfg.device);
  cudaError_t e = bd::launch_get_targets(h->cfg.precision, params_ptr(h), targets_dev, (cudaStream_t)stream);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "get_targets kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_get_controller_state(bd_handle* h, void* ctrl9_dev, void* stream) {
  if (!h || !ctrl9_dev) return fail(BD_EINVAL, "bd_get_controller_state: null argument");
  if (!h->ctrl) return fail(BD_EINVAL, "bd_get_controller_state: the action type has no controller");
  DeviceGuard guard(h->cfg.device);
  cudaError_t e = bd::launch_ctrl_state(h->cfg.precision, params_ptr(h), ctrl9_dev, nullptr, 0, (cudaStream_t)stream);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "ctrl_state kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_set_controller_state(bd_handle* h, const void* ctrl9_dev, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_set_controller_state: null handle");
  if (!h->ctrl) return fail(BD_EINVAL, "bd_set_controller_state: the action type has no controller");
  DeviceGuard guard(h->cfg.device);
  cudaError_t e = bd::launch_ctrl_state(h->cfg.precision, params_ptr(h), nullptr, ctrl9_dev, 1, (cudaStream_t)stream);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "ctrl_state kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_set_action_f32(bd_handle* h, int is_f32) {
  if (!h) return fail(BD_EINVAL, "bd_set_action_f32: null handle");
  if (h->cfg.precision == BD_F32 && !is_f32)
    return fail(BD_EINVAL, "bd_set_action_f32: BD_F32 handles take float actions only");
  h->cfg.action_is_f32 = is_f32 ? 1 : 0;
  if (h->h_actions) {   // staging buffer of bd_step_host is sized for the action element type
    DeviceGuard guard(h->cfg.device);
    cudaFree(h->h_actions); cudaFree(h->h_obs); cudaFree(h->h_reward); cudaFree(h->h_term); cudaFree(h->h_trunc);
    h->h_actions = nullptr; h->h_obs = nullptr; h->h_reward = nullptr; h->h_term = nullptr; h->h_trunc = nullptr;
  }
  refresh_params(h);
  return BD_OK;
}

int bd_episode_stats(bd_handle* h, double* stats3_dev, int reset, void* stream) {
  if (!h) return fail(BD_EINVAL, "bd_episode_stats: null handle");
  if (!h->ep_ret) return fail(BD_EINVAL, "bd_episode_stats: the handle was created with track_episodes = 0");
  DeviceGuard guard(h->cfg.device);
  cudaError_t e = bd::launch_episode_stats(h->ep_acc, stats3_dev, reset, (cudaStream_t)stream);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "episode_stats kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_l2_plan(int n_envs, int n_drones, int act_dim, int buf_slots, int track_episodes, int64_t l2_bytes,
               const char* force, int* keep_state, int* keep_slots) {
  if (!keep_state || !keep_slots) return fail(BD_EINVAL, "bd_l2_plan: null output");
  if (n_envs < 1 || n_drones < 1 || act_dim < 1 || buf_slots < 1 || l2_bytes < 0)
    return fail(BD_EINVAL, "bd_l2_plan: bad shape");
  *keep_state = 0;
  *keep_slots = 0;
  if (force && *force) {   // an empty override counts as unset
    if (strcmp(force, "off") == 0) return BD_OK;
    *keep_state = 1;
    if (strcmp(force, "state") == 0) return BD_OK;
    char* end = nullptr;
    const long k = strtol(force, &end, 10);
    if (end == force || *end != '\0' || k < 0) {
      *keep_state = 0;
      return fail(BD_EINVAL, "BD_L2_KEEP=%s: expected off, state or a slot count", force);
    }
    *keep_slots = (int)(k < buf_slots - 1 ? k : buf_slots - 1);
    return BD_OK;
  }
  const long long n = (long long)n_envs * n_drones;
  const long long state = n * 64 + (long long)n_envs * (track_episodes ? 8 : 4);   // 4 float4 planes, counter, return
  const long long slot = n * act_dim * 4;
  // evict_last bytes that still pay off, measured (profiles/README.md, "L2 residency budget"): 3/10 of the L2, about
  // 40 MB on a B200.  Beyond it the step gets slower again — kept lines crowd out the streaming traffic, and every tile
  // runs on a different SM each step, so a line may be wanted in both L2 partitions.
  const long long budget = l2_bytes * 3 / 10;
  if (state > budget) return BD_OK;
  *keep_state = 1;
  const long long k = (budget - state) / slot;
  *keep_slots = (int)(k < buf_slots - 1 ? k : buf_slots - 1);
  return BD_OK;
}

int bd_l2_policy(const bd_handle* h, int* keep_state, int* keep_slots) {
  if (!h || !keep_state || !keep_slots) return fail(BD_EINVAL, "bd_l2_policy: null argument");
  *keep_state = h->l2_keep_state;
  *keep_slots = h->l2_keep_slots;
  return BD_OK;
}

}  // extern "C"

namespace bd {
SnapLayout snap_layout(long long n_envs, long long n_drones, int act_dim, int buf_slots, int real_bytes, int flags) {
  SnapLayout L;
  const long long n = n_envs * n_drones;
  long long off = (long long)sizeof(SnapHeader);
  auto plane = [&](long long bytes) {
    const long long at = off;
    off += (bytes + kSnapAlign - 1) / kSnapAlign * kSnapAlign;
    return at;
  };
  for (int k = 0; k < 4; ++k) L.kin[k] = plane(n * 4 * real_bytes);
  L.angv = (flags & BD_SNAP_ANGV) ? plane(n * 4 * real_bytes) : -1;
  L.ctrl_stride = (n * real_bytes + kSnapAlign - 1) / kSnapAlign * kSnapAlign;
  L.ctrl = -1;
  if (flags & BD_SNAP_CTRL) {
    L.ctrl = off;
    off += (long long)kCtrlPlanesHost * L.ctrl_stride;
  }
  L.ring_stride = (n * act_dim * 4 + kSnapAlign - 1) / kSnapAlign * kSnapAlign;
  L.ring = off;
  off += (long long)buf_slots * L.ring_stride;
  L.stepc = plane(n_envs * 4);
  L.ep_ret = (flags & BD_SNAP_EPISODES) ? plane(n_envs * 4) : -1;
  L.bytes = off;
  return L;
}
}  // namespace bd

namespace {

// FNV-1a over everything a restore needs to match besides N and M (which the header carries in the clear): task,
// action type, airframe, precision, aero terms, integrator, frequencies, airframe / controller / spiral constants and
// the episode length.  Seed, reset behaviour, action dtype, L2 plan and the optional planes may differ.
uint64_t snap_fingerprint(const bd_config& c) {
  uint64_t f = 1469598103934665603ull;
  auto mix = [&](const void* p, size_t n) {
    const unsigned char* b = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < n; ++i) { f ^= b[i]; f *= 1099511628211ull; }
  };
  const int32_t ints[] = {c.task, c.act_type, c.drone_model, c.precision, c.aero_flags, c.integrator, c.pyb_freq, c.ctrl_freq};
  mix(ints, sizeof(ints));
  const double dbl[] = {c.episode_len_sec, c.mass, c.arm, c.kf, c.km, c.ixx, c.iyy, c.izz, c.g, c.thrust2weight,
                        c.gnd_eff_coeff, c.prop_radius, c.drag_coeff_xy, c.drag_coeff_z, c.dw_coeff_1, c.dw_coeff_2,
                        c.dw_coeff_3, c.spiral_radius, c.spiral_period, c.height_rate, c.ctrl_mass, c.ctrl_kf, c.speed_limit};
  mix(dbl, sizeof(dbl));
  mix(c.prop_xy, sizeof(c.prop_xy));
  mix(c.target_center, sizeof(c.target_center));
  return f;
}

int snap_flags(const bd_handle* h) {
  return (h->cfg.keep_ang_vel ? BD_SNAP_ANGV : 0) | (h->ctrl ? BD_SNAP_CTRL : 0) | (h->ep_ret ? BD_SNAP_EPISODES : 0);
}

bd::SnapLayout handle_layout(const bd_handle* h, int flags) {
  return bd::snap_layout(h->cfg.n_envs, h->cfg.n_drones, h->A, h->B, (int)h->real, flags);
}

// the checks bd_save_snapshot and bd_load_snapshot share
int snap_precheck(bd_handle* h, const void* snap, void* stream, const char* what) {
  if (!h || !snap) return fail(BD_EINVAL, "%s: null argument", what);
  if ((uintptr_t)snap & (bd::kSnapAlign - 1)) return fail(BD_EINVAL, "%s: the snapshot buffer must be 256-byte aligned", what);
  if (h->poisoned)
    return fail(BD_EINVAL, "%s: an earlier launch of this handle failed half-way through a step; destroy the handle", what);
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing((cudaStream_t)stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone)
    return fail(BD_EINVAL, "%s: not capturable (the stream is capturing a CUDA graph)", what);
  return BD_OK;
}

}  // namespace

extern "C" {

int bd_snapshot_layout(int n_envs, int n_drones, int act_dim, int buf_slots, int precision, int flags, int64_t* bytes) {
  if (!bytes) return fail(BD_EINVAL, "bd_snapshot_layout: null output");
  *bytes = 0;
  if (n_envs < 1 || n_drones < 1 || n_drones > bd::kMaxDrones || act_dim < 1 || act_dim > 4 || buf_slots < 1)
    return fail(BD_EINVAL, "bd_snapshot_layout: bad shape");
  if (precision != BD_F32 && precision != BD_F64) return fail(BD_EINVAL, "bd_snapshot_layout: unknown precision");
  if (flags & ~(BD_SNAP_ANGV | BD_SNAP_CTRL | BD_SNAP_EPISODES)) return fail(BD_EINVAL, "bd_snapshot_layout: unknown flag");
  *bytes = bd::snap_layout(n_envs, n_drones, act_dim, buf_slots, precision == BD_F64 ? 8 : 4, flags).bytes;
  return BD_OK;
}

int64_t bd_snapshot_bytes(const bd_handle* h) {
  if (!h) return fail(BD_EINVAL, "bd_snapshot_bytes: null handle");
  return handle_layout(h, snap_flags(h)).bytes;
}

int bd_save_snapshot(bd_handle* h, void* snap_dev, void* stream) {
  int rc = snap_precheck(h, snap_dev, stream, "bd_save_snapshot");
  if (rc) return rc;
  DeviceGuard guard(h->cfg.device);
  const int flags = snap_flags(h);
  const bd::SnapLayout L = handle_layout(h, flags);
  bd::SnapHeader hdr;
  memset(&hdr, 0, sizeof(hdr));
  hdr.magic = bd::kSnapMagic; hdr.version = bd::kSnapVersion;
  hdr.precision = h->cfg.precision; hdr.n_envs = h->cfg.n_envs; hdr.n_drones = h->cfg.n_drones;
  hdr.act_dim = h->A; hdr.buf_slots = h->B; hdr.flags = (uint32_t)flags;
  hdr.fingerprint = snap_fingerprint(h->cfg);
  hdr.bytes = L.bytes;
  bd_get_rng_state(h, hdr.rng);   // rng[1] is recomputed on the device from the step count the ring head uses
  hdr.task = h->cfg.task; hdr.act_type = h->cfg.act_type; hdr.drone_model = h->cfg.drone_model;
  hdr.aero_flags = h->cfg.aero_flags; hdr.integrator = h->cfg.integrator;
  hdr.pyb_freq = h->cfg.pyb_freq; hdr.ctrl_freq = h->cfg.ctrl_freq;
  // a plain launch (no programmatic serialization): it starts after the previous step has completed
  cudaError_t e = bd::launch_snapshot(h->cfg.precision, params_ptr(h), snap_dev, L, hdr, nullptr, 1, 0, (cudaStream_t)stream);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "snapshot kernel launch failed: %s", cudaGetErrorString(e));
  return BD_OK;
}

int bd_load_snapshot(bd_handle* h, const void* snap_dev, const uint8_t* env_mask_dev, void* stream) {
  int rc = snap_precheck(h, snap_dev, stream, "bd_load_snapshot");
  if (rc) return rc;
  const bool full = env_mask_dev == nullptr;
  if (full && h->graph_mode)
    return fail(BD_EINVAL, "bd_load_snapshot: a full restore is not available after a step was captured into a CUDA graph "
                           "(captured launches carry the Philox offset); restore with an env mask instead");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  bd::SnapHeader hdr;
  BD_CUDA(cudaMemcpyAsync(&hdr, snap_dev, sizeof(hdr), cudaMemcpyDeviceToHost, st));
  BD_CUDA(cudaStreamSynchronize(st));
  const bd_config& c = h->cfg;
  if (hdr.magic != bd::kSnapMagic) return fail(BD_EINVAL, "bd_load_snapshot: not a snapshot (bad magic 0x%08x)", hdr.magic);
  if (hdr.version != bd::kSnapVersion)
    return fail(BD_EINVAL, "bd_load_snapshot: snapshot format version %u, this library reads version %u", hdr.version,
                bd::kSnapVersion);
  if (hdr.precision != BD_F32 && hdr.precision != BD_F64) return fail(BD_EINVAL, "bd_load_snapshot: corrupt header");
  if (hdr.n_envs != c.n_envs || hdr.n_drones != c.n_drones)
    return fail(BD_EINVAL, "bd_load_snapshot: the snapshot holds %d envs x %d drones, the handle %d x %d", hdr.n_envs,
                hdr.n_drones, c.n_envs, c.n_drones);
  if (hdr.task != c.task) return fail(BD_EINVAL, "bd_load_snapshot: the snapshot is of task %d, the handle of task %d", hdr.task, c.task);
  if (hdr.act_type != c.act_type)
    return fail(BD_EINVAL, "bd_load_snapshot: the snapshot has act_type %d, the handle %d", hdr.act_type, c.act_type);
  if (hdr.precision != c.precision)
    return fail(BD_EINVAL, "bd_load_snapshot: the snapshot has precision %s, the handle %s", hdr.precision ? "fp64" : "fp32",
                c.precision ? "fp64" : "fp32");
  if (hdr.pyb_freq != c.pyb_freq || hdr.ctrl_freq != c.ctrl_freq)
    return fail(BD_EINVAL, "bd_load_snapshot: the snapshot has pyb_freq %d / ctrl_freq %d, the handle %d / %d", hdr.pyb_freq,
                hdr.ctrl_freq, c.pyb_freq, c.ctrl_freq);
  if (hdr.fingerprint != snap_fingerprint(c))
    return fail(BD_EINVAL, "bd_load_snapshot: the snapshot was taken with a different configuration (drone model, physics, "
                           "integrator, airframe, controller or spiral constants, or episode length)");
  if (hdr.act_dim != h->A || hdr.buf_slots != h->B) return fail(BD_EINVAL, "bd_load_snapshot: corrupt header");
  if (hdr.flags & ~(uint32_t)(BD_SNAP_ANGV | BD_SNAP_CTRL | BD_SNAP_EPISODES))
    return fail(BD_EINVAL, "bd_load_snapshot: unknown plane flags 0x%x", hdr.flags);
  const int need = snap_flags(h);
  if ((need & ~(int)hdr.flags) != 0)
    return fail(BD_EINVAL, "bd_load_snapshot: the handle needs planes the snapshot lacks (%s%s%s)",
                (need & ~hdr.flags & BD_SNAP_ANGV) ? "world angular velocity, keep_ang_vel " : "",
                (need & ~hdr.flags & BD_SNAP_CTRL) ? "controller memory " : "",
                (need & ~hdr.flags & BD_SNAP_EPISODES) ? "episode returns, track_episodes" : "");
  const bd::SnapLayout L = handle_layout(h, (int)hdr.flags);
  if (hdr.bytes != L.bytes)
    return fail(BD_EINVAL, "bd_load_snapshot: the header says %lld bytes, its layout %lld (truncated or corrupt)",
                (long long)hdr.bytes, (long long)L.bytes);
  if (full) {   // exactly what bd_set_rng_state does
    h->cfg.seed = hdr.rng[0];
    h->philox_base = (uint32_t)hdr.rng[1] - (uint32_t)h->total_steps;
    h->reset_epoch = (int)hdr.rng[2];
    refresh_params(h);
  }
  cudaError_t e = bd::launch_snapshot(h->cfg.precision, params_ptr(h), const_cast<void*>(snap_dev), L, hdr, env_mask_dev, 0,
                                      full ? 1 : 0, st);
  h->launches++;
  if (e != cudaSuccess) return fail(BD_ECUDA, "snapshot kernel launch failed: %s", cudaGetErrorString(e));
  h->restored = true;   // the next step launch must not read ring planes before griddepcontrol.wait
  return BD_OK;
}

int bd_obs_dim(const bd_handle* h) { return h ? h->D : BD_EINVAL; }
int bd_act_dim(const bd_handle* h) { return h ? h->A : BD_EINVAL; }
int bd_action_buffer_size(const bd_handle* h) { return h ? h->B : BD_EINVAL; }
int bd_substeps(const bd_handle* h) { return h ? h->S : BD_EINVAL; }
int64_t bd_launch_count(const bd_handle* h) { return h ? h->launches : 0; }

}  // extern "C"
