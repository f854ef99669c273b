// s2d_api.cu - the C ABI of libsoccer2d.so (include/soccer2d.h) and the kernel launches behind it.
//
// Host side of the drop-in boundary for Soccer2DEnv.step/reset (soccer_2d_env.py:179-269): a handle holds
// parameters and launch geometry only; every device buffer belongs to the caller.  Nothing here runs the
// simulation on the CPU: without a CUDA device s2d_create fails with S2D_ERR_NO_DEVICE.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "s2d_fullgame.cuh"
#include "s2d_rollout.cuh"
#include "s2d_rollout_tc5.cuh"

using namespace s2d;

struct S2DSim {
  S2DConfig cfg;
  S2DBuffers buf;
  KernelParams kp;
  float4* d_table = nullptr;
  float* d_types = nullptr;  // heterogeneous players: [S2D_MAX_PLAYER_TYPES][PT_ROW]
  uint8_t* d_type_of = nullptr;  // per-match assignment: [np][Nr]
  bool hetero = false;
  bool default_sp = false;  // cfg.sp == rcssserver defaults: use the constant-folded kernels
  bool bound = false;
  // host-buffer pipeline (s2d_bind_pipeline_slot / s2d_submit_host / s2d_wait_host): up to kSlots slots of actions +
  // outputs; slot 0 = the buffers of s2d_bind
  bool piped = false;
  S2DBuffers pbuf[S2D_MAX_PIPELINE_SLOTS];
  KernelParams pkp[S2D_MAX_PIPELINE_SLOTS];
  bool slot_bound[S2D_MAX_PIPELINE_SLOTS] = {false, false, false, false};
  cudaStream_t st_in = nullptr, st_compute = nullptr, st_out = nullptr;
  cudaEvent_t ev_in[S2D_MAX_PIPELINE_SLOTS] = {}, ev_kernel[S2D_MAX_PIPELINE_SLOTS] = {}, ev_out[S2D_MAX_PIPELINE_SLOTS] = {};
  cudaEvent_t ev_user = nullptr;  // end of the last caller-stream operation that touched the shared state
  bool used[S2D_MAX_PIPELINE_SLOTS] = {false, false, false, false};
  bool user_pending = false;
  int fg_lanes_per_match = 0;  // FULLGAME: 0 = chosen by the shard size (launch_step); S2D_FG_LANES overrides (tuning)
  int last_d2h_copies = 0;  // device-to-host copies the last host-buffer step issued (1 = the packed block)
  int grid = 0;
  uint64_t env_steps = 0;
  char err[512];
};

static thread_local char g_create_err[512] = "";

static int fail(S2DSim* h, int code, const char* fmt, ...) {
  char* dst = h ? h->err : g_create_err;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define S2D_CUDA(h, expr)                                                                              \
  do {                                                                                                 \
    cudaError_t err__ = (expr);                                                                        \
    if (err__ != cudaSuccess)                                                                          \
      return fail(h, S2D_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(err__), __FILE__, \
                  __LINE__);                                                                           \
  } while (0)

// RAII: run on the handle's device without changing the caller's current device
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

namespace {
__global__ void fill_sincos_memo(float2* memo) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < kSinCosMemoSize) sincos_deg(static_cast<float>(j - kSinCosMemoHalf), memo[j].x, memo[j].y);
}
}  // namespace

extern "C" {

int s2d_abi_version(void) { return S2D_ABI_VERSION; }

const char* s2d_error_string(int code) {
  switch (code) {
    case S2D_OK: return "ok";
    case S2D_ERR_INVALID: return "invalid argument or configuration";
    case S2D_ERR_UNBOUND: return "buffers not bound (s2d_bind) or a required buffer is NULL";
    case S2D_ERR_CUDA: return "CUDA runtime error";
    case S2D_ERR_NO_DEVICE: return "no usable CUDA device (there is no CPU fallback)";
    default: return "unknown error code";
  }
}

const char* s2d_last_error(S2DHandle h) { return h ? h->err : g_create_err; }

int s2d_default_server_param(S2DServerParam* sp) {
  if (!sp) return S2D_ERR_INVALID;
  default_server_param(*sp);  // rcssserver defaults (s2d_params.h)
  return S2D_OK;
}
int s2d_default_config(S2DConfig* c, int scenario) {
  if (!c) return S2D_ERR_INVALID;
  memset(c, 0, sizeof(*c));
  c->struct_size = static_cast<int32_t>(sizeof(S2DConfig));
  c->scenario = scenario;
  c->num_envs = 1;
  c->action_mode = S2D_ACT_CONTINUOUS;  // reach_ball_env.py:34 use_continuous_action=True
  c->action_space_size = 16;            // :35
  c->max_steps = 200;                   // :33
  c->auto_reset = 1;
  c->change_ball_position = 1;          // :26
  c->change_ball_velocity = 0;          // :27
  c->players_per_side = scenario == S2D_SCENARIO_FULLGAME ? 11 : 1;
  c->half_time_cycles = 3000;
  if (scenario == S2D_SCENARIO_SHOOT) {  // Discrete(24) = 16 dashes + 8 kicks
    c->action_mode = S2D_ACT_DISCRETE;
    c->action_space_size = 24;
    c->kick_actions = 8;
  }
  if (scenario == S2D_SCENARIO_FULLGAME) c->action_mode = S2D_ACT_COMMAND;
  c->min_distance_to_ball = 5.0f;       // :32
  c->goto_dist_thr = 0.5f;
  return s2d_default_server_param(&c->sp);
}

static bool config_ok(const S2DConfig* c, char* why, size_t n) {
  if (!c) { snprintf(why, n, "config is NULL"); return false; }
  if (c->struct_size != static_cast<int32_t>(sizeof(S2DConfig))) {
    snprintf(why, n, "S2DConfig.struct_size %d != %zu (ABI mismatch)", c->struct_size, sizeof(S2DConfig));
    return false;
  }
  if (c->num_envs < 1) { snprintf(why, n, "num_envs must be >= 1"); return false; }
  if (c->scenario < S2D_SCENARIO_REACHBALL || c->scenario > S2D_SCENARIO_FULLGAME) {
    snprintf(why, n, "scenario %d does not exist", c->scenario);
    return false;
  }
  if (c->scenario == S2D_SCENARIO_FULLGAME) {
    if (c->players_per_side < 1 || c->players_per_side > 11) { snprintf(why, n, "players_per_side must be in 1..11"); return false; }
    if (c->half_time_cycles < 1) { snprintf(why, n, "half_time_cycles must be >= 1"); return false; }
  }
  const bool mode_ok = c->scenario == S2D_SCENARIO_FULLGAME
                           ? c->action_mode == S2D_ACT_COMMAND
                           : c->scenario == S2D_SCENARIO_SHOOT
                                 ? (c->action_mode == S2D_ACT_DISCRETE || c->action_mode == S2D_ACT_COMMAND)
                                 : (c->action_mode >= S2D_ACT_DISCRETE && c->action_mode <= S2D_ACT_COMMAND);
  if (!mode_ok) {
    snprintf(why, n, "action_mode %d is not valid for scenario %d", c->action_mode, c->scenario);
    return false;
  }
  if (c->action_mode == S2D_ACT_DISCRETE && (c->action_space_size < 1 || c->action_space_size > 256)) {
    snprintf(why, n, "action_space_size must be in 1..256");
    return false;
  }
  if (c->scenario == S2D_SCENARIO_SHOOT && c->action_mode == S2D_ACT_DISCRETE &&
      (c->kick_actions < 1 || c->kick_actions >= c->action_space_size)) {
    snprintf(why, n, "SHOOT Discrete(n) needs 1 <= kick_actions < action_space_size");
    return false;
  }
  if (c->max_steps < 0) { snprintf(why, n, "max_steps must be >= 0"); return false; }
  if (c->collision_model != S2D_COLLISION_MIDPOINT && c->collision_model != S2D_COLLISION_BACKTRACE) {
    snprintf(why, n, "collision_model %d does not exist", c->collision_model);
    return false;
  }
  return true;
}

static size_t action_elem_bytes(const S2DConfig* c) {
  switch (c->action_mode) {
    case S2D_ACT_DISCRETE: return 1;
    case S2D_ACT_CONTINUOUS: return 4;
    case S2D_ACT_TURNING: return 16;
    default: return 16 * static_cast<size_t>(s2d_num_players(c));
  }
}

size_t s2d_state_bytes(const S2DConfig* c) {
  if (!c) return 0;
  if (c->scenario == S2D_SCENARIO_FULLGAME) return FgLayout{c->num_envs, 2 * c->players_per_side}.bytes();
  return static_cast<size_t>(c->num_envs) * kStateBytesPerEnv;
}
size_t s2d_action_bytes(const S2DConfig* c) { return c ? static_cast<size_t>(c->num_envs) * action_elem_bytes(c) : 0; }
size_t s2d_stats_bytes(const S2DConfig* c) { return c ? sizeof(unsigned long long) * kStatSlots * kStatWords : 0; }
int s2d_obs_dim(const S2DConfig* c) { return !c ? 0 : c->scenario == S2D_SCENARIO_FULLGAME ? kFgObsDim : kObsDim; }
int s2d_num_players(const S2DConfig* c) {
  if (!c) return 0;
  return c->scenario == S2D_SCENARIO_FULLGAME ? 2 * c->players_per_side : 1;
}

int s2d_create(const S2DConfig* cfg, S2DHandle* out) {
  if (!out) return fail(nullptr, S2D_ERR_INVALID, "out handle pointer is NULL");
  *out = nullptr;
  char why[256];
  if (!config_ok(cfg, why, sizeof(why))) return fail(nullptr, S2D_ERR_INVALID, "%s", why);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    cudaGetLastError();
    return fail(nullptr, S2D_ERR_NO_DEVICE, "no CUDA device is visible; libsoccer2d has no CPU path");
  }
  if (cfg->device < 0 || cfg->device >= ndev)
    return fail(nullptr, S2D_ERR_INVALID, "device %d out of range (0..%d)", cfg->device, ndev - 1);
  S2DSim* h = new (std::nothrow) S2DSim();
  if (!h) return fail(nullptr, S2D_ERR_INVALID, "out of host memory");
  h->cfg = *cfg;
  h->err[0] = 0;
  memset(&h->buf, 0, sizeof(h->buf));
  DeviceGuard guard(cfg->device);

  KernelParams& kp = h->kp;
  float4 table[256];
  make_kernel_params(*cfg, kp, table);
  h->default_sp = is_default_server_param(cfg->sp) && cfg->collision_model == S2D_COLLISION_MIDPOINT;
  // one allocation: the action table, then the memo of sincos_deg over whole degrees (written by sincos_deg itself)
  cudaError_t e = cudaMalloc(&h->d_table, sizeof(table) + sizeof(float2) * kSinCosMemoSize);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_table, table, sizeof(table), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    float2* memo = reinterpret_cast<float2*>(h->d_table + 256);
    fill_sincos_memo<<<(kSinCosMemoSize + 255) / 256, 256>>>(memo);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    kp.sincos_memo = memo;
  }
  if (e != cudaSuccess) {
    fail(nullptr, S2D_ERR_CUDA, "allocating the action table failed: %s", cudaGetErrorString(e));
    if (h->d_table) cudaFree(h->d_table);
    delete h;
    return S2D_ERR_CUDA;
  }
  kp.action_table = h->d_table;
  if (const char* v = getenv("S2D_FG_LANES")) {  // tuning aid: lanes per match of the 11 v 11 kernel (1, 2)
    const int l = atoi(v);
    if (l == 1 || l == 2) h->fg_lanes_per_match = l;
  }
  h->grid = cfg->scenario == S2D_SCENARIO_FULLGAME ? static_cast<int>((cfg->num_envs + kFgBlock - 1) / kFgBlock)  // thread = match
                                                   : static_cast<int>((cfg->num_envs + kBlock - 1) / kBlock);
  *out = h;
  return S2D_OK;
}

int s2d_destroy(S2DHandle h) {
  if (!h) return S2D_OK;
  {
    DeviceGuard guard(h->cfg.device);
    if (h->d_table) cudaFree(h->d_table);
    if (h->d_types) cudaFree(h->d_types);
    if (h->d_type_of) cudaFree(h->d_type_of);
    if (h->st_in) {
      cudaStreamSynchronize(h->st_in);
      cudaStreamSynchronize(h->st_compute);
      cudaStreamSynchronize(h->st_out);
      for (int k = 0; k < S2D_MAX_PIPELINE_SLOTS; ++k) {
        if (h->ev_in[k]) cudaEventDestroy(h->ev_in[k]);
        if (h->ev_kernel[k]) cudaEventDestroy(h->ev_kernel[k]);
        if (h->ev_out[k]) cudaEventDestroy(h->ev_out[k]);
      }
      if (h->ev_user) cudaEventDestroy(h->ev_user);
      cudaStreamDestroy(h->st_in);
      cudaStreamDestroy(h->st_compute);
      cudaStreamDestroy(h->st_out);
    }
  }
  delete h;
  return S2D_OK;
}

// ---- ordering between the caller's stream and the pipeline's internal streams -------------------------------
// The state and the statistics are shared by every slot and by the caller-stream entry points; slot 0's actions and
// outputs are the buffers of s2d_bind.  before_user_op makes the caller's stream wait (on the device, the host does not
// block) for every kernel the pipeline has submitted and for the copies that still read slot 0's outputs;
// after_user_op records where that caller-stream work ends so that the next s2d_submit_host waits for it.
static int before_user_op(S2DSim* h, cudaStream_t s) {
  if (!h->piped) return S2D_OK;
  for (int k = 0; k < S2D_MAX_PIPELINE_SLOTS; ++k)
    if (h->used[k]) S2D_CUDA(h, cudaStreamWaitEvent(s, h->ev_kernel[k], 0));
  if (h->used[0]) S2D_CUDA(h, cudaStreamWaitEvent(s, h->ev_out[0], 0));
  return S2D_OK;
}
static int after_user_op(S2DSim* h, cudaStream_t s) {
  if (!h->piped) return S2D_OK;
  S2D_CUDA(h, cudaEventRecord(h->ev_user, s));
  h->user_pending = true;
  return S2D_OK;
}

static void slot_params(S2DSim* h, int k) {
  KernelParams& kp = h->pkp[k];
  kp = h->kp;  // constants, state, stats, player types
  kp.actions = h->pbuf[k].actions;
  kp.obs = h->pbuf[k].obs;
  kp.reward = h->pbuf[k].reward;
  kp.done = h->pbuf[k].done;
  kp.result = h->pbuf[k].result;
  kp.terminal_obs = h->pbuf[k].terminal_obs;
}

int s2d_bind(S2DHandle h, const S2DBuffers* b) {
  if (!h) return S2D_ERR_INVALID;
  if (!b) return fail(h, S2D_ERR_INVALID, "buffers pointer is NULL");
  if (!b->state || !b->actions || !b->obs || !b->reward || !b->done || !b->result || !b->stats)
    return fail(h, S2D_ERR_UNBOUND, "state, actions, obs, reward, done, result and stats are required");
  if ((reinterpret_cast<uintptr_t>(b->state) & 255) || (reinterpret_cast<uintptr_t>(b->actions) & 15) ||
      (reinterpret_cast<uintptr_t>(b->obs) & 15) || (b->terminal_obs && (reinterpret_cast<uintptr_t>(b->terminal_obs) & 15)))
    return fail(h, S2D_ERR_INVALID, "state must be 256-byte aligned; actions / obs / terminal_obs 16-byte aligned");
  if (h->cfg.scenario == S2D_SCENARIO_FULLGAME &&
      ((reinterpret_cast<uintptr_t>(b->actions) & 31) || (reinterpret_cast<uintptr_t>(b->obs) & 31) ||
       (b->terminal_obs && (reinterpret_cast<uintptr_t>(b->terminal_obs) & 31))))
    return fail(h, S2D_ERR_INVALID, "FULLGAME: actions / obs / terminal_obs must be 32-byte aligned (256-bit accesses)");
  h->buf = *b;
  h->kp.state = b->state;
  h->kp.actions = b->actions;
  h->kp.obs = b->obs;
  h->kp.reward = b->reward;
  h->kp.done = b->done;
  h->kp.result = b->result;
  h->kp.terminal_obs = b->terminal_obs;
  h->kp.stats = static_cast<unsigned long long*>(b->stats);
  h->bound = true;
  if (h->piped) {  // a re-bind (new action tensor, new state) reaches the pipeline's parameter blocks too
    h->pbuf[0] = h->buf;
    for (int k = 0; k < S2D_MAX_PIPELINE_SLOTS; ++k) {
      if (!h->slot_bound[k]) continue;
      h->pbuf[k].state = b->state;
      h->pbuf[k].stats = b->stats;
      slot_params(h, k);
    }
  }
  return S2D_OK;
}

int s2d_fence(S2DHandle h, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->piped) return S2D_OK;
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  return after_user_op(h, s);
}

int s2d_clear(S2DHandle h, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  S2D_CUDA(h, cudaMemsetAsync(h->buf.state, 0, s2d_state_bytes(&h->cfg), s));
  S2D_CUDA(h, cudaMemsetAsync(h->buf.stats, 0, s2d_stats_bytes(&h->cfg), s));
  h->env_steps = 0;
  return after_user_op(h, s);
}

static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

int s2d_output_layout(const S2DConfig* c, S2DOutputLayout* out) {
  if (!c || !out || c->num_envs < 1) return S2D_ERR_INVALID;
  const size_t n = static_cast<size_t>(c->num_envs), row = static_cast<size_t>(s2d_obs_dim(c)) * sizeof(float);
  out->obs = 0;
  out->reward = align256(n * row);
  out->done = out->reward + align256(n * sizeof(float));
  out->result = out->done + align256(n);
  out->step_bytes = out->result + n;
  out->bytes = out->result + align256(n);
  out->terminal_obs = out->bytes;
  out->bytes_with_terminal_obs = out->bytes + align256(n * row);
  return S2D_OK;
}

int s2d_reset(S2DHandle h, const uint8_t* device_mask_or_null, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  if (h->cfg.scenario == S2D_SCENARIO_FULLGAME) {
    const int np = 2 * h->cfg.players_per_side, ht = h->cfg.half_time_cycles;
    if (h->hetero) fullgame_reset_kernel<true><<<h->grid, kFgBlock, 0, s>>>(h->kp, device_mask_or_null, np, ht);
    else fullgame_reset_kernel<false><<<h->grid, kFgBlock, 0, s>>>(h->kp, device_mask_or_null, np, ht);
  }
  else if (h->cfg.scenario == S2D_SCENARIO_SHOOT) {
    if (h->cfg.noise) reset_kernel<S2D_SCENARIO_SHOOT, true><<<h->grid, kBlock, 0, s>>>(h->kp, device_mask_or_null);
    else reset_kernel<S2D_SCENARIO_SHOOT, false><<<h->grid, kBlock, 0, s>>>(h->kp, device_mask_or_null);
  } else {
    if (h->cfg.noise) reset_kernel<S2D_SCENARIO_REACHBALL, true><<<h->grid, kBlock, 0, s>>>(h->kp, device_mask_or_null);
    else reset_kernel<S2D_SCENARIO_REACHBALL, false><<<h->grid, kBlock, 0, s>>>(h->kp, device_mask_or_null);
  }
  S2D_CUDA(h, cudaGetLastError());
  return after_user_op(h, s);
}

// one launch of the scenario's step kernel with the given parameter block
static cudaError_t launch_step(S2DSim* h, const KernelParams& kp, int k_substeps, cudaStream_t s) {
#define S2D_LAUNCH(SCN, ACT)                                                                   \
  do {                                                                                         \
    if (h->cfg.noise) step_kernel<SCN, ACT, kVarNoisy><<<h->grid, kBlock, 0, s>>>(kp, k_substeps);             \
    else if (h->default_sp) step_kernel<SCN, ACT, kVarDefault><<<h->grid, kBlock, 0, s>>>(kp, k_substeps);  \
    else step_kernel<SCN, ACT, kVarRuntime><<<h->grid, kBlock, 0, s>>>(kp, k_substeps);                     \
  } while (0)
  if (h->cfg.scenario == S2D_SCENARIO_FULLGAME) {
    const int np = 2 * h->cfg.players_per_side, ht = h->cfg.half_time_cycles;
    // One thread per match fills the GPU from about 10^5 matches on (148 SMs x 20 warps x 32).  A small shard is bound
    // by the latency of its slowest warp; two lanes sharing a match shorten the player loop (measured on 2^18 matches in
    // total: 45 -> 41 us per cycle at 32 K matches per GPU; no gain from 64 K on, none from four lanes: profiles/README.md).
    const int64_t nr = static_cast<int64_t>(FgLayout{h->cfg.num_envs, np}.nr());
    const int lpm = h->fg_lanes_per_match > 0 ? h->fg_lanes_per_match : nr <= 49152 ? 2 : 1;
    const int g1 = static_cast<int>(nr / kFgBlock);
// (a non-zero scripted-player mask selects the same kernel with the script compiled in: s2d_scripted.cu)
#define S2D_FG_GO(VAR, NP, LPM, GRID)                                                                \
  do {                                                                                               \
    if (script) {                                                                                    \
      const cudaError_t e = launch_fullgame_scripted(VAR, NP, LPM, GRID, kp, k_substeps, np, ht, s); \
      if (e != cudaSuccess) return e;                                                                \
    }                                                                                                \
    else fullgame_step_kernel<VAR, NP, LPM><<<GRID, kFgBlock, 0, s>>>(kp, k_substeps, np, ht);       \
  } while (0)
#define S2D_FG(VAR)                                 \
  do {                                              \
    if (lpm == 2) S2D_FG_GO(VAR, 22, 2, g1 * 2);    \
    else S2D_FG_GO(VAR, 22, 1, g1);                 \
  } while (0)
    const bool script = kp.scripted_mask != 0u;
    if (h->hetero && h->cfg.noise) S2D_FG_GO(kVarHeteroNoisy, 0, 1, g1);
    else if (h->hetero && np == 22) S2D_FG_GO(kVarHetero, 22, 1, g1);
    else if (h->hetero) S2D_FG_GO(kVarHetero, 0, 1, g1);
    else if (h->cfg.noise) S2D_FG_GO(kVarNoisy, 0, 1, g1);
    else if (!h->default_sp && np == 22) S2D_FG(kVarRuntime);
    else if (!h->default_sp) S2D_FG_GO(kVarRuntime, 0, 1, g1);
    else if (np == 22) S2D_FG(kVarDefault);
    else S2D_FG_GO(kVarDefault, 0, 1, g1);
#undef S2D_FG
#undef S2D_FG_GO
  } else if (h->cfg.scenario == S2D_SCENARIO_SHOOT) {
    if (h->cfg.action_mode == S2D_ACT_DISCRETE) S2D_LAUNCH(S2D_SCENARIO_SHOOT, S2D_ACT_DISCRETE);
    else S2D_LAUNCH(S2D_SCENARIO_SHOOT, S2D_ACT_COMMAND);
  } else {
    switch (h->cfg.action_mode) {
      case S2D_ACT_DISCRETE: S2D_LAUNCH(S2D_SCENARIO_REACHBALL, S2D_ACT_DISCRETE); break;
      case S2D_ACT_CONTINUOUS: S2D_LAUNCH(S2D_SCENARIO_REACHBALL, S2D_ACT_CONTINUOUS); break;
      case S2D_ACT_TURNING: S2D_LAUNCH(S2D_SCENARIO_REACHBALL, S2D_ACT_TURNING); break;
      default: S2D_LAUNCH(S2D_SCENARIO_REACHBALL, S2D_ACT_COMMAND); break;
    }
  }
#undef S2D_LAUNCH
  return cudaGetLastError();
}

int s2d_step(S2DHandle h, int k_substeps, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  if (k_substeps < 1 || k_substeps > kMaxSubsteps)
    return fail(h, S2D_ERR_INVALID, "k_substeps must be in 1..%d", kMaxSubsteps);
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  S2D_CUDA(h, launch_step(h, h->kp, k_substeps, s));
  h->env_steps += static_cast<uint64_t>(h->cfg.num_envs) * static_cast<uint64_t>(k_substeps);
  return after_user_op(h, s);
}

// Device-to-host copies of one step's outputs.  When the host pointers mirror the device layout (one block carved as
// s2d_output_layout says - or any other common layout with obs first and result last) the outputs leave in ONE copy.
static int copy_outputs(S2DSim* h, const S2DBuffers& b, float* h_obs, float* h_reward, uint8_t* h_done, uint8_t* h_result,
                        cudaStream_t s) {
  const size_t n = static_cast<size_t>(h->cfg.num_envs);
  const size_t obs_bytes = n * s2d_obs_dim(&h->cfg) * sizeof(float);
  if (h_obs && h_reward && h_done && h_result) {
    const char* d0 = reinterpret_cast<const char*>(b.obs);
    const char* h0 = reinterpret_cast<const char*>(h_obs);
    const ptrdiff_t dr = reinterpret_cast<const char*>(b.reward) - d0, dd = reinterpret_cast<const char*>(b.done) - d0,
                    ds = reinterpret_cast<const char*>(b.result) - d0;
    const bool mirrored = reinterpret_cast<const char*>(h_reward) - h0 == dr && reinterpret_cast<const char*>(h_done) - h0 == dd &&
                          reinterpret_cast<const char*>(h_result) - h0 == ds;
    const bool ordered = dr >= static_cast<ptrdiff_t>(obs_bytes) && dd >= dr + static_cast<ptrdiff_t>(n * sizeof(float)) &&
                         ds >= dd + static_cast<ptrdiff_t>(n);
    // one block: at most 3 x 255 bytes of padding travel along
    if (mirrored && ordered && static_cast<size_t>(ds) + n <= obs_bytes + n * 6 + 3 * 256) {
      S2D_CUDA(h, cudaMemcpyAsync(h_obs, b.obs, static_cast<size_t>(ds) + n, cudaMemcpyDeviceToHost, s));
      h->last_d2h_copies = 1;
      return S2D_OK;
    }
  }
  if (h_obs) S2D_CUDA(h, cudaMemcpyAsync(h_obs, b.obs, obs_bytes, cudaMemcpyDeviceToHost, s));
  if (h_reward) S2D_CUDA(h, cudaMemcpyAsync(h_reward, b.reward, n * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (h_done) S2D_CUDA(h, cudaMemcpyAsync(h_done, b.done, n, cudaMemcpyDeviceToHost, s));
  if (h_result) S2D_CUDA(h, cudaMemcpyAsync(h_result, b.result, n, cudaMemcpyDeviceToHost, s));
  h->last_d2h_copies = (h_obs != nullptr) + (h_reward != nullptr) + (h_done != nullptr) + (h_result != nullptr);
  return S2D_OK;
}

// ---- pipelined host-buffer stepping ----------------------------------------------------------------------
// Slot s owns a device actions buffer and device output buffers (slot 0 = the buffers of s2d_bind, the others are
// given here).  s2d_submit_host enqueues, on three internal streams, H2D(actions) -> step kernel -> D2H(outputs) for
// one slot; consecutive submissions rotate the slots, so the copies of step i overlap the kernel and the copies of
// the following steps.  The step kernels themselves stay in submission order (they share the state).

int s2d_bind_pipeline_slot(S2DHandle h, int slot, const S2DBuffers* second) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind must come first");
  if (slot < 1 || slot >= S2D_MAX_PIPELINE_SLOTS) return fail(h, S2D_ERR_INVALID, "slot must be in 1..%d (slot 0 = the buffers of s2d_bind)", S2D_MAX_PIPELINE_SLOTS - 1);
  if (!second || !second->actions || !second->obs || !second->reward || !second->done || !second->result)
    return fail(h, S2D_ERR_UNBOUND, "a pipeline slot needs actions, obs, reward, done and result buffers");
  if ((reinterpret_cast<uintptr_t>(second->actions) & 15) || (reinterpret_cast<uintptr_t>(second->obs) & 15) ||
      (second->terminal_obs && (reinterpret_cast<uintptr_t>(second->terminal_obs) & 15)))
    return fail(h, S2D_ERR_INVALID, "actions / obs / terminal_obs must be 16-byte aligned");
  if (h->cfg.scenario == S2D_SCENARIO_FULLGAME &&
      ((reinterpret_cast<uintptr_t>(second->actions) & 31) || (reinterpret_cast<uintptr_t>(second->obs) & 31) ||
       (second->terminal_obs && (reinterpret_cast<uintptr_t>(second->terminal_obs) & 31))))
    return fail(h, S2D_ERR_INVALID, "FULLGAME: actions / obs / terminal_obs must be 32-byte aligned (256-bit accesses)");
  DeviceGuard guard(h->cfg.device);
  if (!h->st_in) {
    S2D_CUDA(h, cudaStreamCreateWithFlags(&h->st_in, cudaStreamNonBlocking));
    S2D_CUDA(h, cudaStreamCreateWithFlags(&h->st_compute, cudaStreamNonBlocking));
    S2D_CUDA(h, cudaStreamCreateWithFlags(&h->st_out, cudaStreamNonBlocking));
    for (int k = 0; k < S2D_MAX_PIPELINE_SLOTS; ++k) {
      S2D_CUDA(h, cudaEventCreateWithFlags(&h->ev_in[k], cudaEventDisableTiming));
      S2D_CUDA(h, cudaEventCreateWithFlags(&h->ev_kernel[k], cudaEventDisableTiming));
      S2D_CUDA(h, cudaEventCreateWithFlags(&h->ev_out[k], cudaEventDisableTiming));
    }
    S2D_CUDA(h, cudaEventCreateWithFlags(&h->ev_user, cudaEventDisableTiming));
  }
  if (h->used[slot]) S2D_CUDA(h, cudaEventSynchronize(h->ev_out[slot]));  // re-binding a slot that is in flight
  h->pbuf[0] = h->buf;
  h->slot_bound[0] = true;
  slot_params(h, 0);
  h->pbuf[slot] = h->buf;  // state and stats are shared
  h->pbuf[slot].actions = second->actions;
  h->pbuf[slot].obs = second->obs;
  h->pbuf[slot].reward = second->reward;
  h->pbuf[slot].done = second->done;
  h->pbuf[slot].result = second->result;
  h->pbuf[slot].terminal_obs = second->terminal_obs;
  h->slot_bound[slot] = true;
  h->used[slot] = false;
  slot_params(h, slot);
  h->piped = true;
  return S2D_OK;
}

int s2d_bind_pipeline(S2DHandle h, const S2DBuffers* second) { return s2d_bind_pipeline_slot(h, 1, second); }

int s2d_submit_host(S2DHandle h, int k_substeps, int slot, const void* h_actions, float* h_obs, float* h_reward,
                    uint8_t* h_done, uint8_t* h_result) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->piped) return fail(h, S2D_ERR_UNBOUND, "s2d_bind_pipeline has not been called");
  if (slot < 0 || slot >= S2D_MAX_PIPELINE_SLOTS || !h->slot_bound[slot]) return fail(h, S2D_ERR_INVALID, "slot %d is not bound", slot);
  if (!h_actions) return fail(h, S2D_ERR_INVALID, "h_actions is NULL");
  if (k_substeps < 1 || k_substeps > kMaxSubsteps)
    return fail(h, S2D_ERR_INVALID, "k_substeps must be in 1..%d", kMaxSubsteps);
  DeviceGuard guard(h->cfg.device);
  const S2DBuffers& b = h->pbuf[slot];
  if (h->user_pending) {  // caller-stream work on the shared state / slot 0's buffers comes first
    S2D_CUDA(h, cudaStreamWaitEvent(h->st_in, h->ev_user, 0));
    S2D_CUDA(h, cudaStreamWaitEvent(h->st_compute, h->ev_user, 0));
    h->user_pending = false;
  }
  // actions[slot] may be overwritten once the kernel that read them is done; outputs[slot] once their D2H is done
  if (h->used[slot]) S2D_CUDA(h, cudaStreamWaitEvent(h->st_in, h->ev_kernel[slot], 0));
  S2D_CUDA(h, cudaMemcpyAsync(b.actions, h_actions, s2d_action_bytes(&h->cfg) * k_substeps, cudaMemcpyHostToDevice, h->st_in));
  S2D_CUDA(h, cudaEventRecord(h->ev_in[slot], h->st_in));
  S2D_CUDA(h, cudaStreamWaitEvent(h->st_compute, h->ev_in[slot], 0));
  if (h->used[slot]) S2D_CUDA(h, cudaStreamWaitEvent(h->st_compute, h->ev_out[slot], 0));
  S2D_CUDA(h, launch_step(h, h->pkp[slot], k_substeps, h->st_compute));
  S2D_CUDA(h, cudaEventRecord(h->ev_kernel[slot], h->st_compute));
  S2D_CUDA(h, cudaStreamWaitEvent(h->st_out, h->ev_kernel[slot], 0));
  if (int rc = copy_outputs(h, b, h_obs, h_reward, h_done, h_result, h->st_out)) return rc;
  S2D_CUDA(h, cudaEventRecord(h->ev_out[slot], h->st_out));
  h->used[slot] = true;
  h->env_steps += static_cast<uint64_t>(h->cfg.num_envs) * static_cast<uint64_t>(k_substeps);
  return S2D_OK;
}

int s2d_wait_host(S2DHandle h, int slot) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->piped) return fail(h, S2D_ERR_UNBOUND, "s2d_bind_pipeline has not been called");
  if (slot < 0 || slot >= S2D_MAX_PIPELINE_SLOTS || !h->slot_bound[slot]) return fail(h, S2D_ERR_INVALID, "slot %d is not bound", slot);
  if (!h->used[slot]) return S2D_OK;
  DeviceGuard guard(h->cfg.device);
  S2D_CUDA(h, cudaEventSynchronize(h->ev_out[slot]));
  return S2D_OK;
}

int s2d_step_host(S2DHandle h, int k_substeps, const void* h_actions, float* h_obs, float* h_reward, uint8_t* h_done,
                  uint8_t* h_result, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  if (!h_actions) return fail(h, S2D_ERR_INVALID, "h_actions is NULL");
  if (k_substeps < 1 || k_substeps > kMaxSubsteps)
    return fail(h, S2D_ERR_INVALID, "k_substeps must be in 1..%d", kMaxSubsteps);
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  S2D_CUDA(h, cudaMemcpyAsync(h->buf.actions, h_actions, s2d_action_bytes(&h->cfg) * k_substeps, cudaMemcpyHostToDevice, s));
  const int rc = s2d_step(h, k_substeps, stream);
  if (rc != S2D_OK) return rc;
  if (int rc2 = copy_outputs(h, h->buf, h_obs, h_reward, h_done, h_result, s)) return rc2;
  return after_user_op(h, s);
}

int s2d_stats(S2DHandle h, S2DStats* out, void* stream) {
  if (!h || !out) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  std::vector<unsigned long long> host(kStatSlots * kStatWords);
  S2D_CUDA(h, cudaMemcpyAsync(host.data(), h->buf.stats, host.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
  S2D_CUDA(h, cudaStreamSynchronize(s));
  memset(out, 0, sizeof(*out));
  for (int k = 0; k < kStatSlots; ++k) {
    const unsigned long long* slot = host.data() + static_cast<size_t>(k) * kStatWords;
    out->episodes += slot[ST_EPISODES];
    out->goals += slot[ST_GOALS];
    out->outs += slot[ST_OUTS];
    out->timeouts += slot[ST_TIMEOUTS];
    out->episode_steps += slot[ST_EP_STEPS];
    double r;
    memcpy(&r, slot + ST_RETURN, sizeof(r));
    out->return_sum += r;
  }
  out->env_steps = h->env_steps;
  return S2D_OK;
}

int s2d_env_steps(S2DHandle h, uint64_t* out) {
  if (!h || !out) return S2D_ERR_INVALID;
  *out = h->env_steps;
  return S2D_OK;
}

int s2d_stats_reset(S2DHandle h, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  DeviceGuard guard(h->cfg.device);
  if (int rc = before_user_op(h, static_cast<cudaStream_t>(stream))) return rc;
  S2D_CUDA(h, cudaMemsetAsync(h->buf.stats, 0, s2d_stats_bytes(&h->cfg), static_cast<cudaStream_t>(stream)));
  h->env_steps = 0;
  return after_user_op(h, static_cast<cudaStream_t>(stream));
}

int s2d_export_env(S2DHandle h, int64_t i, S2DEnvSnapshot* out, void* stream) {
  if (!h || !out) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  if (i < 0 || i >= h->cfg.num_envs) return fail(h, S2D_ERR_INVALID, "env index %lld out of range", static_cast<long long>(i));
  DeviceGuard guard(h->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  const char* base = static_cast<const char*>(h->buf.state);
  const size_t n = static_cast<size_t>(h->cfg.num_envs);
  if (h->cfg.scenario == S2D_SCENARIO_FULLGAME) {
    const int np = 2 * h->cfg.players_per_side, pps = h->cfg.players_per_side;
    const FgLayout L{h->cfg.num_envs, np};
    float4 pa[kFgMaxPlayers], pb[kFgMaxPlayers], ball, ef;
    float pc[kFgMaxPlayers];
    uint4 ei, ej;
    // match-minor planes: player j of match i sits at row j, column i - one strided copy per plane
    const size_t col = static_cast<size_t>(i);
    S2D_CUDA(h, cudaMemcpy2DAsync(pa, 16, base + L.pa() + col * 16, L.nr() * 16, 16, np, cudaMemcpyDeviceToHost, s));
    S2D_CUDA(h, cudaMemcpy2DAsync(pb, 16, base + L.pb() + col * 16, L.nr() * 16, 16, np, cudaMemcpyDeviceToHost, s));
    S2D_CUDA(h, cudaMemcpy2DAsync(pc, 4, base + L.pc() + col * 4, L.nr() * 4, 4, np, cudaMemcpyDeviceToHost, s));
    S2D_CUDA(h, cudaMemcpyAsync(&ball, base + L.eb() + static_cast<size_t>(i) * 16, 16, cudaMemcpyDeviceToHost, s));
    S2D_CUDA(h, cudaMemcpyAsync(&ef, base + L.ef() + static_cast<size_t>(i) * 16, 16, cudaMemcpyDeviceToHost, s));
    S2D_CUDA(h, cudaMemcpyAsync(&ei, base + L.ei() + static_cast<size_t>(i) * 16, 16, cudaMemcpyDeviceToHost, s));
    S2D_CUDA(h, cudaMemcpyAsync(&ej, base + L.ej() + static_cast<size_t>(i) * 16, 16, cudaMemcpyDeviceToHost, s));
    S2D_CUDA(h, cudaStreamSynchronize(s));
    memset(out, 0, sizeof(*out));
    out->step_number = static_cast<int32_t>(ei.x);
    out->cycle = static_cast<int32_t>(ei.y);
    out->episode = static_cast<int32_t>(ei.z);
    out->game_mode_type = static_cast<int32_t>(ei.w & 0xff);
    out->game_mode_side = static_cast<int32_t>((ei.w >> 8) & 3);
    out->stoped_cycle = static_cast<int32_t>((ei.w >> 12) & 0xff);  // cycles the current dead ball has waited
    out->ball_collided = static_cast<int32_t>((ei.w >> 20) & 1);
    out->flags = static_cast<int32_t>(((ei.w >> 21) & 1) ? S2D_FLAG_DONE : 0) | (out->ball_collided ? S2D_FLAG_BALL_COLLIDED : 0);
    out->left_score = static_cast<int32_t>(ej.x);
    out->right_score = static_cast<int32_t>(ej.y);
    out->ball_x = ball.x; out->ball_y = ball.y; out->ball_vx = ball.z; out->ball_vy = ball.w;
    out->episode_return = ef.x;
    out->num_players = np;
    for (int j = 0; j < np; ++j) {
      S2DPlayerSnapshot& q = out->players[j];
      q.x = pa[j].x; q.y = pa[j].y; q.vx = pa[j].z; q.vy = pa[j].w;
      q.body_direction = pb[j].x; q.stamina = pb[j].y; q.effort = pb[j].z; q.recovery = pb[j].w;
      q.stamina_capacity = pc[j];
      q.side = j < pps ? S2D_SIDE_LEFT : S2D_SIDE_RIGHT;
      q.uniform_number = (j < pps ? j : j - pps) + 1;
      q.collided = (ej.z >> j) & 1;
      q.kicked = (ej.w >> j) & 1;
    }
    return S2D_OK;
  }
  float4 f[4];
  uint4 u;
  for (int p = 0; p < 4; ++p)
    S2D_CUDA(h, cudaMemcpyAsync(&f[p], base + (p * n + static_cast<size_t>(i)) * 16, 16, cudaMemcpyDeviceToHost, s));
  S2D_CUDA(h, cudaMemcpyAsync(&u, base + (4 * n + static_cast<size_t>(i)) * 16, 16, cudaMemcpyDeviceToHost, s));
  S2D_CUDA(h, cudaStreamSynchronize(s));
  memset(out, 0, sizeof(*out));
  out->cycle = static_cast<int32_t>(u.y);
  out->game_mode_type = S2D_PM_PLAY_ON;  // the trainer forces PlayOn every cycle (soccer_2d_env.py:242)
  out->game_mode_side = S2D_SIDE_LEFT;
  out->step_number = static_cast<int32_t>(u.x);
  out->episode = static_cast<int32_t>(u.z);
  out->flags = static_cast<int32_t>(u.w);
  out->ball_x = f[2].x; out->ball_y = f[2].y; out->ball_vx = f[2].z; out->ball_vy = f[2].w;
  out->mem_distance_to_ball = f[3].x;
  out->mem_body_ball_angle_diff = f[3].y;
  out->episode_return = f[3].w;
  out->ball_collided = (u.w & S2D_FLAG_BALL_COLLIDED) ? 1 : 0;
  out->num_players = 1;
  S2DPlayerSnapshot& p = out->players[0];
  p.x = f[0].x; p.y = f[0].y; p.vx = f[0].z; p.vy = f[0].w;
  p.body_direction = f[1].x; p.stamina = f[1].y; p.effort = f[1].z; p.recovery = f[1].w;
  p.stamina_capacity = f[3].z;
  p.side = S2D_SIDE_LEFT;
  p.uniform_number = 1;  // DoMovePlayer(our_side=True, uniform_number=1), reach_ball_env.py:190-194
  p.collided = (u.w & S2D_FLAG_PLAYER_COLLIDED) ? 1 : 0;
  p.kicked = (u.w & S2D_FLAG_KICKED) ? 1 : 0;
  return S2D_OK;
}

// ---- heterogeneous players ---------------------------------------------------------------------------------
// host-side Philox4x32-10, the same function as s2d_math.cuh's (counter = (env lo, env hi, index, purpose<<24 | sub))
static void philox_host(uint64_t seed, uint64_t env, uint32_t index, uint32_t purpose, uint32_t sub, uint32_t out[4]) {
  uint32_t c0 = static_cast<uint32_t>(env), c1 = static_cast<uint32_t>(env >> 32), c2 = index, c3 = (purpose << 24) | sub;
  uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
  for (int i = 0; i < 10; ++i) {
    const uint64_t p0 = static_cast<uint64_t>(0xD2511F53u) * c0, p1 = static_cast<uint64_t>(0xCD9E8D57u) * c2;
    const uint32_t n0 = static_cast<uint32_t>(p1 >> 32) ^ c1 ^ k0, n2 = static_cast<uint32_t>(p0 >> 32) ^ c3 ^ k1;
    c1 = static_cast<uint32_t>(p1);
    c3 = static_cast<uint32_t>(p0);
    c0 = n0;
    c2 = n2;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

static S2DPlayerType default_player_type(const S2DServerParam& sp) {
  S2DPlayerType t{};
  t.player_decay = sp.player_decay;
  t.inertia_moment = sp.inertia_moment;
  t.dash_power_rate = sp.dash_power_rate;
  t.stamina_inc_max = sp.stamina_inc_max;
  t.kickable_margin = sp.kickable_margin;
  t.kick_rand = sp.kick_rand;
  t.extra_stamina = sp.extra_stamina;
  t.effort_max = sp.effort_max;
  t.effort_min = sp.effort_min;
  t.kick_power_rate = sp.kick_power_rate;
  return t;
}

// rcssserver HeteroPlayer (heteroplayer.cpp; default player.conf): four independent trade-offs, re-drawn until the
// speed the type can sustain, effort_max * dash_power_rate * max_dash_power / (1 - player_decay), lies within 0.1
// below player_speed_max.  Draws: Philox (seed, type id, trial, purpose 4), one word per trade-off, in float.
int s2d_generate_player_types(uint64_t seed, const S2DServerParam* sp, S2DPlayerType* out, int n) {
  if (!sp || !out || n < 1 || n > S2D_MAX_PLAYER_TYPES) return S2D_ERR_INVALID;
  out[0] = default_player_type(*sp);
  for (int id = 1; id < n; ++id) {
    S2DPlayerType t = out[0];
    for (uint32_t trial = 0; trial < 1000u; ++trial) {
      uint32_t w[4];
      philox_host(seed, static_cast<uint64_t>(id), trial, 4u, 0u, w);
      const float u0 = static_cast<float>(w[0] >> 8) * (1.0f / 16777216.0f), u1 = static_cast<float>(w[1] >> 8) * (1.0f / 16777216.0f);
      const float u2 = static_cast<float>(w[2] >> 8) * (1.0f / 16777216.0f), u3 = static_cast<float>(w[3] >> 8) * (1.0f / 16777216.0f);
      const float d_decay = -0.1f + 0.2f * u0;          // player_decay_delta_min / max
      const float d_dash = -0.0012f + 0.002f * u1;      // new_dash_power_rate_delta_min / max
      const float d_kick = -0.1f + 0.2f * u2;           // kickable_margin_delta_min / max
      const float d_extra = 50.0f * u3;                 // extra_stamina_delta_min / max
      S2DPlayerType c = out[0];
      c.player_decay = sp->player_decay + d_decay;
      c.inertia_moment = sp->inertia_moment + d_decay * 25.0f;   // inertia_moment_delta_factor
      c.dash_power_rate = sp->dash_power_rate + d_dash;
      c.stamina_inc_max = sp->stamina_inc_max + d_dash * -6000.0f;  // new_stamina_inc_max_delta_factor
      c.kickable_margin = sp->kickable_margin + d_kick;
      c.kick_rand = sp->kick_rand + d_kick * 1.0f;               // kick_rand_delta_factor
      c.extra_stamina = sp->extra_stamina + d_extra;
      c.effort_max = sp->effort_max + d_extra * -0.004f;         // effort_max_delta_factor
      c.effort_min = sp->effort_min + d_extra * -0.004f;         // effort_min_delta_factor
      const float real_speed_max = c.effort_max * c.dash_power_rate * sp->max_dash_power / (1.0f - c.player_decay);
      if (sp->player_speed_max - 0.1f < real_speed_max && real_speed_max < sp->player_speed_max) {
        t = c;
        break;
      }
    }
    out[id] = t;
  }
  return S2D_OK;
}

static int set_player_types(S2DHandle h, const S2DPlayerType* types, int n, const uint8_t* type_of_player, bool per_match) {
  if (!h) return S2D_ERR_INVALID;
  if (h->cfg.scenario != S2D_SCENARIO_FULLGAME) return fail(h, S2D_ERR_INVALID, "player types exist in the FULLGAME scenario only");
  if (n == 0) {
    h->hetero = false;
    return S2D_OK;
  }
  const int np = 2 * h->cfg.players_per_side;
  if (!types || !type_of_player || n < 1 || n > S2D_MAX_PLAYER_TYPES) return fail(h, S2D_ERR_INVALID, "need 1..%d player types and the type of each of the %d players", S2D_MAX_PLAYER_TYPES, np);
  float rows[S2D_MAX_PLAYER_TYPES * PT_ROW] = {};
  for (int k = 0; k < n; ++k) {
    const S2DPlayerType& t = types[k];
    if (!(t.player_decay >= 0.0f && t.player_decay < 1.0f) || !(t.kickable_margin > 0.0f) || !(t.effort_min <= t.effort_max) ||
        !(t.dash_power_rate > 0.0f) || !(t.inertia_moment >= 0.0f))
      return fail(h, S2D_ERR_INVALID, "player type %d is not physical (decay in [0,1), kickable_margin > 0, effort_min <= effort_max, ...)", k);
    float* r = rows + k * PT_ROW;
    r[PT_PLAYER_DECAY] = t.player_decay;
    r[PT_INERTIA_MOMENT] = t.inertia_moment;
    r[PT_DASH_POWER_RATE] = t.dash_power_rate;
    r[PT_STAMINA_INC_MAX] = t.stamina_inc_max;
    r[PT_KICKABLE_MARGIN] = t.kickable_margin;
    r[PT_KICK_RAND] = t.kick_rand;
    r[PT_EXTRA_STAMINA] = t.extra_stamina;
    r[PT_EFFORT_MAX] = t.effort_max;
    r[PT_EFFORT_MIN] = t.effort_min;
    r[PT_KICK_POWER_RATE] = t.kick_power_rate;
    r[PT_KICKABLE_AREA] = h->cfg.sp.player_size + h->cfg.sp.ball_size + t.kickable_margin;  // as S2D_DERIVED_PARAMS
  }
  uint8_t type_of[32] = {};
  std::vector<uint8_t> planes;  // per match: transposed to the state's match-minor order, padding columns = type 0
  const FgLayout L{h->cfg.num_envs, np};
  if (per_match) {
    planes.assign(L.nr() * np, 0);
    for (int64_t e = 0; e < h->cfg.num_envs; ++e)
      for (int j = 0; j < np; ++j) {
        const uint8_t t = type_of_player[e * np + j];
        if (t >= n) return fail(h, S2D_ERR_INVALID, "player %d of match %lld has type %d, but there are %d types", j, static_cast<long long>(e), t, n);
        planes[static_cast<size_t>(j) * L.nr() + e] = t;
      }
  } else {
    for (int j = 0; j < np; ++j) {
      if (type_of_player[j] >= n) return fail(h, S2D_ERR_INVALID, "player %d has type %d, but there are %d types", j, type_of_player[j], n);
      type_of[j] = type_of_player[j];
    }
  }
  DeviceGuard guard(h->cfg.device);
  if (!h->d_types) S2D_CUDA(h, cudaMalloc(&h->d_types, sizeof(rows)));
  S2D_CUDA(h, cudaMemcpy(h->d_types, rows, sizeof(rows), cudaMemcpyHostToDevice));  // synchronous: later launches see it
  if (per_match) {
    if (!h->d_type_of) S2D_CUDA(h, cudaMalloc(&h->d_type_of, planes.size()));
    S2D_CUDA(h, cudaMemcpy(h->d_type_of, planes.data(), planes.size(), cudaMemcpyHostToDevice));
  }
  h->kp.player_types = h->d_types;
  h->kp.type_of_match = per_match ? h->d_type_of : nullptr;
  memcpy(h->kp.type_of, type_of, sizeof(type_of));
  for (int k = 0; k < S2D_MAX_PIPELINE_SLOTS; ++k)
    if (h->slot_bound[k]) slot_params(h, k);
  h->hetero = true;
  return S2D_OK;
}

int s2d_set_scripted_players(S2DHandle h, uint32_t mask) {
  if (!h) return S2D_ERR_INVALID;
  if (h->cfg.scenario != S2D_SCENARIO_FULLGAME) return fail(h, S2D_ERR_INVALID, "scripted players exist in FULLGAME only");
  const int np = s2d_num_players(&h->cfg);
  if (np < 32 && (mask >> np) != 0u)
    return fail(h, S2D_ERR_INVALID, "scripted-player mask 0x%x names players beyond the %d of a match", mask, np);
  h->kp.scripted_mask = mask;  // (the parameter block goes with each launch: the next one enqueued sees it)
  for (int k = 0; k < S2D_MAX_PIPELINE_SLOTS; ++k)
    if (h->slot_bound[k]) slot_params(h, k);
  return S2D_OK;
}

int s2d_set_player_types(S2DHandle h, const S2DPlayerType* types, int n, const uint8_t* type_of_player) {
  return set_player_types(h, types, n, type_of_player, false);
}
int s2d_set_player_types_per_match(S2DHandle h, const S2DPlayerType* types, int n, const uint8_t* type_of_player) {
  return set_player_types(h, types, n, type_of_player, true);
}

static int rollout_mlp(S2DHandle h, const S2DMlpPolicy* policy, int k_substeps, float epsilon, void* actions_out,
                       void* q_out, const TrajOut& traj, bool actor, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!h->bound) return fail(h, S2D_ERR_UNBOUND, "s2d_bind has not been called");
  const bool shoot = h->cfg.scenario == S2D_SCENARIO_SHOOT;
  const int mode = h->cfg.action_mode;
  if (actor) {
    if (h->cfg.scenario != S2D_SCENARIO_REACHBALL || (mode != S2D_ACT_CONTINUOUS && mode != S2D_ACT_TURNING))
      return fail(h, S2D_ERR_INVALID, "s2d_rollout_actor_collect: REACHBALL with Box(1) or Box(4) actions only");
  } else if (h->cfg.scenario == S2D_SCENARIO_FULLGAME || mode != S2D_ACT_DISCRETE || h->cfg.action_space_size > (shoot ? 24 : 16)) {
    return fail(h, S2D_ERR_INVALID, "s2d_rollout_mlp: REACHBALL with Discrete(n <= 16) or SHOOT with Discrete(n <= 24) actions only");
  }
  if (!policy || !policy->w1 || !policy->b1 || !policy->w2 || !policy->b2 || !policy->w3 || !policy->b3 || policy->hidden != kMlpHidden)
    return fail(h, S2D_ERR_INVALID, "s2d_rollout_mlp: six weight pointers and hidden = %d are required", kMlpHidden);
  if (k_substeps < 1 || k_substeps > kMaxSubsteps) return fail(h, S2D_ERR_INVALID, "k_substeps must be in 1..%d", kMaxSubsteps);
  if (!(epsilon >= 0.0f && epsilon <= 1.0f)) return fail(h, S2D_ERR_INVALID, "epsilon / noise must be in [0, 1]");
  DeviceGuard guard(h->cfg.device);
  const int outputs = actor ? (mode == S2D_ACT_TURNING ? 4 : 1) : h->cfg.action_space_size;
  const MlpWeights w{policy->w1, policy->b1, policy->w2, policy->b2, policy->w3, policy->b3, kObsDim, outputs};
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int rc = before_user_op(h, s)) return rc;
  uint8_t* ao = static_cast<uint8_t*>(actions_out);
  float* qo = static_cast<float*>(q_out);
#define S2D_ROLLOUT(SCN, ACT)                                                                                         \
  do {                                                                                                                \
    if (h->cfg.noise) rollout_mlp_kernel<SCN, kVarNoisy, ACT><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj); \
    else if (h->default_sp) rollout_mlp_kernel<SCN, kVarDefault, ACT><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj); \
    else rollout_mlp_kernel<SCN, kVarRuntime, ACT><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj); \
  } while (0)
  if (policy->precision < 0 || policy->precision > 2)
    return fail(h, S2D_ERR_INVALID, "precision: 0 (TF32, tcgen05), 1 (bf16, mma.sync), 2 (TF32, mma.sync)");
  if (policy->precision == 0) {  // the network on tcgen05 (TF32 operands, accumulators in tensor memory)
#define S2D_TC5(SCN, ACT)                                                                                              \
  do {                                                                                                                 \
    if (h->cfg.noise) rollout_mlp_tc5_kernel<SCN, kVarNoisy, ACT><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj); \
    else if (h->default_sp) rollout_mlp_tc5_kernel<SCN, kVarDefault, ACT><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj); \
    else rollout_mlp_tc5_kernel<SCN, kVarRuntime, ACT><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj); \
  } while (0)
    if (actor && mode == S2D_ACT_TURNING) S2D_TC5(S2D_SCENARIO_REACHBALL, S2D_ACT_TURNING);
    else if (actor) S2D_TC5(S2D_SCENARIO_REACHBALL, S2D_ACT_CONTINUOUS);
    else if (shoot) S2D_TC5(S2D_SCENARIO_SHOOT, S2D_ACT_DISCRETE);
    else S2D_TC5(S2D_SCENARIO_REACHBALL, S2D_ACT_DISCRETE);
#undef S2D_TC5
    S2D_CUDA(h, cudaGetLastError());
    h->env_steps += static_cast<uint64_t>(h->cfg.num_envs) * static_cast<uint64_t>(k_substeps);
    return after_user_op(h, s);
  }
  if (policy->precision == 1 && (actor || h->cfg.noise))
    return fail(h, S2D_ERR_INVALID, "precision 1 (bf16): Q-networks on a handle without noise only");
  if (policy->precision == 1) {
    if (shoot) {
      if (h->default_sp) rollout_mlp_kernel<S2D_SCENARIO_SHOOT, kVarDefault, S2D_ACT_DISCRETE, true><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj);
      else rollout_mlp_kernel<S2D_SCENARIO_SHOOT, kVarRuntime, S2D_ACT_DISCRETE, true><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj);
    } else {
      if (h->default_sp) rollout_mlp_kernel<S2D_SCENARIO_REACHBALL, kVarDefault, S2D_ACT_DISCRETE, true><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj);
      else rollout_mlp_kernel<S2D_SCENARIO_REACHBALL, kVarRuntime, S2D_ACT_DISCRETE, true><<<h->grid, kBlock, 0, s>>>(h->kp, k_substeps, w, epsilon, ao, qo, traj);
    }
  } else if (actor && mode == S2D_ACT_TURNING) S2D_ROLLOUT(S2D_SCENARIO_REACHBALL, S2D_ACT_TURNING);
  else if (actor) S2D_ROLLOUT(S2D_SCENARIO_REACHBALL, S2D_ACT_CONTINUOUS);
  else if (shoot) S2D_ROLLOUT(S2D_SCENARIO_SHOOT, S2D_ACT_DISCRETE);
  else S2D_ROLLOUT(S2D_SCENARIO_REACHBALL, S2D_ACT_DISCRETE);
#undef S2D_ROLLOUT
  S2D_CUDA(h, cudaGetLastError());
  h->env_steps += static_cast<uint64_t>(h->cfg.num_envs) * static_cast<uint64_t>(k_substeps);
  return after_user_op(h, s);
}

int s2d_rollout_mlp(S2DHandle h, const S2DMlpPolicy* policy, int k_substeps, float epsilon, void* actions_out,
                    void* q_out, void* stream) {
  return rollout_mlp(h, policy, k_substeps, epsilon, actions_out, q_out, TrajOut{nullptr, nullptr, nullptr, nullptr, nullptr},
                     false, stream);
}

int s2d_rollout_mlp_collect(S2DHandle h, const S2DMlpPolicy* policy, int k_substeps, float epsilon,
                            const S2DTrajectory* t, void* stream) {
  if (!h) return S2D_ERR_INVALID;
  if (!t) return fail(h, S2D_ERR_INVALID, "trajectory pointer is NULL");
  return rollout_mlp(h, policy, k_substeps, epsilon, nullptr, nullptr, TrajOut{t->obs, t->actions, nullptr, t->reward, t->done},
                     false, stream);
}

int s2d_rollout_actor_collect(S2DHandle h, const S2DMlpPolicy* actor, int k_substeps, float noise,
                              const S2DTrajectory* t, void* stream) {
  const TrajOut traj = t ? TrajOut{t->obs, nullptr, t->actions_f, t->reward, t->done}
                         : TrajOut{nullptr, nullptr, nullptr, nullptr, nullptr};
  return rollout_mlp(h, actor, k_substeps, noise, nullptr, nullptr, traj, true, stream);
}

int s2d_pipeline_info(S2DHandle h, int* slots_bound, int* d2h_copies_last_step) {
  if (!h) return S2D_ERR_INVALID;
  int nb = 0;
  for (int k = 0; k < S2D_MAX_PIPELINE_SLOTS; ++k) nb += h->slot_bound[k] ? 1 : 0;
  if (slots_bound) *slots_bound = nb;
  if (d2h_copies_last_step) *d2h_copies_last_step = h->last_d2h_copies;
  return S2D_OK;
}

int s2d_launch_info(S2DHandle h, int* grid, int* block, int* kernels_per_step) {
  if (!h) return S2D_ERR_INVALID;
  if (grid) *grid = h->grid;
  if (block) *block = kBlock;
  if (kernels_per_step) *kernels_per_step = 1;
  if (block && h->cfg.scenario == S2D_SCENARIO_FULLGAME) *block = kFgBlock;
  return S2D_OK;
}

}  // extern "C"
