// ctk_engine.cu -- the C ABI of libctk_b200.so (include/ctk_b200.h): handle, device buffers, per-tick launch
// sequences for MPPI / CEM / RPGD.  No torch types, no CPU fallback: every entry point fails if CUDA does.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <memory>
#include <string>
#include <vector>

#include "../../include/ctk_b200.h"
#include "ctk_derive.h"
#include "ctk_launch.h"
#include "ctk_mlp_tc.cuh"

using namespace ctk;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(call)                                                                                     \
  do {                                                                                               \
    cudaError_t _e = (call);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return fail(CTK_ECUDA, std::string(#call) + ": " + cudaGetErrorString(_e) + " (" __FILE__ ":" + \
                                 std::to_string(__LINE__) + ")");                                    \
  } while (0)
#define REQ(cond, msg) \
  do {                 \
    if (!(cond)) return fail(CTK_EINVAL, std::string("invalid argument: ") + (msg)); \
  } while (0)

// Owning device (or, Pinned, page-locked host) allocation of n elements of T: move-only, freed in the destructor, converts to
// T* so that kernel argument structs and copies take it as they took the raw pointer.  zero: cudaMemset / memset after the
// allocation (the mailbox, partials and record buffers rely on starting at zero).
template <typename T, bool Pinned = false>
class Owned {
 public:
  Owned() = default;
  Owned(const Owned&) = delete;
  Owned& operator=(const Owned&) = delete;
  Owned(Owned&& o) noexcept : p_(o.p_) { o.p_ = nullptr; }
  Owned& operator=(Owned&& o) noexcept {
    if (this != &o) { reset(); p_ = o.p_; o.p_ = nullptr; }
    return *this;
  }
  ~Owned() { reset(); }
  operator T*() const { return p_; }
  T* get() const { return p_; }
  void reset() {
    if (p_ && Pinned) cudaFreeHost(p_);
    else if (p_) cudaFree(p_);
    p_ = nullptr;
  }
  // frees what was held first; on failure the pointer stays null
  cudaError_t alloc(size_t n, bool zero = true, unsigned int host_flags = cudaHostAllocDefault) {
    reset();
    const size_t bytes = (n ? n : 1) * sizeof(T);
    void* q = nullptr;
    cudaError_t e = Pinned ? cudaHostAlloc(&q, bytes, host_flags) : cudaMalloc(&q, bytes);
    if (e != cudaSuccess) return e;
    p_ = static_cast<T*>(q);
    if (zero && Pinned) memset(q, 0, bytes);
    else if (zero) e = cudaMemset(q, 0, bytes);
    return e;
  }

 private:
  T* p_ = nullptr;
};
template <typename T>
using Pinned = Owned<T, true>;

struct ctk_handle {
  ctk_config cfg;
  OdeC ode;
  FwdK fwd;
  CostC cost;
  MlpDev mlp;
  Owned<DevConsts> d_kc;  // device copy of {fwd, cost}
  Owned<float> d_kx;      // device: {lo, hi, k_du2, k_udu}
  cudaStream_t stream = nullptr;
  int N = 0, NG = 0, off = 0, H = 0, period = 1, n_ind = 0, nblocks = 0;
  int mppi_grid = 0, mppi_block = 0, mppi_rpb = 0, mppi_iters = 0, mppi_stash = 0, num_sms = 0;  // rpb: rollouts per block
  // K1 for the ODE predictor (ctk_kernels_mppi_ode.cuh)
  ctk_ode_params ode_p{};
  ctk_cost_params cost_p{};
  OdeHot ode_hot{};
  bool ode_kernel = false;     // MPPI + ODE predictor + intermediate_steps == 1 + few inducing points
  int ode_ilp = 2, ode_period_t = 0, ode_grid = 0, ode_block = 0, ode_fshare16 = 16;
  Owned<unsigned long long> d_trace;  // optional per-block phase timeline of the last ODE-kernel launch
  size_t ode_smem = 0;
  // fused tick finish / cross-GPU exchange (MppiFuse)
  Owned<unsigned long long> d_mbox;               // local mailbox (layout: MppiFuse)
  unsigned int bseq = 0;                          // sequence number of the exchange barrier (ctk_exchange_barrier)
  bool chain_hint = false;                        // set by ctk_step_device_n for ticks 1.. of a chain: the tick may poll the hand-over
  bool chain_next = false;                        // set by ctk_step_device_n for ticks that a chained tick follows: publish the hand-over
  unsigned long long* mbox_peer[CTK_MAX_PEERS] = {nullptr};
  bool mbox_ipc[CTK_MAX_PEERS] = {false};
  int xworld = 1, xrank = 0;
  unsigned int xseq = 0;
  // common
  Owned<float> d_u_prev, d_u_out, d_J;
  Pinned<float> h_pin;     // MAPPED pinned memory: s[8] | u, status, sequence flag .. [16) | one [H] state array (HostMirror layout)
  float* d_pin = nullptr;  // the device's view of h_pin
  Pinned<char> h_log[8];   // pinned host buffers of ctk_get_log_view, by log id
  size_t h_log_cap[8] = {0};
  HostMirror mirror{nullptr, 0};  // non-null only while a host-facing tick (ctk_step / ctk_step_state) is being enqueued
  unsigned int hseq = 0;
  // mppi
  Owned<float> d_u_nom, d_partials, d_record;
  // cem
  Owned<float> d_mu, d_sd;
  Owned<uint64_t> d_keys[2];
  Owned<int32_t> d_elite_idx;
  int elite_log_cap = 0, elite_log_rows = 0;
  int cem_it = 0, cem_iters = 0, cem_cand = 0;
  uint64_t* cem_cand_ptr = nullptr;
  NoiseSrc cem_noise{};
  Owned<unsigned long long> d_cem_cand, d_cem_dist;  // persistent CEM tick: tagged candidate / distribution slots
  unsigned int cem_seq = 0;
  int cem_tick_per_sm = -1;  // resident blocks per SM of the persistent tick kernel (re-queried when the instantiation changes)
  bool cem_coop_refused = false;  // the runtime refused the cooperative launch once: multi-launch path from then on
  // rpgd
  Owned<float> d_Q[2], d_m[2], d_v[2], d_ages[2];
  int cur = 0;
  const float* pending_s = nullptr;  // gradient-assisted CEM modes: state pointer of the tick in flight
  Owned<float> d_unom_log, d_ages_log, d_Q_log;
  Owned<int32_t> d_best_idx;
  // logs
  Owned<float> d_log_traj_soa, d_log_Q_soa, d_log_tmp;
  // top-M logging (ctk_get_log_top): K4 key buffers, gathered rows, pinned host staging
  Owned<uint64_t> d_top_keys[2];
  Owned<float> d_top_out;
  Pinned<float> h_top;
  size_t top_keys_cap = 0, top_out_cap = 0;
  // injected noise queue
  Owned<float> d_inj;
  size_t inj_cap = 0, inj_size = 0, inj_pos = 0;
  // mlp
  Owned<float> d_mlp;
  Owned<uint8_t> d_mlp_tc;  // tcgen05 engine blob (ctk_mlp_tc.cuh)
  Owned<float> d_rnn_h;     // recurrent predictor: saved hidden state [2][2 hid] (row 0 current, row 1 before the last update)
  const float* step_s = nullptr;  // state pointer of the tick in flight (staged MPPI ticks: predictor.update runs in ctk_step_finish)
  // environments beyond the CartPole (ctk_kernels_env.cuh): env id, dimensions, parameter block, per-input limits
  int env = 0, ns = 6, nu = 1;
  EnvParams env_p{};
  bool env_p_set = false;
  float lo_v[kEnvMaxControls] = {0}, hi_v[kEnvMaxControls] = {0};
  // multi-client batching (ctk_step_batch): per-client state sits behind the pointers of client 0 at fixed strides
  int nclients = 1;
  uint32_t client_tick[kMaxBatchClients] = {0};
  Pinned<float> h_batch;  // [nclients][2] u, status
  size_t mbox_stride = 0, partials_stride = 0;
  // counters
  int64_t count = 0, adam_step = 0, tick = 0, launches = 0;
  bool was_reset = false;
  // optional CUDA-event timing of the dominant (rollout) kernel, for bench.py's live roofline measurement
  bool timing = false;
  std::vector<cudaEvent_t> ev;  // pairs
  size_t ev_used = 0;
  std::string last_kernel;  // instantiation of the last rollout-kernel launch (ctk_last_kernel: tests pin the production kernels)

  ~ctk_handle() {
    close_peers();
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
  void close_peers() {  // the IPC-mapped peer mailboxes of ctk_exchange_connect
    for (int r = 0; r < CTK_MAX_PEERS; ++r) {
      if (mbox_ipc[r] && mbox_peer[r]) cudaIpcCloseMemHandle(mbox_peer[r]);
      mbox_peer[r] = nullptr; mbox_ipc[r] = false;
    }
  }
};

struct KernelTimer {  // records an event pair around the dominant kernel launch when timing is enabled
  ctk_handle* h;
  bool on;
  explicit KernelTimer(ctk_handle* hh) : h(hh), on(false) {
    if (!h->timing) return;
    if (h->ev_used + 2 > h->ev.size()) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
      h->ev.push_back(a);
      h->ev.push_back(b);
    }
    on = cudaEventRecord(h->ev[h->ev_used], h->stream) == cudaSuccess;
  }
  ~KernelTimer() {
    if (on) {
      cudaEventRecord(h->ev[h->ev_used + 1], h->stream);
      h->ev_used += 2;
    }
  }
};

// ---------------------------------------------------------------------------------------------------------------
static void mppi_ode_geometry(ctk_handle* h);
static PredKind pred_kind(const ctk_handle* h);
static bool tile_engine(PredKind pred);

// Host-side constants of the rollout kernels (and, MPPI, the ODE kernel's geometry) from cfg / ode_p / cost_p: no device access
static void derive_consts(ctk_handle* h) {
  if (h->env != 0) return;  // general environments carry their constants in the kernel parameters (EnvParams)
  h->cem_tick_per_sm = -1;  // the cost kind selects the persistent tick's instantiation (register count): re-query its occupancy
  if (h->cfg.optimizer == CTK_OPT_MPPI) {
    const ctk_config& c = h->cfg;
    MppiCorr mc{(double)c.mppi_cc_weight, (double)c.mppi_coef_du2, (double)c.mppi_R, (double)c.mppi_half_R,
                (double)c.mppi_neg_inv_LBD, (double)c.mppi_stdev, (double)c.action_low, (double)c.action_high};
    derive_ode_hot(h->ode_p, h->cost_p, h->H, mc, h->ode_hot);
    mppi_ode_geometry(h);
  } else if (h->cfg.optimizer == CTK_OPT_CEM) {
    // K3s (scaled-variable CEM rollout): the same constants with a zero MPPI correction
    const ctk_config& c = h->cfg;
    MppiCorr mc{0.0, 0.0, 0.0, 0.0, 0.0, 0.0, (double)c.action_low, (double)c.action_high};
    derive_ode_hot(h->ode_p, h->cost_p, h->H, mc, h->ode_hot);
    h->ode_kernel = c.predictor == CTK_PRED_ODE && h->ode_p.intermediate_steps <= 1 && getenv("CTK_CEM_GENERIC") == nullptr;
  }
}

// Copies the constants derive_consts / derive_* produced to d_kc / d_kx
static cudaError_t upload_consts(ctk_handle* h) {
  if (h->env != 0) return cudaSuccess;
  DevConsts kc;
  kc.fwd = h->fwd;
  kc.cost = h->cost;
  kc.ode = h->ode;
  const ctk_config& c = h->cfg;
  const float kx[4] = {c.action_low, c.action_high, (float)((double)c.mppi_cc_weight * (double)c.mppi_coef_du2),
                       (float)((double)c.mppi_cc_weight * (double)c.mppi_R)};
  // the stream may still run kernels that read the old constants: order the copies on it
  cudaError_t e = cudaMemcpyAsync(h->d_kc, &kc, sizeof(kc), cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(h->d_kx, kx, sizeof(kx), cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);  // kc / kx are stack variables
  return e;
}

// Noise source for one consumer: the next rows*per_rollout injected draws if the queue is non-empty (error if it
// holds fewer), else in-kernel Philox.
static int make_noise(ctk_handle* h, uint32_t stream_id, int per_rollout, int uniform, size_t rows, NoiseSrc* out) {
  NoiseSrc ns{};
  ns.key0 = (uint32_t)(h->cfg.seed & 0xffffffffull);
  ns.key1 = (uint32_t)(h->cfg.seed >> 32);
  ns.tick = (uint32_t)h->tick;
  ns.stream = stream_id;
  ns.per_rollout = per_rollout;
  ns.uniform = uniform;
  ns.inj = nullptr;
  const size_t need = rows * (size_t)per_rollout;
  if (h->inj_size > h->inj_pos && need > 0) {
    if (h->inj_size - h->inj_pos < need)
      return fail(CTK_EINVAL, "injected-noise queue holds " + std::to_string(h->inj_size - h->inj_pos) + " draws, this consumer needs " +
                                  std::to_string(need));
    ns.inj = h->d_inj + h->inj_pos;
    h->inj_pos += need;
  }
  *out = ns;
  return CTK_OK;
}

// K4: hierarchical bitonic top-k (tf.argsort(...)[:k], ties -> lower index), one launch per level, ping-ponging between b0 and b1
// from level lvl on.  Input: the costs `cost` of n rollouts, or (cost == nullptr) the n candidate keys `keys`.  Levels run until at
// most 1024 keys are left -- exact_k: until exactly k are (one block) -- and at least one runs on costs.  On return keys / n hold
// the result.
static cudaError_t topk_levels(const float* cost, const uint64_t*& keys, int& n, int lvl, int off, int k, bool exact_k, uint64_t* b0,
                               uint64_t* b1, cudaStream_t stream, int64_t& launches) {
  while (cost != nullptr || n > TOPK_THREADS || (exact_k && n != k)) {
    const int nb = (n + TOPK_THREADS - 1) / TOPK_THREADS;
    uint64_t* out = (lvl++ & 1) ? b1 : b0;
    launches++;
    const cudaError_t e = launch_topk_level(cost, keys, n, off, k, out, stream);
    if (e != cudaSuccess) return e;
    cost = nullptr; keys = out; n = nb * k;
  }
  return cudaSuccess;
}

// outer iterations of this CEM tick (optimizer_cem_tf.py:92)
static int cem_tick_iters(const ctk_handle* h) {
  return (h->cfg.cem_warmup && h->count == 0) ? h->cfg.cem_warmup_iterations : h->cfg.cem_outer_it;
}

// next value of a wrapping sequence number that skips 0 (0 marks an empty slot)
static unsigned int next_seq(unsigned int& seq) {
  if (++seq == 0) seq = 1;
  return seq;
}

// ---------------------------------------------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------------------------------------------
extern "C" const char* ctk_last_error(void) { return g_err.c_str(); }
extern "C" int ctk_abi_version(void) { return CTK_ABI_VERSION; }

extern "C" int ctk_destroy(ctk_handle* h) {
  if (!h) return CTK_OK;
  cudaSetDevice(h->cfg.device);
  delete h;
  return CTK_OK;
}

static int inducing_points(int H, int period) { return (int)std::ceil((double)(H - 1) / (double)period) + 1; }  // Interpolator.py:79-84
// rows of the CEM elite-index log: the outer iterations of the longest tick (the warm-up tick may run more)
static int elite_log_rows_max(const ctk_config& c) {
  return (c.cem_warmup && c.cem_warmup_iterations > c.cem_outer_it) ? c.cem_warmup_iterations : c.cem_outer_it;
}

// Every rejection that needs nothing but the arguments: a configuration that cannot run is refused before the device is touched
static int check_config(const ctk_config* cfg, const ctk_ode_params* ode, const ctk_cost_params* cost) {
  REQ(cfg->abi_version == CTK_ABI_VERSION, "abi_version mismatch");
  REQ(cfg->optimizer >= CTK_OPT_MPPI && cfg->optimizer <= CTK_OPT_RPGD, "unknown optimizer");
  REQ(cfg->predictor == CTK_PRED_ODE || cfg->predictor == CTK_PRED_MLP || cfg->predictor == CTK_PRED_GRU, "unknown predictor");
  REQ(cfg->environment == CTK_ENV_CARTPOLE || cfg->environment == CTK_ENV_DUBINS_CAR, "unregistered environment");
  int env_ns = 6, env_nu = 1;
  env_dims(cfg->environment, &env_ns, &env_nu);
  REQ(cfg->num_states == env_ns && cfg->num_control_inputs == env_nu,
      "num_states / num_control_inputs do not match the registered environment (CartPole: 6 / 1, Dubins car: 3 / 2)");
  if (cfg->environment != CTK_ENV_CARTPOLE)
    REQ(cfg->predictor == CTK_PRED_ODE && cfg->num_rollouts == cfg->num_rollouts_global && cfg->num_clients <= 1 && !cfg->cem_uniform_actions,
        "environments other than the CartPole: MPPI, CEM and the gradient optimizers with the environment's ODE, unsharded, one client "
        "(the network predictors are CartPole functors)");
  REQ(cfg->num_rollouts >= 1 && cfg->mpc_horizon >= 1, "num_rollouts and mpc_horizon must be >= 1");
  REQ(cfg->num_rollouts_global >= cfg->num_rollouts && cfg->rollout_offset >= 0 &&
          cfg->rollout_offset + cfg->num_rollouts <= cfg->num_rollouts_global, "bad shard geometry");
  REQ(cost->kind == CTK_COST_DEFAULT || cost->kind == CTK_COST_QUADRATIC_BOUNDARY_GRAD, "unregistered cost function");
  REQ(cfg->action_low <= cfg->action_high, "action_low > action_high");
  if (cfg->optimizer == CTK_OPT_RPGD) {
    REQ(cfg->rpgd_resamp_per >= 1 || cfg->rpgd_gradient_mode != 0, "rpgd_resamp_per must be >= 1");
    REQ(cfg->rpgd_outer_its >= 0 && cfg->rpgd_first_iter_count >= 0, "RPGD iteration counts must be >= 0");
  }
  const int B = cfg->num_clients > 1 ? cfg->num_clients : 1;
  REQ(B <= kMaxBatchClients, "num_clients must be <= 16");
  REQ(B == 1 || (cfg->optimizer == CTK_OPT_MPPI && cfg->predictor == CTK_PRED_ODE && !cfg->logging && cfg->num_rollouts == cfg->num_rollouts_global),
      "multi-client handles are implemented for MPPI with the ODE predictor, logging off, unsharded");
  const int N = cfg->num_rollouts, H = cfg->mpc_horizon, period = cfg->period_interpolation_inducing_points;
  if (cfg->optimizer != CTK_OPT_CEM && period < 1) return fail(CTK_EINVAL, "period_interpolation_inducing_points must be >= 1");
  if (cfg->environment != CTK_ENV_CARTPOLE && cfg->optimizer != CTK_OPT_RPGD) {
    if (cfg->optimizer == CTK_OPT_MPPI && (inducing_points(H, period) * env_nu > 32 || H * env_nu > 1024))
      return fail(CTK_EINVAL, "environment MPPI: n_ind * nu <= 32 and H * nu <= 1024");
    if (cfg->optimizer == CTK_OPT_CEM &&
        !(cfg->cem_best_k >= 1 && cfg->cem_best_k <= 512 && cfg->cem_best_k <= N && H * env_nu <= 1024 && cfg->cem_outer_it >= 1))
      return fail(CTK_EINVAL, "environment CEM needs 1 <= cem_best_k <= min(512, num_rollouts), H * nu <= 1024, cem_outer_it >= 1");
  } else if (cfg->optimizer == CTK_OPT_CEM) {
    if (!(cfg->cem_best_k >= 1 && cfg->cem_best_k <= 512 && cfg->cem_best_k <= cfg->num_rollouts_global && H <= 1024 && cfg->cem_outer_it >= 1))
      return fail(CTK_EINVAL, "CEM needs 1 <= cem_best_k <= min(512, num_rollouts), mpc_horizon <= 1024, cem_outer_it >= 1");
  } else if (cfg->optimizer == CTK_OPT_RPGD) {
    if (!(N <= 1024 && cfg->rpgd_keep_k >= 1 && cfg->rpgd_keep_k <= N && N == cfg->num_rollouts_global && cfg->predictor == CTK_PRED_ODE &&
          ode->intermediate_steps <= 1 && cfg->rpgd_shift_previous >= 0))
      return fail(CTK_EINVAL, "RPGD needs num_rollouts <= 1024 (replicas only, no sharding), the ODE predictor with "
                              "intermediate_steps == 1 and 1 <= keep_k <= num_rollouts");
    if (cfg->rpgd_gradient_mode >= 2 && !(cfg->rpgd_gradient_mode <= 3 && cfg->cem_best_k >= 1 && cfg->cem_best_k <= N && cfg->cem_outer_it >= 1 &&
                                          period == 1 && elite_log_rows_max(*cfg) >= 1))
      return fail(CTK_EINVAL, "gradient-assisted CEM needs 1 <= cem_best_k <= num_rollouts, cem_outer_it >= 1 and inducing-point period 1");
    // environments: the gradient kernel keeps states, q, g, m and v of every horizon step in shared memory (ctk_kernels_env_rpgd.cuh)
    if (cfg->environment != CTK_ENV_CARTPOLE && env_rpgd_smem_bytes(cfg->environment, H) > kEnvRpgdSmemMax) {
      int max_h = 1;
      while (env_rpgd_smem_bytes(cfg->environment, max_h + 1) <= kEnvRpgdSmemMax) ++max_h;
      return fail(CTK_EINVAL, "environment gradient optimizers: mpc_horizon too large for the shared-memory tape of H * (ns + 4 nu) floats "
                              "per trajectory (max " + std::to_string(max_h) + ")");
    }
  }
  return CTK_OK;
}

// K1 geometry of the CartPole MPPI rollout kernels: one CTA per SM, block sized so that every thread runs the same number of
// rollouts (no tail wave).  Needs num_sms; allocates nothing.
static int mppi_geometry(ctk_handle* h) {
  const int N = h->N;
  const PredInfo pred = pred_info(pred_kind(h));
  const int maxb = pred.max_threads;
  const long long slots = (long long)h->num_sms * maxb;
  const int r = (int)((N + slots - 1) / slots);                                  // rollouts per thread
  int T = (int)(((((long long)N + (long long)r * h->num_sms - 1) / ((long long)r * h->num_sms)) + 31) / 32 * 32);
  if (T > maxb) T = maxb;
  if (T < 32) T = 32;
  h->mppi_block = T;
  h->mppi_grid = (int)std::min<long long>(h->num_sms, ((long long)N + T - 1) / T);  // every SM gets a CTA
  if (h->mppi_grid < 1) h->mppi_grid = 1;
  h->mppi_iters = (int)((N + (long long)h->mppi_grid * T - 1) / ((long long)h->mppi_grid * T));
  h->mppi_stash = ((size_t)h->n_ind * T * sizeof(float) <= 96 * 1024) ? 1 : 0;
  if ((size_t)h->n_ind * T * sizeof(float) > 100 * 1024) {  // accumulator array must fit: shrink the block
    T = (int)((100 * 1024 / sizeof(float) / (size_t)h->n_ind) / 32 * 32);
    if (T < 32) return fail(CTK_EINVAL, "MPPI: too many inducing points for the shared-memory accumulators");
    h->mppi_block = T;
    h->mppi_grid = (int)std::min<long long>(h->num_sms, ((long long)N + T - 1) / T);
    h->mppi_stash = 0;
  }
  h->mppi_rpb = h->mppi_block;
  if (tile_engine(pred_kind(h))) {
    // tcgen05 MLP engines (ctk_mlp_tc.cuh): one CTA per SM, every CTA an equal contiguous share of the population (kBalanced); rollouts per
    // block = tiles in flight x 128 (kRolloutsPerBlock)
    h->mppi_block = pred.max_threads; h->mppi_rpb = pred.rollouts_per_pass;
    h->mppi_grid = (int)std::min<long long>((long long)h->num_sms, ((long long)N + 127) / 128);
    if (h->mppi_grid < 1) h->mppi_grid = 1;
    h->mppi_iters = (int)((N + (long long)h->mppi_grid * h->mppi_rpb - 1) / ((long long)h->mppi_grid * h->mppi_rpb));
    h->mppi_stash = 0;
    // what the operand tiles leave of the 227 KB for the per-rollout accumulators [n_ind][rollouts per block]
    if ((size_t)h->n_ind * h->mppi_rpb * sizeof(float) > pred.acc_smem_bytes) return fail(CTK_EINVAL, "tcgen05 MLP engine: too many inducing points (shared memory is taken by the operand tiles)");
  }
  h->partials_stride = (size_t)(h->num_sms > h->mppi_grid ? h->num_sms : h->mppi_grid) * (h->mppi_iters + 1) * (h->n_ind + 2);
  if (h->mppi_grid > CTK_MBOX_BLOCKS || h->num_sms > CTK_MBOX_BLOCKS) return fail(CTK_EINVAL, "device has more SMs than the mailbox has block slots (CTK_MBOX_BLOCKS)");
  h->mbox_stride = (mbox_total_slots(h->n_ind, h->H) + 1) & ~(size_t)1;  // even: the records are polled with 16-byte loads
  return CTK_OK;
}

extern "C" int ctk_create(const ctk_config* cfg, const ctk_ode_params* ode, const ctk_cost_params* cost, ctk_handle** out) {
  REQ(cfg && ode && cost && out, "null pointer");
  int rc = check_config(cfg, ode, cost);
  if (rc != CTK_OK) return rc;
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  REQ(cfg->device >= 0 && cfg->device < ndev, "no such CUDA device");
  CU(cudaSetDevice(cfg->device));

  std::unique_ptr<ctk_handle> owner(new ctk_handle());  // a failing create frees whatever it allocated
  ctk_handle* h = owner.get();
  const int B = cfg->num_clients > 1 ? cfg->num_clients : 1;
  h->cfg = *cfg;
  h->N = cfg->num_rollouts; h->NG = cfg->num_rollouts_global; h->off = cfg->rollout_offset; h->H = cfg->mpc_horizon;
  h->ode_p = *ode; h->cost_p = *cost;
  h->nclients = B;
  h->env = cfg->environment;
  env_dims(cfg->environment, &h->ns, &h->nu);
  for (int c = 0; c < kEnvMaxControls; ++c) { h->lo_v[c] = cfg->action_low; h->hi_v[c] = cfg->action_high; }
  derive_ode(*ode, h->ode);
  derive_fwd(*ode, h->fwd);
  derive_cost(*cost, h->H, h->cost);
  h->mlp = MlpDev{0, nullptr, 0, nullptr, nullptr};
  h->nblocks = (h->N + 127) / 128;
  if (cfg->optimizer == CTK_OPT_MPPI || cfg->optimizer == CTK_OPT_RPGD) {
    h->period = cfg->period_interpolation_inducing_points;
    h->n_ind = inducing_points(h->H, h->period);
  }
  const int N = h->N, H = h->H, nu = h->nu;
  auto A = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && rc == CTK_OK) rc = fail(CTK_ECUDA, std::string("cudaMalloc ") + what + ": " + cudaGetErrorString(e));
  };
  // geometry checks that need the SM count, before any allocation
  if (h->env == 0 && cfg->optimizer != CTK_OPT_RPGD) {
    cudaDeviceProp prop;
    A(cudaGetDeviceProperties(&prop, cfg->device), "props");
    if (rc != CTK_OK) return rc;
    h->num_sms = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    if (cfg->optimizer == CTK_OPT_MPPI && (rc = mppi_geometry(h)) != CTK_OK) return rc;
  }
  derive_consts(h);
  if (B > 1 && !(h->ode_kernel && h->ode_ilp == 1))
    return fail(CTK_EINVAL, "multi-client handles run the one-rollout-per-thread ODE kernel: intermediate_steps == 1, few inducing points, "
                            "num_rollouts <= 1024 x SMs per client");

  A(h->d_u_prev.alloc((size_t)(B > nu ? B : nu)), "u_prev"); A(h->d_u_out.alloc(4 + 2 * (size_t)B), "u_out");
  A(h->d_J.alloc((size_t)N * B), "J");
  if (B > 1) A(h->h_batch.alloc(2 * (size_t)B, false), "pinned (batch results)");
  A(h->d_kc.alloc(1, false), "consts");
  A(h->d_kx.alloc(4), "kx");
  A(h->h_pin.alloc(32 + 2 * (size_t)H, true, cudaHostAllocMapped), "pinned");
  if (h->h_pin) A(cudaHostGetDevicePointer((void**)&h->d_pin, h->h_pin, 0), "pinned (device view)");
  if (cfg->logging) {
    A(h->d_log_traj_soa.alloc((size_t)(H + 1) * h->ns * N), "log_traj");
    A(h->d_log_Q_soa.alloc((size_t)H * nu * N), "log_Q");
    if (h->env == 0) A(h->d_log_tmp.alloc((size_t)(H + 1) * 6 * N), "log_tmp");
  }
  // state arrays are flat [H][nu] ([H] x clients for multi-client MPPI)
  if (cfg->optimizer == CTK_OPT_MPPI) A(h->d_u_nom.alloc((size_t)H * nu * B), "u_nom");
  if (cfg->optimizer == CTK_OPT_CEM || (cfg->optimizer == CTK_OPT_RPGD && cfg->rpgd_gradient_mode >= 2)) {
    // CEM distribution and per-iteration elite log (gradient-assisted CEM: on top of the RPGD population)
    A(h->d_mu.alloc((size_t)H * nu), "mu"); A(h->d_sd.alloc((size_t)H * nu), "sd");
    h->elite_log_cap = elite_log_rows_max(*cfg);
    A(h->d_elite_idx.alloc((size_t)h->elite_log_cap * cfg->cem_best_k), "elite_idx");
  }
  if (cfg->optimizer == CTK_OPT_CEM) {  // K4 keys: level-0 candidates of 256-rollout blocks (CartPole: fused top-k) or 1024-key blocks
    const int blk = h->env == 0 ? 256 : 1024;
    const size_t nk = (size_t)((N + blk - 1) / blk) * cfg->cem_best_k + 1024;
    A(h->d_keys[0].alloc(nk), "keys0"); A(h->d_keys[1].alloc(nk), "keys1");
  }
  if (h->env == 0 && cfg->optimizer == CTK_OPT_MPPI) {
    A(h->d_partials.alloc(h->partials_stride * B), "partials");
    A(h->d_record.alloc((size_t)(h->n_ind + 2) * B), "record");
    A(h->d_mbox.alloc(h->mbox_stride * B), "mailbox");
    h->mbox_peer[0] = h->d_mbox;
  } else if (h->env == 0 && cfg->optimizer == CTK_OPT_CEM) {
    // persistent single-launch tick (cem_tick_kernel): tagged slots for one resident grid
    A(h->d_cem_cand.alloc((size_t)2 * h->num_sms * 128), "cem_cand");  // [blocks <= 2 x SMs][k <= 128]
    A(h->d_mbox.alloc(cem_mbox_slots()), "mailbox");  // fused cross-GPU candidate exchange (CemRefitArgs)
    h->mbox_peer[0] = h->d_mbox;
    A(h->d_cem_dist.alloc((size_t)2 * 512), "cem_dist");
  } else if (cfg->optimizer == CTK_OPT_RPGD) {
    for (int i = 0; i < 2; ++i) {
      A(h->d_Q[i].alloc((size_t)N * H * nu), "Q"); A(h->d_m[i].alloc((size_t)N * H * nu), "m");
      A(h->d_v[i].alloc((size_t)N * H * nu), "v"); A(h->d_ages[i].alloc((size_t)N), "ages");
    }
    A(h->d_unom_log.alloc((size_t)H * nu), "unom_log"); A(h->d_ages_log.alloc((size_t)N), "ages_log");
    A(h->d_Q_log.alloc((size_t)N * H * nu), "Q_log");
    A(h->d_best_idx.alloc((size_t)N), "best_idx");
  }
  if (rc == CTK_OK) A(upload_consts(h), "upload_consts");
  if (rc != CTK_OK) return rc;
  *out = owner.release();
  return CTK_OK;
}

extern "C" int ctk_set_stream(ctk_handle* h, void* s) { REQ(h, "null handle"); h->stream = (cudaStream_t)s; return CTK_OK; }
extern "C" int ctk_set_cost_params(ctk_handle* h, const ctk_cost_params* c) {
  REQ(h && c, "null pointer");
  REQ(c->kind == CTK_COST_DEFAULT || c->kind == CTK_COST_QUADRATIC_BOUNDARY_GRAD, "unregistered cost function");
  h->cost_p = *c;
  derive_cost(*c, h->H, h->cost);
  CU(cudaSetDevice(h->cfg.device));
  derive_consts(h);
  CU(upload_consts(h));
  return CTK_OK;
}
extern "C" int ctk_set_ode_params(ctk_handle* h, const ctk_ode_params* o) {
  REQ(h && o, "null pointer");
  REQ(!(h->cfg.optimizer == CTK_OPT_RPGD && o->intermediate_steps > 1), "RPGD adjoint supports intermediate_steps == 1");
  h->ode_p = *o;
  derive_ode(*o, h->ode);
  derive_fwd(*o, h->fwd);
  CU(cudaSetDevice(h->cfg.device));
  derive_consts(h);
  CU(upload_consts(h));
  return CTK_OK;
}

extern "C" int ctk_set_mlp_weights(ctk_handle* h, const ctk_mlp_weights* w) {
  REQ(h && w && w->W1 && w->b1 && w->W2 && w->b2 && w->W3 && w->b3, "null pointer");
  REQ(w->hidden >= 16 && w->hidden <= 128 && w->hidden % 16 == 0, "hidden must be a multiple of 16 in [16,128]");
  REQ(h->cfg.predictor == CTK_PRED_MLP, "ctk_set_mlp_weights on a handle whose predictor is not CTK_PRED_MLP");
  // every rejection before the current weights are touched: a rejected call leaves the handle as it was
  const bool tc_engine = h->cfg.mlp_engine != CTK_MLP_SIMT;
  if (tc_engine) {
    REQ(h->cfg.mlp_engine >= CTK_MLP_TCGEN05 && h->cfg.mlp_engine <= CTK_MLP_TCGEN05_FAST, "unknown mlp_engine");
    REQ(w->hidden == kTcHidden, "the tcgen05 MLP engines are built for hidden == 128 (use mlp_engine=simt otherwise)");
    REQ(h->cfg.optimizer == CTK_OPT_MPPI || h->cfg.optimizer == CTK_OPT_CEM, "the tcgen05 MLP engines are implemented for MPPI and CEM");
  }
  CU(cudaSetDevice(h->cfg.device));
  const int hid = w->hidden, nf = mlp_blob_floats(hid);
  std::vector<float> blob((size_t)nf, 0.0f);
  float* p = blob.data();
  memcpy(p, w->W1, sizeof(float) * 6 * hid); p += 6 * hid;
  memcpy(p, w->b1, sizeof(float) * hid); p += hid;
  memcpy(p, w->W2, sizeof(float) * hid * hid); p += hid * hid;
  memcpy(p, w->b2, sizeof(float) * hid); p += hid;
  for (int k = 0; k < 5; ++k) for (int j = 0; j < hid; ++j) p[k * hid + j] = w->W3[j * 5 + k];  // W3T[5][hid]
  p += 5 * hid;
  memcpy(p, w->b3, sizeof(float) * 5);
  CU(h->d_mlp.alloc((size_t)nf));
  CU(cudaMemcpy(h->d_mlp, blob.data(), sizeof(float) * nf, cudaMemcpyHostToDevice));
  h->mlp = MlpDev{hid, h->d_mlp, nf, nullptr, nullptr};
  if (tc_engine) {
    // W2 as three bf16 terms (w = w1 + w2 + w3, round-to-nearest-even each), B operand tiles: row n = output unit, k = input unit
    std::vector<uint8_t> tc(kTcBlobBytes, 0);
    auto bf16_rn = [](float f) -> uint16_t {
      uint32_t x; memcpy(&x, &f, 4);
      if ((x & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((x >> 16) | 0x40);  // NaN
      x += 0x7fffu + ((x >> 16) & 1u);
      return (uint16_t)(x >> 16);
    };
    auto bf16_f = [](uint16_t u) -> float { uint32_t x = (uint32_t)u << 16; float f; memcpy(&f, &x, 4); return f; };
    for (int k = 0; k < 128; ++k)
      for (int n = 0; n < 128; ++n) {
        const float wv = w->W2[k * 128 + n];
        const uint16_t t1 = bf16_rn(wv); const float r1 = wv - bf16_f(t1);
        const uint16_t t2 = bf16_rn(r1); const float r2 = r1 - bf16_f(t2);
        const uint16_t t3 = bf16_rn(r2);
        const uint32_t off = tc_tile_offset(n, k);
        memcpy(&tc[0 * kTcTileBytes + off], &t1, 2); memcpy(&tc[1 * kTcTileBytes + off], &t2, 2); memcpy(&tc[2 * kTcTileBytes + off], &t3, 2);
      }
    float* f = reinterpret_cast<float*>(tc.data() + 3 * kTcTileBytes);
    memcpy(f, w->W1, sizeof(float) * 6 * 128); f += 6 * 128;
    memcpy(f, w->b1, sizeof(float) * 128); f += 128;
    memcpy(f, w->b2, sizeof(float) * 128); f += 128;
    for (int k = 0; k < 5; ++k) for (int j = 0; j < 128; ++j) f[k * 128 + j] = w->W3[j * 5 + k];
    f += 5 * 128;
    memcpy(f, w->b3, sizeof(float) * 5);
    {  // B1: layer 1 on the tensor core (single-product engines).  Row n = hidden unit, K = 48: [w1 w1 w1 w2 w2 w3] of W1[:, n] (six
       // inputs each), the three terms of b1[n], zeros -- against the operand row [x1 x2 x3 x1 x2 x1 | 1 1 1 | 0 ..] of the kernel
      uint8_t* b1t = tc.data() + 3 * kTcTileBytes + kTcBlobFloats * 4;
      auto put = [&](int n, int k, uint16_t v) { memcpy(b1t + tc_tile_offset(n, k), &v, 2); };
      for (int n = 0; n < 128; ++n) {
        uint16_t t[6][3];
        for (int i = 0; i < 6; ++i) {
          const float wv = w->W1[i * 128 + n];
          t[i][0] = bf16_rn(wv); const float r1 = wv - bf16_f(t[i][0]);
          t[i][1] = bf16_rn(r1); const float r2 = r1 - bf16_f(t[i][1]);
          t[i][2] = bf16_rn(r2);
        }
        for (int i = 0; i < 6; ++i) {
          put(n, i, t[i][0]); put(n, 6 + i, t[i][0]); put(n, 12 + i, t[i][0]);
          put(n, 18 + i, t[i][1]); put(n, 24 + i, t[i][1]);
          put(n, 30 + i, t[i][2]);
        }
        const float bv = w->b1[n];
        const uint16_t c1 = bf16_rn(bv); const float q1 = bv - bf16_f(c1);
        const uint16_t c2 = bf16_rn(q1); const float q2 = q1 - bf16_f(c2);
        put(n, 36, c1); put(n, 37, c2); put(n, 38, bf16_rn(q2));
      }
    }
    CU(h->d_mlp_tc.alloc(kTcBlobBytes, false));
    CU(cudaMemcpy(h->d_mlp_tc, tc.data(), kTcBlobBytes, cudaMemcpyHostToDevice));
    h->mlp.tc_blob = h->d_mlp_tc;
  }
  return CTK_OK;
}

extern "C" int ctk_set_gru_weights(ctk_handle* h, const ctk_gru_weights* w) {
  REQ(h && w && w->Wi1 && w->Wh1 && w->bi1 && w->bh1 && w->Wi2 && w->Wh2 && w->bi2 && w->bh2 && w->W3 && w->b3, "null pointer");
  REQ(h->cfg.predictor == CTK_PRED_GRU, "ctk_set_gru_weights on a handle whose predictor is not CTK_PRED_GRU");
  REQ(w->hidden >= 8 && w->hidden <= 32 && w->hidden % 8 == 0, "GRU hidden width must be a multiple of 8 in [8,32]");
  CU(cudaSetDevice(h->cfg.device));
  const int hid = w->hidden, g = 3 * hid, nf = gru_blob_floats(hid);
  std::vector<float> blob((size_t)nf, 0.0f);
  float* p = blob.data();
  auto put = [&](const float* src, size_t n) { memcpy(p, src, sizeof(float) * n); p += n; };
  put(w->Wi1, (size_t)6 * g); put(w->Wh1, (size_t)hid * g); put(w->bi1, g); put(w->bh1, g);
  put(w->Wi2, (size_t)hid * g); put(w->Wh2, (size_t)hid * g); put(w->bi2, g); put(w->bh2, g);
  for (int k = 0; k < 5; ++k) for (int j = 0; j < hid; ++j) p[k * hid + j] = w->W3[j * 5 + k];  // W3T[5][hid]
  p += 5 * hid;
  memcpy(p, w->b3, sizeof(float) * 5);
  CU(cudaStreamSynchronize(h->stream));  // kernels in flight may still read the old blob
  h->d_rnn_h.reset();
  CU(h->d_mlp.alloc((size_t)nf));
  CU(cudaMemcpy(h->d_mlp, blob.data(), sizeof(float) * nf, cudaMemcpyHostToDevice));
  CU(h->d_rnn_h.alloc((size_t)4 * hid));  // zero state (SI_Toolkit resets the RNN when the predictor is configured)
  h->mlp = MlpDev{hid, h->d_mlp, nf, nullptr, h->d_rnn_h};
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// noise queue
// ---------------------------------------------------------------------------------------------------------------
extern "C" int ctk_push_injected_noise(ctk_handle* h, const float* z, size_t n) {
  REQ(h && (z || n == 0), "null pointer");
  CU(cudaSetDevice(h->cfg.device));
  if (h->inj_pos == h->inj_size) h->inj_pos = h->inj_size = 0;  // fully consumed: rewind
  if (h->inj_size + n > h->inj_cap) {
    // grow; pending kernels may still read the old buffer -> sync first
    CU(cudaStreamSynchronize(h->stream));
    const size_t cap = (h->inj_size + n) * 2;
    Owned<float> nb;
    CU(nb.alloc(cap, false));
    if (h->inj_size) CU(cudaMemcpy(nb, h->d_inj, h->inj_size * sizeof(float), cudaMemcpyDeviceToDevice));
    h->d_inj = std::move(nb);
    h->inj_cap = cap;
  }
  CU(cudaMemcpyAsync(h->d_inj + h->inj_size, z, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->inj_size += n;
  return CTK_OK;
}
extern "C" int ctk_clear_injected_noise(ctk_handle* h) {
  REQ(h, "null handle");
  h->inj_pos = h->inj_size = 0;
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// reset
// ---------------------------------------------------------------------------------------------------------------
// Sampling arguments of the initial population and of K8, with per-input limits.  The CartPole draws over [rpgd_sample_min,
// rpgd_sample_max] (the gradient-tf tail redraw of K8 over the action limits: rpgd_select_prepare); other environments draw uniformly
// over each input's own [low, high] when the whole control space is sampled (optimizer_rpgd.py:199-205) and always for gradient-tf
// (optimizer_gradient_tf.py:171-177)
static RpgdSelectArgs rpgd_sample_args(ctk_handle* h, NoiseSrc ns) {
  const ctk_config& c = h->cfg;
  RpgdSelectArgs a{};
  a.N = h->N; a.H = h->H; a.k = c.rpgd_keep_k; a.period = h->period; a.n_ind = h->n_ind;
  a.shift_previous = c.rpgd_shift_previous;
  a.noise = ns; a.dist = c.rpgd_distribution;
  a.s_mean = c.rpgd_sample_mean; a.s_std = c.rpgd_sample_stdev;
  const bool whole = h->env != 0 && (c.rpgd_sample_whole_space != 0 || c.rpgd_gradient_mode == 1);
  for (int i = 0; i < kEnvMaxControls; ++i) {
    a.lo[i] = h->lo_v[i]; a.hi[i] = h->hi_v[i];
    a.s_min[i] = whole ? h->lo_v[i] : c.rpgd_sample_min;
    a.s_max[i] = whole ? h->hi_v[i] : c.rpgd_sample_max;
  }
  return a;
}

// Mid-range warm start of `rows` control rows, per input (optimizer_mppi.py:227-231, optimizer_cem_tf.py:113-117), flat [rows][nu].
// The CartPole's limits are the config's (ctk_set_control_limits).
static std::vector<float> mid_range(const ctk_handle* h, size_t rows) {
  std::vector<float> v(rows * h->nu);
  for (size_t t = 0; t < rows; ++t) for (int c = 0; c < h->nu; ++c) v[t * h->nu + c] = 0.5f * (h->lo_v[c] + h->hi_v[c]);
  return v;
}

extern "C" int ctk_reset(ctk_handle* h) {
  REQ(h, "null handle");
  CU(cudaSetDevice(h->cfg.device));
  const std::vector<float> mid = mid_range(h, (size_t)h->H * h->nclients), sd((size_t)h->H * h->nu, h->cfg.cem_initial_action_stdev);
  // self.u, the previous_input of the cost, is reset ONLY by optimizer_cem_tf.optimizer_reset (optimizer_cem_tf.py:117); MPPI (:227-231),
  // RPGD (:527-548), random-action, gradient-tf and the gradient-assisted CEM variants keep the last applied control
  if (h->cfg.optimizer == CTK_OPT_CEM && !h->cfg.cem_uniform_actions) CU(cudaMemsetAsync(h->d_u_prev, 0, sizeof(float) * h->nu, h->stream));
  if (h->cfg.optimizer == CTK_OPT_MPPI) {
    CU(cudaMemcpyAsync(h->d_u_nom, mid.data(), sizeof(float) * mid.size(), cudaMemcpyHostToDevice, h->stream));
  } else if (h->cfg.optimizer == CTK_OPT_CEM) {
    CU(cudaMemcpyAsync(h->d_mu, mid.data(), sizeof(float) * mid.size(), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_sd, sd.data(), sizeof(float) * sd.size(), cudaMemcpyHostToDevice, h->stream));
    if (h->env == 0) CU(cudaStreamSynchronize(h->stream));
    h->cem_it = 0;
  } else if (h->cfg.rpgd_gradient_mode >= 2) {
    // optimizer_cem_naive_grad_tf.py:116-119 / optimizer_cem_grad_bharadhwaj_tf.py:180-184: only the distribution (and count) is
    // reset; the Keras Adam slots of the bharadhwaj variant survive optimizer_reset()
    CU(cudaMemcpyAsync(h->d_mu, mid.data(), sizeof(float) * h->H * h->nu, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_sd, sd.data(), sizeof(float) * h->H * h->nu, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  } else {
    NoiseSrc ns{};
    int rcn = make_noise(h, STREAM_RPGD_INIT, h->n_ind * h->nu, h->cfg.rpgd_distribution == CTK_DIST_UNIFORM, (size_t)h->N, &ns);
    if (rcn != CTK_OK) return rcn;
    h->cur = 0;
    h->launches++;
    RpgdSelectArgs a = rpgd_sample_args(h, ns);
    a.Qn = h->d_Q[0]; a.mn = h->d_m[0]; a.vn = h->d_v[0]; a.agesn = h->d_ages[0];
    CU(launch_rpgd_init(h->nu, a, h->stream));
    h->adam_step = 0;
  }
  CU(cudaStreamSynchronize(h->stream));
  h->count = 0;
  h->was_reset = true;
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// environments beyond the CartPole (SURVEY 8f.3): parameter block, per-input limits, the tick as a plain launch sequence
// ---------------------------------------------------------------------------------------------------------------
extern "C" int ctk_set_env_params(ctk_handle* h, const float* p, int n) {
  REQ(h && p && n >= 0 && n <= 24, "null pointer or more than 24 parameters");
  REQ(h->env != 0, "ctk_set_env_params is for environments other than the CartPole (use ctk_set_ode_params / ctk_set_cost_params)");
  for (int i = 0; i < 24; ++i) h->env_p.p[i] = i < n ? p[i] : 0.0f;
  h->env_p_set = true;
  return CTK_OK;
}
extern "C" int ctk_set_control_limits(ctk_handle* h, const float* low, const float* high, int nu) {
  REQ(h && low && high && nu == h->nu, "null pointer or nu != num_control_inputs");
  for (int c = 0; c < nu; ++c) REQ(low[c] <= high[c], "action_low > action_high");
  REQ(h->env != 0 || (low[0] == h->cfg.action_low && high[0] == h->cfg.action_high), "the CartPole kernels take their limits from ctk_config");
  for (int c = 0; c < nu; ++c) { h->lo_v[c] = low[c]; h->hi_v[c] = high[c]; }
  return CTK_OK;
}

static S0e make_s0e(const ctk_handle* h, const float* s_dev, const float* s_host) {
  S0e s{};
  s.p = s_dev;
  if (s_dev == nullptr) for (int i = 0; i < h->ns; ++i) s.v[i] = s_host[i];
  return s;
}

static int env_rpgd_tick(ctk_handle* h, const S0e& s0, float* u_out_dev);
static int env_tick(ctk_handle* h, const S0e& s0, float* u_out_dev) {
  const ctk_config& c = h->cfg;
  if (!h->env_p_set) return fail(CTK_ESTATE, "environment parameters not set (ctk_set_env_params)");
  const int nu = h->nu;
  h->tick++;
  if (c.optimizer == CTK_OPT_RPGD) return env_rpgd_tick(h, s0, u_out_dev);
  if (c.optimizer == CTK_OPT_MPPI) {
    EnvMppiArgs a{};
    int rcn = make_noise(h, STREAM_MPPI, h->n_ind * nu, 0, (size_t)h->NG, &a.noise);
    if (rcn != CTK_OK) return rcn;
    a.N = h->N; a.off = h->off; a.H = h->H; a.period = h->period; a.n_ind = h->n_ind;
    a.s0 = s0; a.u_nom = h->d_u_nom; a.u_prev = h->d_u_prev;
    a.stdev = c.mppi_stdev;
    a.k_du2 = (float)((double)c.mppi_cc_weight * (double)c.mppi_coef_du2);
    a.k_udu = (float)((double)c.mppi_cc_weight * (double)c.mppi_R);
    a.k_uu = (float)((double)c.mppi_cc_weight * (double)c.mppi_half_R);
    a.neg_inv_lbd = c.mppi_neg_inv_LBD;
    for (int i = 0; i < kEnvMaxControls; ++i) { a.lo[i] = h->lo_v[i]; a.hi[i] = h->hi_v[i]; }
    a.env = h->env_p; a.J = h->d_J; a.log_traj = h->d_log_traj_soa; a.log_Q = h->d_log_Q_soa;
    a.u_out = u_out_dev; a.freeze_prev = c.freeze_previous_input;
    h->launches += 2;
    {
      KernelTimer kt(h);
      CU(launch_env_mppi(h->env, c.logging != 0, a, h->stream));
    }
    h->last_kernel = std::string("env_mppi_rollout_kernel<DubinsEnv,") + (c.logging ? "1" : "0") + ">" + (a.noise.inj ? " [injected noise]" : " [philox]");
    return CTK_OK;
  }
  // CEM: optimizer_cem_tf.py:83-111
  const int iters = cem_tick_iters(h);
  if (iters < 1) return fail(CTK_EINVAL, "CEM iteration count < 1");
  h->elite_log_rows = 0;
  h->cem_iters = iters;
  for (int it = 0; it < iters; ++it) {
    EnvCemArgs a{};
    int rcn = make_noise(h, STREAM_CEM | ((uint32_t)it << 8), h->H * nu, 0, (size_t)h->NG, &a.noise);
    if (rcn != CTK_OK) return rcn;
    a.N = h->N; a.off = h->off; a.H = h->H; a.s0 = s0; a.mu = h->d_mu; a.sd = h->d_sd; a.u_prev = h->d_u_prev;
    for (int i = 0; i < kEnvMaxControls; ++i) { a.lo[i] = h->lo_v[i]; a.hi[i] = h->hi_v[i]; }
    a.env = h->env_p; a.J = h->d_J; a.log_traj = h->d_log_traj_soa; a.log_Q = h->d_log_Q_soa;
    h->launches++;
    {
      KernelTimer kt(h);
      CU(launch_env_cem_rollout(h->env, c.logging != 0, a, h->stream));
    }
    h->last_kernel = std::string("env_cem_rollout_kernel<DubinsEnv,") + (c.logging ? "1" : "0") + ">" + (a.noise.inj ? " [injected noise]" : " [philox]");
    const int k = c.cem_best_k;
    int n = h->N;
    const uint64_t* kin = nullptr;
    CU(topk_levels(h->d_J, kin, n, 0, h->off, k, false, h->d_keys[0], h->d_keys[1], h->stream, h->launches));
    EnvCemRefitArgs r{};
    r.H = h->H; r.nu = nu; r.k = k; r.cnt = n; r.cand = kin; r.noise = a.noise;
    for (int i = 0; i < kEnvMaxControls; ++i) { r.lo[i] = h->lo_v[i]; r.hi[i] = h->hi_v[i]; }
    r.mu = h->d_mu; r.sd = h->d_sd; r.last = (it == iters - 1) ? 1 : 0;
    r.sd_min = c.cem_stdev_min; r.sd_init = c.cem_initial_action_stdev;
    r.u_prev = h->d_u_prev; r.u_out = u_out_dev; r.freeze_prev = c.freeze_previous_input;
    r.elite_idx_out = (h->elite_log_rows < h->elite_log_cap) ? h->d_elite_idx + (size_t)h->elite_log_rows * k : nullptr;
    h->launches++;
    CU(launch_env_cem_refit(r, h->stream));
    if (r.elite_idx_out) h->elite_log_rows++;
  }
  h->count++;
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// the tick
// ---------------------------------------------------------------------------------------------------------------

// the tcgen05 engines of ctk_mlp_tc.cuh: a pass of a block covers a fixed number of rollouts (tiles in flight x 128)
static bool tile_engine(PredKind pred) { return pred_info(pred).rollouts_per_pass > 0; }
static PredKind pred_kind(const ctk_handle* h) {
  if (h->cfg.predictor == CTK_PRED_GRU) return PredKind::Gru;
  if (h->cfg.predictor != CTK_PRED_MLP) return PredKind::Ode;
  if (h->cfg.optimizer == CTK_OPT_RPGD) return PredKind::MlpSimt;
  switch (h->cfg.mlp_engine) {
    case CTK_MLP_TCGEN05: return PredKind::MlpTc;
    case CTK_MLP_TCGEN05_BF16: return PredKind::MlpTcBf16;
    case CTK_MLP_TCGEN05_FAST: return PredKind::MlpTcFast;
    default: return PredKind::MlpSimt;
  }
}
static const char* pred_name(const ctk_handle* h) { return pred_info(pred_kind(h)).name; }  // the rollout kernel's functor (last_kernel)
static size_t pred_smem_floats(const ctk_handle* h) { return pred_info(pred_kind(h)).smem_floats(h->mlp); }

// Launch geometry of the ODE kernel: one CTA per SM, block sized so that every thread runs the same number of
// rollout groups (no partially filled last wave); the iteration count with the least padding wins.
static void mppi_ode_geometry(ctk_handle* h) {
  const ctk_config& c = h->cfg;
  h->ode_kernel = false;
  if (c.predictor != CTK_PRED_ODE || h->ode_p.intermediate_steps > 1 || h->num_sms <= 0) return;
  if (getenv("CTK_K1_GENERIC")) return;
  const long long N = h->N, sms = h->num_sms;
  // two rollouts per thread pay off once a thread runs several of them; below one full wave of single-rollout threads
  // (<= 1024 per SM) more warps hide the step latency better than more chains per warp (measured, profiles/)
  int ilp = (N <= sms * 1024) ? 1 : 2;
  if (const char* e = getenv("CTK_K1_ILP")) { const int v = atoi(e); if (v == 1 || v == 2) ilp = v; }
  int maxb = mppi_ode_max_block(ilp, c.logging != 0);
  if (const char* e = getenv("CTK_K1_BLOCK")) { const int v = atoi(e) / 32 * 32; if (v >= 32 && v <= maxb) maxb = v; }
  // shared memory: draws stash [n_ind][ilp*T] + accumulators [n_ind][T] + small fixed part, <= 200 KB
  const long long fixed = (long long)mppi_ode_smem_bytes(h->H, h->period, h->n_ind, ilp, 0);
  const long long per_thread = 4ll * h->n_ind * (ilp + 1);
  const long long tmax_smem = (200 * 1024 - fixed) / per_thread / 32 * 32;
  if (tmax_smem < 32) return;  // too many inducing points: generic kernel (regenerates the draws)
  if (maxb > tmax_smem) maxb = (int)tmax_smem;
  // Every block takes an equal contiguous share of the population, cut into units of 32 x ilp rollouts dealt round-robin to its warps
  // (ctk_kernels_mppi_ode.cuh).  Blocks of whole warp quads (warp w runs on SM sub-partition w % 4, and the kernel's duration is the
  // instruction count of the busiest sub-partition); as many warps as there are units, up to the register / shared-memory bound.
  // Small populations: a block narrower than 4 warps leaves the tick finish (block 0 polls and combines gridDim x (n_ind+2)
  // records, then updates u_nom[H]) to one or two warps while the rollout phase gains nothing from spreading single warps over
  // more SMs -- measured at N = 2000: rollouts 5.5 us, finish 19 us with 63 blocks x 32 threads.
  int min_T = 128;
  if (const char* e = getenv("CTK_K1_MIN_BLOCK")) { const int v = atoi(e) / 32 * 32; if (v >= 32) min_T = v; }
  if (min_T > maxb) min_T = maxb;
  const long long unit = 32ll * ilp;
  long long G = std::min<long long>(sms, (N + (long long)min_T * ilp - 1) / ((long long)min_T * ilp));
  if (G < 1) G = 1;
  const long long per_block = (N + G - 1) / G;                   // rollouts of the largest share
  const long long U = (per_block + unit - 1) / unit;             // its units
  const long long Wmax = maxb / 32 >= 1 ? maxb / 32 : 1;
  const long long rounds = (U + Wmax - 1) / Wmax;                // units per warp (at most)
  long long W = (U + rounds - 1) / rounds;                       // as few warps as that many rounds need: equal loads
  if (W * 32 < min_T) W = min_T / 32;
  if (W % 4 != 0 && (W + 3) / 4 * 4 * 32 <= maxb) W = (W + 3) / 4 * 4;
  h->ode_ilp = ilp;
  h->ode_block = (int)(W * 32);
  h->ode_grid = (int)G;
  // the finisher's reduced share (ctk_kernels_mppi_ode.cuh) only when every SM carries a block of at least 8 warps
  double share = 0.75;
  if (const char* e = getenv("CTK_K1_FINISHER_SHARE")) { const double v = atof(e); if (v >= 0.1 && v <= 1.0) share = v; }
  h->ode_fshare16 = (G == sms && h->ode_block >= 256) ? (int)(share * 16.0 + 0.5) : 16;
  if (h->ode_fshare16 < 1) h->ode_fshare16 = 1;
  const int best_T = h->ode_block;
  h->ode_period_t = (h->period == 10) ? 10 : 0;
  if (getenv("CTK_K1_NO_UNROLL")) h->ode_period_t = 0;
  h->ode_smem = mppi_ode_smem_bytes(h->H, h->period, h->n_ind, ilp, best_T);
  h->ode_kernel = true;
}

// s_dev == nullptr: the state sits in h_pin[0..5] (host caller) and travels inside the kernel parameters
static S0 make_s0(const ctk_handle* h, const float* s_dev) {
  S0 s{};
  s.p = s_dev;
  if (s_dev == nullptr) for (int i = 0; i < 6; ++i) s.v[i] = h->h_pin[i];
  return s;
}

static int make_fuse(ctk_handle* h, int mode, float* u_out_dev, MppiFuse* out) {
  MppiFuse f{};
  f.mode = mode;
  f.world = 1; f.rank = 0; f.seq = 0;
  if (mode != 0) next_seq(h->xseq);  // every shard ticks in lock step: the same sequence everywhere
  f.seq = h->xseq;
  f.record_out = h->d_record;
  f.mbox_local = h->d_mbox;
  f.handover = h->d_mbox + mbox_handover_offset(h->n_ind);
  f.publish_handover = h->chain_next ? 1 : 0;  // only a following chained tick reads it
  h->chain_next = false;
  {
    static const int hops_env = getenv("CTK_EXCHANGE_HOPS") ? atoi(getenv("CTK_EXCHANGE_HOPS")) : 0;
    f.hops = (hops_env == 1 || hops_env == 2) ? hops_env : 2;  // measured at 8 GPUs (profiles/): two hops 32.0 us per chained tick, one hop 33.4
  }
  f.trace = h->d_trace ? h->d_trace + (size_t)(h->xseq & 3u) * CTK_MBOX_BLOCKS * 8 : nullptr;
  f.chained = (mode == 2 && h->chain_hint && h->ode_kernel && h->xseq > 1) ? 1 : 0;
  h->chain_hint = false;
  for (int r = 0; r < CTK_MAX_PEERS; ++r) f.mbox_peer[r] = h->mbox_peer[r];
  f.u_nom = h->d_u_nom; f.u_prev = h->d_u_prev; f.u_out = u_out_dev; f.freeze_prev = h->cfg.freeze_previous_input;
  if (mode == 2) f.host = h->mirror;
  if (mode == 2 && h->xworld > 1) { f.world = h->xworld; f.rank = h->xrank; }
  *out = f;
  return CTK_OK;
}

// predictor.update(s, Q0 = new u_nom[0]) of a recurrent predictor (reference optimizer_mppi.py:192,195-197), after the tick's u_nom update
static int rnn_update(ctk_handle* h, const float* s_dev) {
  if (h->cfg.predictor != CTK_PRED_GRU) return CTK_OK;
  h->launches++;
  CU(launch_gru_update(make_s0(h, s_dev), h->d_u_nom, h->mlp, h->d_rnn_h, h->stream));
  return CTK_OK;
}

static MppiOdeArgs mppi_ode_args(const ctk_handle* h, const S0& s0, const NoiseSrc& ns, const MppiFuse& fuse) {
  MppiOdeArgs a{};
  a.N = h->N; a.off = h->off; a.H = h->H; a.period = h->period; a.n_ind = h->n_ind;
  a.fshare16 = h->ode_fshare16;
  a.per16 = (double)h->N / (double)(h->ode_fshare16 + 16 * (h->ode_grid - 1));
  a.trace = h->d_trace;
  a.s0 = s0; a.u_nom = h->d_u_nom; a.u_prev = h->d_u_prev; a.noise = ns; a.k = h->ode_hot;
  a.J = h->d_J; a.partials = h->d_partials; a.log_traj_soa = h->d_log_traj_soa; a.log_Q_soa = h->d_log_Q_soa;
  a.fuse = fuse;
  return a;
}

// mode 1: rollouts + shard record (staged exchange follows)   mode 2: whole tick incl. cross-GPU exchange and u_nom update
static int mppi_local(ctk_handle* h, const float* s_dev, int mode, float* u_out_dev) {
  NoiseSrc ns{};
  int rcn = make_noise(h, STREAM_MPPI, h->n_ind, 0, (size_t)h->NG, &ns);
  if (rcn != CTK_OK) return rcn;
  const ctk_config& c = h->cfg;
  const bool log = c.logging != 0;
  MppiFuse fuse{};
  make_fuse(h, mode, u_out_dev, &fuse);
  if (h->ode_kernel) {
    const MppiOdeArgs a = mppi_ode_args(h, make_s0(h, s_dev), ns, fuse);
    h->launches++;
    KernelTimer kt(h);
    const char* tail = "";
    cudaError_t e = launch_mppi_ode(h->cost.kind, log, h->ode_period_t, h->ode_ilp, h->ode_grid, h->ode_block, h->ode_smem, h->stream, a, &tail);
    h->last_kernel = "mppi_ode_kernel<" + std::to_string(h->cost.kind) + tail;
    if (e != cudaSuccess) return fail(CTK_ECUDA, std::string("mppi_ode_kernel: ") + cudaGetErrorString(e));
    return CTK_OK;
  }
  MppiArgs a{};
  a.N = h->N; a.off = h->off; a.H = h->H; a.period = h->period; a.n_ind = h->n_ind;
  a.s0 = make_s0(h, s_dev); a.u_nom = h->d_u_nom; a.u_prev = h->d_u_prev; a.noise = ns;
  a.stdev = c.mppi_stdev; a.lo = c.action_low; a.hi = c.action_high;
  // :154-155 constants pre-multiplied by cc_weight (k_du2, k_udu live in d_kx); the 0.5 R u^2 term shares u^2 with the
  // cost's own cc term (k_cc)
  a.k_du2 = 0.f; a.k_udu = 0.f;
  a.k_uu = (float)((double)c.mppi_cc_weight * (double)c.mppi_half_R);
  a.neg_inv_lbd = c.mppi_neg_inv_LBD;
  a.stash = h->mppi_stash;
  a.uk.k_dd = h->cost.k_dd; a.uk.k_bar = h->cost.k_bar; a.uk.k_ep = h->cost.k_ep; a.uk.k_cc = h->cost.k_cc + a.k_uu;
  a.uk.k_ccrc = h->cost.k_ccrc;
  a.uk.k_du2 = (float)((double)c.mppi_cc_weight * (double)c.mppi_coef_du2);
  a.uk.k_udu = (float)((double)c.mppi_cc_weight * (double)c.mppi_R);
  a.uk.cU = h->fwd.cU; a.uk.kTm = h->fwd.kTm; a.uk.h = h->fwd.h; a.uk.hk = h->fwd.hk; a.uk.K1p = h->fwd.K1p;
  a.kc = h->d_kc; a.kx = h->d_kx; a.mlp = h->mlp;
  a.J = h->d_J; a.partials = h->d_partials;
  a.log_traj_soa = h->d_log_traj_soa; a.log_Q_soa = h->d_log_Q_soa;
  a.fuse = fuse;
  const size_t smem = sizeof(float) * ((size_t)((h->H + 1) & ~1) + 2 * h->period + 32 + 42 * (h->n_ind + 1) + 16 +
                                       (h->mppi_stash ? (size_t)h->n_ind * h->mppi_rpb : 0) + (size_t)h->n_ind * h->mppi_rpb +
                                       pred_smem_floats(h));
  h->launches++;
  KernelTimer kt(h);
  if (tile_engine(pred_kind(h)) && h->mlp.tc_blob == nullptr) return fail(CTK_ESTATE, "tcgen05 MLP engine without weights");
  cudaError_t e = launch_mppi_rollout(pred_kind(h), h->cost.kind, log, h->mppi_grid, h->mppi_block, smem,
                                      h->stream, a);
  h->last_kernel = std::string("mppi_rollout_kernel<") + pred_name(h) + "," +
                   std::to_string(h->cost.kind) + "," + (log ? "1" : "0") + ">" + (ns.inj ? " [injected noise]" : " [philox]");
  if (e != cudaSuccess) return fail(CTK_ECUDA, std::string("mppi_rollout_kernel: ") + cudaGetErrorString(e));
  h->step_s = s_dev;
  if (mode == 2) return rnn_update(h, s_dev);
  return CTK_OK;
}

static int mppi_finish(ctk_handle* h, const float* gathered, int G, float* u_out_dev) {
  const ctk_config& c = h->cfg;
  MppiFinalize fin{};
  fin.enable = 1;
  fin.H = h->H; fin.period = h->period; fin.n_ind = h->n_ind; fin.stdev = c.mppi_stdev; fin.lo = c.action_low; fin.hi = c.action_high;
  fin.neg_inv_lbd = c.mppi_neg_inv_LBD; fin.u_nom = h->d_u_nom; fin.u_prev = h->d_u_prev; fin.u_out = u_out_dev;
  fin.freeze_prev = c.freeze_previous_input;
  h->launches++;
  CU(launch_mppi_combine(gathered, G, h->n_ind, c.mppi_neg_inv_LBD, nullptr, fin, h->stream));
  return rnn_update(h, h->step_s);
}

// The whole CEM tick in one persistent launch, when the population fits one resident grid and is not sharded
struct CemTickGeom { int G, k2, runs_pad, big_floats, rb; size_t smem; };
static bool cem_tick_geometry(const ctk_handle* h, CemTickGeom* g) {
  const ctk_config& c = h->cfg;
  int RB = cem_tick_rollouts_per_block();
  if (const char* e = getenv("CTK_CEM_RB")) { const int v = atoi(e); if (v == 32 || v == 64 || v == 128 || v == 256 || v == 512) RB = v; }
  g->rb = RB;
  g->G = (h->N + RB - 1) / RB;
  g->k2 = 32;
  while (g->k2 < c.cem_best_k) g->k2 <<= 1;
  g->runs_pad = 1;
  while (g->runs_pad < g->G) g->runs_pad <<= 1;
  const long long run_floats = 2ll * g->runs_pad * g->k2;  // uint64 keys
  g->big_floats = (int)std::max<long long>(8192, run_floats);
  g->smem = sizeof(float) * ((size_t)((2 * h->H + 3) & ~3) + (size_t)g->big_floats);
  return run_floats <= 40 * 1024;  // <= 160 KB of candidate runs
}
static bool cem_persistent_ok(ctk_handle* h) {
  const ctk_config& c = h->cfg;
  if (!(c.optimizer == CTK_OPT_CEM && h->ode_kernel && h->N == h->NG && h->off == 0 && h->xworld == 1 && c.cem_best_k <= 128 &&
        h->H <= 512 && h->num_sms > 0 && h->N <= 65535 && !h->cem_coop_refused && getenv("CTK_CEM_MULTI_LAUNCH") == nullptr))
    return false;
  CemTickGeom g;
  if (!cem_tick_geometry(h, &g)) return false;
  if (h->cem_tick_per_sm < 0) h->cem_tick_per_sm = cem_tick_blocks_per_sm(h->cost.kind, c.logging != 0, g.smem);
  return h->cem_tick_per_sm >= 1 && g.G <= h->cem_tick_per_sm * h->num_sms;  // every block must be resident: blocks wait for each other
}
// random shooting (cem_uniform_actions): Q = z (high - low) + low with z ~ U[0,1)  ==  the CEM sample clip(mu + z sd) with
// mu = low, sd = high - low
static int upload_uniform_dist(ctk_handle* h) {
  const ctk_config& c = h->cfg;
  std::vector<float> mu((size_t)h->H, c.action_low), sd((size_t)h->H, c.action_high - c.action_low);
  CU(cudaMemcpyAsync(h->d_mu, mu.data(), sizeof(float) * h->H, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->d_sd, sd.data(), sizeof(float) * h->H, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));  // mu / sd are stack-lifetime host vectors
  return CTK_OK;
}
// returns 1 if the runtime refused the cooperative launch (grid not co-resident right now): nothing was consumed, the caller runs
// the multi-launch path
static int cem_tick_persistent(ctk_handle* h, const float* s_dev, float* u_out_dev) {
  const ctk_config& c = h->cfg;
  const size_t inj_pos0 = h->inj_pos;
  const unsigned int cem_seq0 = h->cem_seq;
  const int iters = cem_tick_iters(h);
  if (iters < 1) return fail(CTK_EINVAL, "CEM iteration count < 1");
  const int uni = c.cem_uniform_actions ? 1 : 0;
  if (uni) {
    const int rc = upload_uniform_dist(h);
    if (rc != CTK_OK) return rc;
  }
  CemTickArgs a{};
  for (int it = 0; it < iters; ++it) {  // one noise block per outer iteration: consecutive in the injected queue
    NoiseSrc ns{};
    int rcn = make_noise(h, STREAM_CEM | ((uint32_t)it << 8), h->H, uni, (size_t)h->NG, &ns);
    if (rcn != CTK_OK) return rcn;
    if (it == 0) a.noise = ns;
    else if ((ns.inj != nullptr) != (a.noise.inj != nullptr))  // the kernel reads iteration it at inj + it * inj_stride
      return fail(CTK_EINVAL, "injected-noise queue ran out between the outer iterations of a CEM tick: queue all iterations or none");
    h->cem_noise = ns;
  }
  a.inj_stride = (size_t)h->NG * h->H;
  a.N = h->N; a.off = h->off; a.H = h->H; a.k = c.cem_best_k; a.iters = iters;
  a.s0 = make_s0(h, s_dev); a.mu = h->d_mu; a.sd = h->d_sd; a.u_prev = h->d_u_prev; a.u_out = u_out_dev;
  a.freeze_prev = c.freeze_previous_input; a.hot = h->ode_hot; a.J = h->d_J;
  a.log_traj_soa = h->d_log_traj_soa; a.log_Q_soa = h->d_log_Q_soa;
  a.cand = h->d_cem_cand; a.dist = h->d_cem_dist;
  if (h->cem_seq > 0xffff0000u) h->cem_seq = 0;
  a.seq0 = h->cem_seq + 1;
  h->cem_seq += (unsigned int)iters;
  a.sd_min = c.cem_stdev_min; a.sd_init = c.cem_initial_action_stdev;
  a.elite_idx_out = h->d_elite_idx; a.elite_cap = h->elite_log_cap;
  a.host = h->mirror;
  a.trace = h->d_trace;
  h->elite_log_rows = iters < h->elite_log_cap ? iters : h->elite_log_cap;
  h->cem_iters = iters;
  CemTickGeom g;
  cem_tick_geometry(h, &g);
  a.k2 = g.k2; a.runs_pad = g.runs_pad; a.q_cap = g.big_floats; a.rb = g.rb;
  h->launches++;
  cudaError_t e;
  {
    KernelTimer kt(h);
    e = launch_cem_tick(h->cost.kind, c.logging != 0, g.G, g.smem, h->stream, a);
    h->last_kernel = "cem_tick_kernel<" + std::to_string(h->cost.kind) + "," + (c.logging ? "1" : "0") + "," +
                     ((a.noise.inj == nullptr && !a.noise.uniform) ? "1" : "0") + ">";
  }
  if (e == cudaErrorCooperativeLaunchTooLarge || e == cudaErrorLaunchOutOfResources) {
    cudaGetLastError();
    h->cem_coop_refused = true;
    h->inj_pos = inj_pos0; h->cem_seq = cem_seq0; h->launches--;
    return 1;
  }
  if (e != cudaSuccess) return fail(CTK_ECUDA, std::string("cem_tick_kernel: ") + cudaGetErrorString(e));
  h->cem_it = 0;
  h->count++;
  return CTK_OK;
}

// CEM: rollouts + local top-k candidates.  to_k: reduce to exactly k keys (sharded exchange record).
static int cem_local(ctk_handle* h, const float* s_dev, bool to_k) {
  const ctk_config& c = h->cfg;
  if (h->cem_it == 0) {
    h->cem_iters = cem_tick_iters(h);
    if (h->cem_iters < 1) return fail(CTK_EINVAL, "CEM iteration count < 1");
    h->elite_log_rows = 0;
  }
  const int uni = c.cem_uniform_actions ? 1 : 0;
  if (uni && h->cem_it == 0) {
    const int rc = upload_uniform_dist(h);
    if (rc != CTK_OK) return rc;
  }
  NoiseSrc ns{};
  int rcn = make_noise(h, STREAM_CEM | ((uint32_t)h->cem_it << 8), h->H, uni, (size_t)h->NG, &ns);
  if (rcn != CTK_OK) return rcn;
  h->cem_noise = ns;
  h->launches++;
  cudaError_t e;
  int fused_cand = 0;  // > 0: the rollout kernel already left that many level-0 candidate keys in d_keys[0]
  if (h->ode_kernel) {
    CemOdeArgs a{};
    a.N = h->N; a.off = h->off; a.H = h->H; a.s0 = make_s0(h, s_dev); a.mu = h->d_mu; a.sd = h->d_sd; a.u_prev = h->d_u_prev; a.noise = ns;
    a.k = h->ode_hot; a.J = h->d_J; a.log_traj_soa = h->d_log_traj_soa; a.log_Q_soa = h->d_log_Q_soa;
    int nb = h->nblocks;
    if (c.cem_best_k <= 128 && getenv("CTK_CEM_NO_FUSED_TOPK") == nullptr) {  // level 0 of the top-k inside the rollout kernel
      nb = (h->N + 255) / 256;
      a.cand_out = h->d_keys[0]; a.kk = c.cem_best_k;
      fused_cand = nb * c.cem_best_k;
    }
    KernelTimer kt(h);
    e = launch_cem_ode(h->cost.kind, c.logging != 0, nb, sizeof(float) * 2 * (size_t)h->H, h->stream, a);
    h->last_kernel = "cem_ode_kernel<" + std::to_string(h->cost.kind) + "," + (c.logging ? "1" : "0") + ">" + (ns.inj ? " [injected noise]" : " [philox]");
  } else {
    CemArgs a{};
    a.N = h->N; a.off = h->off; a.H = h->H; a.s0 = make_s0(h, s_dev); a.mu = h->d_mu; a.sd = h->d_sd; a.u_prev = h->d_u_prev; a.noise = ns;
    a.lo = c.action_low; a.hi = c.action_high; a.kc = h->d_kc; a.mlp = h->mlp; a.J = h->d_J;
    a.log_traj_soa = h->d_log_traj_soa; a.log_Q_soa = h->d_log_Q_soa;
    const size_t smem = sizeof(float) * (2 * (size_t)h->H + pred_smem_floats(h));
    KernelTimer kt(h);
    if (tile_engine(pred_kind(h)) && h->mlp.tc_blob == nullptr) return fail(CTK_ESTATE, "tcgen05 MLP engine without weights");
    e = launch_cem_rollout(pred_kind(h), h->cost.kind, c.logging != 0, cem_rollout_grid(pred_kind(h), h->N, h->num_sms), smem, h->stream, a);
    h->last_kernel = std::string("cem_rollout_kernel<") + pred_name(h) + "," +
                     std::to_string(h->cost.kind) + "," + (c.logging ? "1" : "0") + ">" + (ns.inj ? " [injected noise]" : " [philox]");
  }
  if (e != cudaSuccess) return fail(CTK_ECUDA, std::string("cem_rollout_kernel: ") + cudaGetErrorString(e));
  int n = fused_cand > 0 ? fused_cand : h->N;
  const uint64_t* kin = fused_cand > 0 ? h->d_keys[0].get() : nullptr;
  CU(topk_levels(fused_cand > 0 ? nullptr : h->d_J.get(), kin, n, fused_cand > 0 ? 1 : 0, h->off, c.cem_best_k, to_k, h->d_keys[0], h->d_keys[1],
                 h->stream, h->launches));
  h->cem_cand = n;
  h->cem_cand_ptr = const_cast<uint64_t*>(kin);
  return CTK_OK;
}

// fused == true: `cand` holds this shard's k keys, the refit kernel exchanges them with the connected shards through the mailboxes
static int cem_finish(ctk_handle* h, const uint64_t* cand, int cnt, float* u_out_dev, bool fused = false) {
  const ctk_config& c = h->cfg;
  REQ(cnt >= c.cem_best_k && cnt <= TOPK_THREADS, "CEM candidate count must be in [k, 1024]");
  CemRefitArgs a{};
  a.world = 1; a.rank = 0;
  if (fused && h->xworld > 1) {
    REQ(cnt == c.cem_best_k, "fused CEM exchange needs exactly k local candidates");
    a.world = h->xworld; a.rank = h->xrank;
    a.seq = next_seq(h->xseq);
    a.mbox_local = h->d_mbox;
    for (int r = 0; r < CTK_MAX_PEERS; ++r) a.mbox_peer[r] = h->mbox_peer[r];
  }
  a.H = h->H; a.k = c.cem_best_k; a.cnt = cnt; a.cand = cand; a.noise = h->cem_noise; a.lo = c.action_low; a.hi = c.action_high;
  a.mu = h->d_mu; a.sd = h->d_sd; a.last = (h->cem_it == h->cem_iters - 1) ? 1 : 0;
  a.sd_min = c.cem_stdev_min; a.sd_init = c.cem_initial_action_stdev;
  a.u_prev = h->d_u_prev; a.u_out = u_out_dev; a.freeze_prev = c.freeze_previous_input;
  a.elite_idx_out = (h->elite_log_rows < h->elite_log_cap) ? h->d_elite_idx + (size_t)h->elite_log_rows * c.cem_best_k : nullptr;
  if (a.last) a.host = h->mirror;
  h->launches++;
  CU(launch_cem_refit(a, h->stream));
  if (a.elite_idx_out) h->elite_log_rows++;
  h->cem_it++;
  if (a.last) { h->cem_it = 0; h->count++; }
  return CTK_OK;
}

// Adam bias corrections of the first gradient steps of a launch (RpgdGradArgs::bc1_h ...), float64 on the host, rounded once
template <class GradArgs>
static void fill_host_adam(GradArgs& a) {
  a.n_host_adam = a.iters < 8 ? a.iters : 8;
  for (int i = 0; i < a.n_host_adam; ++i) {
    const double step = (double)(a.adam_step0 + i + 1);
    const double bc1d = 1.0 - std::pow(a.beta1, step), bc2d = 1.0 - std::pow(a.beta2, step);
    a.bc1_h[i] = (float)bc1d; a.bc2_h[i] = (float)bc2d;
    a.alpha_h[i] = (float)((double)a.lr * std::sqrt(bc2d) / bc1d);
  }
}

// Gradient step on an environment other than the CartPole (ctk_kernels_env_rpgd.cuh), population [H][nu][N]
static EnvRpgdGradArgs env_rpgd_grad_args(ctk_handle* h, const S0e& s0, int iters, float* Q, float* m, float* v, int adam_form) {
  const ctk_config& c = h->cfg;
  EnvRpgdGradArgs a{};
  a.N = h->N; a.H = h->H; a.iters = iters; a.s0 = s0; a.u_prev = h->d_u_prev;
  a.Q = Q; a.m = m; a.v = v;
  for (int i = 0; i < kEnvMaxControls; ++i) { a.lo[i] = h->lo_v[i]; a.hi[i] = h->hi_v[i]; }
  a.lr = c.rpgd_learning_rate; a.gradmax_clip = c.rpgd_gradmax_clip;
  a.beta1 = c.rpgd_beta_1; a.beta2 = c.rpgd_beta_2; a.eps = c.rpgd_epsilon; a.adam_step0 = h->adam_step; a.adam_form = adam_form;
  a.env = h->env_p; a.J = h->d_J; a.log_traj = h->d_log_traj_soa; a.log_Q = h->d_log_Q_soa;
  fill_host_adam(a);
  return a;
}
static std::string env_grad_kernel_name(const ctk_handle* h, bool fused) {
  return std::string("env_rpgd_grad_kernel<DubinsEnv,") + (h->cfg.logging ? "1" : "0") + ">" + (fused ? " [fused select]" : "");
}

// Gradient-assisted CEM tick (rpgd_gradient_mode 2: optimizer_cem_naive_grad_tf.py:90-114, 3: optimizer_cem_grad_bharadhwaj_tf.py:151-178)
// over nu columns.  The state: s_dev (or h_pin) for the CartPole's gradient kernel, s0e for another environment's.
static int gradcem_tick(ctk_handle* h, const float* s_dev, const S0e& s0e, float* u_out_dev) {
  const ctk_config& c = h->cfg;
  const bool carry = c.rpgd_gradient_mode == 3;
  const int N = h->N, H = h->H, k = c.cem_best_k, nu = h->nu;
  const int iters = carry ? cem_tick_iters(h) : c.cem_outer_it;
  const int kc = carry ? k : 0;
  auto sample = [&](int col0, int cnt, uint32_t sub) -> int {
    if (cnt <= 0) return CTK_OK;
    GradCemSampleArgs a{};
    int rcn = make_noise(h, STREAM_CEM | (sub << 8), H * nu, 0, (size_t)cnt, &a.noise);
    if (rcn != CTK_OK) return rcn;
    a.H = H; a.ld = N; a.col0 = col0; a.cnt = cnt; a.mu = h->d_mu; a.sd = h->d_sd;
    for (int i = 0; i < kEnvMaxControls; ++i) { a.lo[i] = h->lo_v[i]; a.hi[i] = h->hi_v[i]; }
    a.dst = h->d_Q[h->cur];
    h->launches++;
    CU(launch_gradcem_sample(nu, a, h->stream));
    return CTK_OK;
  };
  int rc = carry ? sample(0, k, 0) : CTK_OK;  // bharadhwaj :159 the first "elites" are plain samples
  if (rc != CTK_OK) return rc;
  h->elite_log_rows = 0;
  for (int it = 0; it < iters; ++it) {
    rc = sample(kc, N - kc, (uint32_t)it + 1);
    if (rc != CTK_OK) return rc;
    const bool last = it == iters - 1;
    if (h->env != 0) {
      const EnvRpgdGradArgs a = env_rpgd_grad_args(h, s0e, 1, h->d_Q[h->cur], h->d_m[0], h->d_v[0], carry ? 0 : 2);
      h->launches++;
      {
        KernelTimer kt(h);
        CU(launch_env_rpgd_grad(h->env, c.logging != 0, env_rpgd_smem_bytes(h->env, H), h->stream, a, nullptr));
      }
      h->last_kernel = env_grad_kernel_name(h, false);
    } else {
      RpgdGradArgs a{};
      a.N = N; a.H = H; a.iters = 1; a.s0 = make_s0(h, s_dev); a.u_prev = h->d_u_prev;
      a.Q = h->d_Q[h->cur]; a.m = h->d_m[0]; a.v = h->d_v[0];
      a.lo = c.action_low; a.hi = c.action_high; a.lr = c.rpgd_learning_rate; a.gradmax_clip = c.rpgd_gradmax_clip;
      a.beta1 = c.rpgd_beta_1; a.beta2 = c.rpgd_beta_2; a.eps = c.rpgd_epsilon; a.adam_step0 = h->adam_step;
      a.adam_form = carry ? 0 : 2;
      fill_host_adam(a);
      a.kc = h->d_kc; a.ode = h->ode; a.fwd = h->fwd; a.cost = h->cost; a.J = h->d_J; a.log_traj_soa = h->d_log_traj_soa;
      const int B = 32;
      const bool coef = sizeof(float) * (size_t)H * B * 12 <= 227 * 1024;  // coefficient tape: q, g, m, v and 8 coefficients per step
      const size_t smem = sizeof(float) * (size_t)H * B * (coef ? 12 : 8);
      if (smem > 227 * 1024) return fail(CTK_EINVAL, "mpc_horizon too large for the shared-memory tape (max 227)");
      h->launches++;
      {
        KernelTimer kt(h);
        CU(launch_rpgd_grad(h->cost.kind, c.logging != 0, coef, (N + B - 1) / B, B, smem, h->stream, a));
      }
      // Q_logged of the last population (the environment kernel writes log_Q itself)
      if (last && c.logging) CU(cudaMemcpyAsync(h->d_Q_log, h->d_Q[h->cur], sizeof(float) * N * H, cudaMemcpyDeviceToDevice, h->stream));
    }
    if (carry) h->adam_step += 1;
    GradCemRefitArgs r{};
    r.N = N; r.H = H; r.k = k; r.J = h->d_J; r.Q = h->d_Q[h->cur]; r.Q_carry = carry ? h->d_Q[h->cur ^ 1].get() : nullptr;
    r.mu = h->d_mu; r.sd = h->d_sd; r.last = last ? 1 : 0; r.u_from_mean = carry ? 0 : 1;
    r.sd_min = c.cem_stdev_min; r.sd_init = c.cem_initial_action_stdev;
    for (int i = 0; i < kEnvMaxControls; ++i) { r.lo[i] = h->lo_v[i]; r.hi[i] = h->hi_v[i]; }
    r.u_prev = h->d_u_prev; r.u_out = u_out_dev; r.freeze_prev = c.freeze_previous_input;
    r.elite_idx_out = (it < h->elite_log_cap) ? h->d_elite_idx + (size_t)it * k : nullptr;
    if (last) r.host = h->mirror;
    h->launches++;
    CU(launch_gradcem_refit(nu, r, h->stream));
    if (r.elite_idx_out) h->elite_log_rows++;
    if (carry) h->cur ^= 1;
  }
  h->count++;
  return CTK_OK;
}

static int rpgd_local(ctk_handle* h, const float* s_dev, const RpgdSelectArgs* fused_select = nullptr) {
  const ctk_config& c = h->cfg;
  if (c.rpgd_gradient_mode >= 2) { h->pending_s = s_dev; return CTK_OK; }  // the whole tick runs in rpgd_finish (needs u_out)
  const int iters = (h->count == 0) ? c.rpgd_first_iter_count : c.rpgd_outer_its;  // optimizer_rpgd.py:397-400
  RpgdGradArgs a{};
  a.N = h->N; a.H = h->H; a.iters = iters; a.s0 = make_s0(h, s_dev); a.u_prev = h->d_u_prev;
  a.Q = h->d_Q[h->cur]; a.m = h->d_m[h->cur]; a.v = h->d_v[h->cur];
  a.lo = c.action_low; a.hi = c.action_high; a.lr = c.rpgd_learning_rate; a.gradmax_clip = c.rpgd_gradmax_clip;
  a.beta1 = c.rpgd_beta_1; a.beta2 = c.rpgd_beta_2; a.eps = c.rpgd_epsilon; a.adam_step0 = h->adam_step; a.adam_form = c.rpgd_adam_form;
  a.kc = h->d_kc; a.ode = h->ode; a.fwd = h->fwd; a.cost = h->cost; a.J = h->d_J; a.log_traj_soa = h->d_log_traj_soa;
  a.trace = h->d_trace;
  fill_host_adam(a);
  const int B = 32;
  const bool coef = sizeof(float) * (size_t)h->H * B * 12 <= 227 * 1024 && getenv("CTK_RPGD_DIRECT_ADJOINT") == nullptr;
  const size_t smem = sizeof(float) * (size_t)h->H * B * (coef ? 12 : 8);
  const bool log = c.logging != 0;
  if (smem > 227 * 1024) return fail(CTK_EINVAL, "RPGD: mpc_horizon too large for the shared-memory tape (max 227)");
  h->launches++;
  {
    KernelTimer kt(h);
    CU(launch_rpgd_grad(h->cost.kind, log, coef, (h->N + B - 1) / B, B, smem, h->stream, a, coef ? fused_select : nullptr));
  }
  h->adam_step += iters;
  return CTK_OK;
}

// K8 arguments of this tick (draws the resampling noise); the caller launches K8 -- on its own or fused into K6/K7 -- and commits
static int rpgd_select_prepare(ctk_handle* h, float* u_out_dev, RpgdSelectArgs* out) {
  const ctk_config& c = h->cfg;
  const int grad_mode = c.rpgd_gradient_mode == 1 ? 1 : 0;
  const int resample = (!grad_mode && h->count % c.rpgd_resamp_per == 0) ? 1 : 0;  // optimizer_rpgd.py:449
  NoiseSrc ns{};
  if (grad_mode) {  // [N, 1, nu] uniform draws for the vacated last step (optimizer_gradient_tf.py:142-147)
    int rcn = make_noise(h, STREAM_RPGD_RESAMPLE, h->nu, 1, (size_t)h->N, &ns);
    if (rcn != CTK_OK) return rcn;
  } else if (resample && h->N - c.rpgd_keep_k > 0) {
    int rcn = make_noise(h, STREAM_RPGD_RESAMPLE, h->n_ind * h->nu, c.rpgd_distribution == CTK_DIST_UNIFORM, (size_t)(h->N - c.rpgd_keep_k), &ns);
    if (rcn != CTK_OK) return rcn;
  }
  RpgdSelectArgs a = rpgd_sample_args(h, ns);
  a.resample = resample;
  a.tail_resample = grad_mode;
  if (grad_mode) {  // the tail redraw is uniform over the action limits
    a.dist = CTK_DIST_UNIFORM;
    for (int i = 0; i < kEnvMaxControls; ++i) { a.s_min[i] = h->lo_v[i]; a.s_max[i] = h->hi_v[i]; }
  }
  a.J = h->d_J; a.Q = h->d_Q[h->cur]; a.m = h->d_m[h->cur]; a.v = h->d_v[h->cur]; a.ages = h->d_ages[h->cur];
  const int nx = h->cur ^ 1;
  a.Qn = h->d_Q[nx]; a.mn = h->d_m[nx]; a.vn = h->d_v[nx]; a.agesn = h->d_ages[nx];
  a.u_nom_out = h->d_unom_log; a.u_prev = h->d_u_prev; a.u_out = u_out_dev; a.freeze_prev = c.freeze_previous_input;
  a.best_idx_out = h->d_best_idx;
  a.host = h->mirror;
  *out = a;
  return CTK_OK;
}
static void rpgd_select_commit(ctk_handle* h) {
  h->cur ^= 1;
  h->count++;
}

static int rpgd_finish(ctk_handle* h, float* u_out_dev) {
  const ctk_config& c = h->cfg;
  if (c.rpgd_gradient_mode >= 2) return gradcem_tick(h, h->pending_s, S0e{}, u_out_dev);
  RpgdSelectArgs a{};
  int rc = rpgd_select_prepare(h, u_out_dev, &a);
  if (rc != CTK_OK) return rc;
  if (c.logging) {  // Q_logged / trajectory_ages_logged are the values BEFORE the warm-start update (:413-415)
    CU(cudaMemcpyAsync(h->d_Q_log, h->d_Q[h->cur], sizeof(float) * h->N * h->H, cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_ages_log, h->d_ages[h->cur], sizeof(float) * h->N, cudaMemcpyDeviceToDevice, h->stream));
  }
  h->launches++;
  CU(launch_rpgd_select(h->nu, a, h->stream));
  rpgd_select_commit(h);
  return CTK_OK;
}

// One RPGD tick for the host-facing / device-resident callers: a population of one block (N <= 32, C3) runs K6/K7 and K8 as ONE
// launch; larger populations, logging and the gradient-assisted CEM modes take the two-launch path
static int rpgd_tick(ctk_handle* h, const float* s_dev, float* u_out_dev) {
  const ctk_config& c = h->cfg;
  const bool fuse = c.rpgd_gradient_mode < 2 && h->N <= 32 && !c.logging && sizeof(float) * (size_t)h->H * 32 * 12 <= 220 * 1024 &&
                    getenv("CTK_RPGD_DIRECT_ADJOINT") == nullptr && getenv("CTK_RPGD_TWO_LAUNCHES") == nullptr;
  if (!fuse) {
    int rc = rpgd_local(h, s_dev);
    return rc == CTK_OK ? rpgd_finish(h, u_out_dev) : rc;
  }
  RpgdSelectArgs sel{};
  int rc = rpgd_select_prepare(h, u_out_dev, &sel);
  if (rc != CTK_OK) return rc;
  rc = rpgd_local(h, s_dev, &sel);
  if (rc != CTK_OK) return rc;
  rpgd_select_commit(h);
  return CTK_OK;
}

// RPGD / gradient-tf on an environment other than the CartPole: one launch (gradient steps + fused K8) for a population of one block
// with logging off, else two
static int env_rpgd_tick(ctk_handle* h, const S0e& s0, float* u_out_dev) {
  const ctk_config& c = h->cfg;
  if (c.rpgd_gradient_mode >= 2) return gradcem_tick(h, nullptr, s0, u_out_dev);
  RpgdSelectArgs sel{};
  int rc = rpgd_select_prepare(h, u_out_dev, &sel);
  if (rc != CTK_OK) return rc;
  const int iters = (h->count == 0) ? c.rpgd_first_iter_count : c.rpgd_outer_its;  // optimizer_rpgd.py:397-400
  const EnvRpgdGradArgs a = env_rpgd_grad_args(h, s0, iters, h->d_Q[h->cur], h->d_m[h->cur], h->d_v[h->cur], c.rpgd_adam_form);
  const bool fuse = h->N <= kEnvRpgdBlock && !c.logging;
  h->launches++;
  {
    KernelTimer kt(h);
    CU(launch_env_rpgd_grad(h->env, c.logging != 0, env_rpgd_smem_bytes(h->env, h->H), h->stream, a, fuse ? &sel : nullptr));
  }
  h->last_kernel = env_grad_kernel_name(h, fuse);
  h->adam_step += iters;
  if (!fuse) {
    // trajectory_ages_logged: the ages BEFORE the warm-start update (:413-415); Q_logged is written by the gradient kernel
    if (c.logging) CU(cudaMemcpyAsync(h->d_ages_log, h->d_ages[h->cur], sizeof(float) * h->N, cudaMemcpyDeviceToDevice, h->stream));
    h->launches++;
    CU(launch_rpgd_select(h->nu, sel, h->stream));
  }
  rpgd_select_commit(h);
  return CTK_OK;
}

// Preconditions of every tick entry point
static int tick_ready(ctk_handle* h) {
  if (!h->was_reset) return fail(CTK_ESTATE, "ctk_step before ctk_reset");
  CU(cudaSetDevice(h->cfg.device));
  if (h->cfg.predictor != CTK_PRED_ODE && h->mlp.blob == nullptr) return fail(CTK_ESTATE, "network predictor without weights (ctk_set_mlp_weights / ctk_set_gru_weights)");
  return CTK_OK;
}

// One whole tick, enqueued.  The state is s_dev (device) or, s_dev == nullptr, s_host: a general environment takes it from there,
// the CartPole kernels from h_pin, where the caller has put it.
static int run_tick(ctk_handle* h, const float* s_dev, const float* s_host, float* u_out_dev) {
  int rc = tick_ready(h);
  if (rc != CTK_OK) return rc;
  if (h->env != 0) return env_tick(h, make_s0e(h, s_dev, s_host), u_out_dev);
  h->tick++;
  switch (h->cfg.optimizer) {
    case CTK_OPT_MPPI:
      return mppi_local(h, s_dev, 2, u_out_dev);
    case CTK_OPT_CEM:
      rc = cem_persistent_ok(h) ? cem_tick_persistent(h, s_dev, u_out_dev) : 1;
      if (rc == 1) do {
        rc = cem_local(h, s_dev, h->xworld > 1);
        if (rc != CTK_OK) break;
        rc = cem_finish(h, h->cem_cand_ptr, h->cem_cand, u_out_dev, h->xworld > 1);
      } while (rc == CTK_OK && h->cem_it != 0);
      return rc;
    default:
      return rpgd_tick(h, s_dev, u_out_dev);
  }
}

extern "C" int ctk_step_local(ctk_handle* h, const float* s_dev) {
  REQ(h && s_dev, "null pointer");
  REQ(h->env == 0, "the staged (sharded) tick is implemented for the CartPole environment");
  int rc = tick_ready(h);
  if (rc != CTK_OK) return rc;
  switch (h->cfg.optimizer) {
    case CTK_OPT_MPPI:
      h->tick++;
      rc = mppi_local(h, s_dev, 1, nullptr);
      return rc;
    case CTK_OPT_CEM:
      if (h->cem_it == 0) h->tick++;
      rc = cem_local(h, s_dev, true);
      if (rc != CTK_OK) return rc;
      return (h->cem_it < h->cem_iters - 1) ? 1 : 0;
    default:
      h->tick++;
      return rpgd_local(h, s_dev);
  }
}

extern "C" int ctk_partials(ctk_handle* h, float** dev_ptr, size_t* n_floats) {
  REQ(h && dev_ptr && n_floats, "null pointer");
  if (h->cfg.optimizer == CTK_OPT_MPPI) { *dev_ptr = h->d_record; *n_floats = (size_t)h->n_ind + 2; }
  else if (h->cfg.optimizer == CTK_OPT_CEM) { *dev_ptr = (float*)h->cem_cand_ptr; *n_floats = 2 * (size_t)h->cfg.cem_best_k; }
  else { *dev_ptr = nullptr; *n_floats = 0; }
  return CTK_OK;
}

extern "C" int ctk_step_finish(ctk_handle* h, const float* gathered, int G, float* u_out_dev) {
  REQ(h && G >= 1, "null handle or num_shards < 1");
  CU(cudaSetDevice(h->cfg.device));
  switch (h->cfg.optimizer) {
    case CTK_OPT_MPPI:
      REQ(gathered, "null gathered records");
      return mppi_finish(h, gathered, G, u_out_dev);
    case CTK_OPT_CEM:
      REQ(gathered, "null gathered records");
      return cem_finish(h, (const uint64_t*)gathered, G * h->cfg.cem_best_k, u_out_dev);
    default:
      REQ(G == 1, "RPGD is replicas-only");
      return rpgd_finish(h, u_out_dev);
  }
}

static int state_ptr(ctk_handle* h, int which, float** p, size_t* n, bool* tmajor);
static int step_host(ctk_handle* h, const float* s_host, float* u_out_host, const float* state_dev, float* state_out_host, size_t n_state);
extern "C" int ctk_step(ctk_handle* h, const float* s_host, float* u_out_host) { return step_host(h, s_host, u_out_host, nullptr, nullptr, 0); }
// ctk_step + read-back of one [H] state array (MPPI u_nom, CEM dist_mue / stdev) in the SAME device->host copy window and
// synchronisation: the plugin's step() needs u and the warm-start sequence every tick (optimizer_mppi.py:220).
extern "C" int ctk_step_state(ctk_handle* h, const float* s_host, float* u_out_host, int which, float* state_out_host, size_t n) {
  REQ(h && state_out_host, "null pointer");
  float* p; size_t cnt; bool tm;
  int rc = state_ptr(h, which, &p, &cnt, &tm);
  if (rc != CTK_OK) return rc;
  REQ(!tm && n == cnt && cnt <= (size_t)h->H * h->nu, "ctk_step_state reads the [H, nu] state arrays only");
  return step_host(h, s_host, u_out_host, p, state_out_host, n);
}
// Wait until the kernel that finishes the tick has delivered the tagged slots [first, first + count) of the mapped result
// mirror (value | sequence number, one 8-byte store each: host_put in ctk_device.cuh).  Polling pinned host memory replaces
// cudaStreamSynchronize + the device->host copies (measured: ~15 us per step).
static int wait_host_slots(ctk_handle* h, unsigned int seq, int first, int count, float* out) {
  volatile unsigned long long* slots = reinterpret_cast<volatile unsigned long long*>(h->h_pin.get());
  const auto t0 = std::chrono::steady_clock::now();
  unsigned int spins = 0;
  for (int i = 0; i < count; ++i) {
    unsigned long long v;
    while ((unsigned int)((v = slots[first + i]) >> 32) != seq) {
#if defined(__x86_64__) || defined(__i386__)
      __builtin_ia32_pause();
#endif
      if ((++spins & 0xffu) != 0) continue;
      const double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
      // ticks up to a few milliseconds (every BASELINE config: 15 us .. 1.9 ms) are caught by the pause loop -- a nanosleep of 5 us
      // returns after 50-60 us (timer slack), which put C5's p50 at 0.240 ms for a 0.196 ms tick; only a long wait (logging: tens of
      // ms) gives the core away between polls
      if (el > 3e-3) { struct timespec ts = {0, 50000}; nanosleep(&ts, nullptr); }
      if (el < 0.05) continue;
      const cudaError_t e = cudaStreamQuery(h->stream);  // a faulted or finished stream will never publish
      if (e == cudaSuccess) {
        if ((unsigned int)(slots[first + i] >> 32) == seq) continue;
        return fail(CTK_ECUDA, "tick kernels finished without publishing their result to the host mirror");
      }
      if (e != cudaErrorNotReady) return fail(CTK_ECUDA, std::string("tick failed on the device: ") + cudaGetErrorString(e));
      if (el > 60.0) return fail(CTK_ECUDA, "tick did not finish within 60 s");
    }
    const unsigned int bits = (unsigned int)(v & 0xffffffffull);
    memcpy(out + i, &bits, sizeof(float));
  }
  return CTK_OK;
}

// Host-facing tick.  The state travels inside the kernel parameters (S0), the result comes back through the mapped host mirror
// written by the tick's last kernel: no cudaMemcpy and no stream synchronisation on this path.
static int step_host(ctk_handle* h, const float* s_host, float* u_out_host, const float* state_dev, float* state_out_host, size_t n_state) {
  REQ(h && s_host && u_out_host, "null pointer");
  if (h->env != 0) {  // general environments: the launch sequence, then ONE device->host copy of u (and the requested state array)
    int rc = run_tick(h, nullptr, s_host, h->d_u_out);
    if (rc != CTK_OK) return rc;
    CU(cudaMemcpyAsync(u_out_host, h->d_u_out, sizeof(float) * h->nu, cudaMemcpyDeviceToHost, h->stream));
    if (state_dev) CU(cudaMemcpyAsync(state_out_host, state_dev, n_state * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return CTK_OK;
  }
  memcpy(h->h_pin, s_host, sizeof(float) * 6);
  // the mirror carries one [H] array: MPPI's u_nom / RPGD's best sequence; any other state array takes the copy path below
  const bool state_in_mirror = state_dev != nullptr && h->cfg.rpgd_gradient_mode < 2 &&
                               ((h->cfg.optimizer == CTK_OPT_MPPI && state_dev == h->d_u_nom) ||
                                (h->cfg.optimizer == CTK_OPT_RPGD && state_dev == h->d_unom_log));
  h->mirror = HostMirror{h->d_pin, next_seq(h->hseq)};
  int rc = run_tick(h, nullptr, s_host, h->d_u_out);
  h->mirror = HostMirror{nullptr, 0};
  if (rc != CTK_OK) return rc;
  float us[2];  // u, status
  rc = wait_host_slots(h, h->hseq, 4, 2, us);
  if (rc != CTK_OK) return rc;
  u_out_host[0] = us[0];
  if (state_dev) {
    if (state_in_mirror) {
      rc = wait_host_slots(h, h->hseq, 8, (int)n_state, state_out_host);
      if (rc != CTK_OK) return rc;
    } else {
      CU(cudaMemcpyAsync(state_out_host, state_dev, n_state * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
      CU(cudaStreamSynchronize(h->stream));
    }
  }
  if (us[1] != 0.0f) {
    if (h->cfg.optimizer == CTK_OPT_CEM)
      return fail(CTK_ECUDA, "persistent CEM tick: a block of the grid did not publish its candidates / the distribution within 2 s "
                             "(grid not co-resident? another kernel holding SM slots); set CTK_CEM_MULTI_LAUNCH=1 to use the multi-launch path");
    return fail(CTK_ECUDA, h->xworld > 1 ? "cross-GPU exchange timed out: a block record of this grid or of a peer shard did not arrive within 2 s"
                                         : "tick finish timed out: a block of this GPU's grid did not publish its softmin record within 2 s");
  }
  return CTK_OK;
}

// Asynchronous, device-resident tick (no host copies, no synchronisation): with a connected exchange every shard
// calls this once per tick and ends up with the same u_nom / u.
extern "C" int ctk_step_device(ctk_handle* h, const float* s_dev, float* u_out_dev) {
  REQ(h && s_dev, "null pointer");
  REQ(h->cfg.optimizer != CTK_OPT_RPGD || h->xworld == 1, "RPGD is replicas-only (no cross-GPU exchange)");
  return run_tick(h, s_dev, nullptr, u_out_dev ? u_out_dev : h->d_u_out.get());  // general environments: u_out_dev [nu]
}

// n ticks back to back on the handle's stream: tick i reads its state from s_dev + i * s_stride (device memory) and writes
// [u, status] to u_out_dev + i * u_stride.  One C call enqueues the whole chain, so consecutive ticks overlap through programmatic
// dependent launch (the next tick's noise generation runs underneath the previous tick's finish / exchange / launch gap).
extern "C" int ctk_step_device_n(ctk_handle* h, const float* s_dev, size_t s_stride, float* u_out_dev, size_t u_stride, int n) {
  REQ(h && s_dev && n >= 0, "null pointer or negative tick count");
  static const bool handover = getenv("CTK_NO_HANDOVER") == nullptr;
  for (int i = 0; i < n; ++i) {
    // ticks 1.. of the chain: nothing but this handle's previous tick precedes them on the stream, and the caller's states were
    // complete before tick 0 was launched, so they may take u_nom from the previous finisher's tagged hand-over
    h->chain_hint = i > 0 && handover && h->cfg.optimizer == CTK_OPT_MPPI;
    h->chain_next = i + 1 < n && handover && h->cfg.optimizer == CTK_OPT_MPPI;
    int rc = ctk_step_device(h, s_dev + (size_t)i * s_stride, u_out_dev ? u_out_dev + (size_t)i * u_stride : nullptr);
    h->chain_hint = false;
    h->chain_next = false;
    if (rc != CTK_OK) return rc;
  }
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// several clients' ticks in one launch (SURVEY 8f.4)
// ---------------------------------------------------------------------------------------------------------------
extern "C" int ctk_step_batch(ctk_handle* h, const float* s_host, const int32_t* active, float* u_out_host) {
  REQ(h && s_host && u_out_host, "null pointer");
  REQ(h->cfg.optimizer == CTK_OPT_MPPI && h->ode_kernel && h->ode_ilp == 1 && !h->cfg.logging && h->xworld == 1,
      "ctk_step_batch needs an unsharded MPPI handle on the one-rollout-per-thread ODE kernel, logging off");
  if (!h->was_reset) return fail(CTK_ESTATE, "ctk_step_batch before ctk_reset");
  CU(cudaSetDevice(h->cfg.device));
  const int B = h->nclients, ns = h->cfg.num_states;
  MppiBatch b{};
  int n_active = 0;
  for (int c = 0; c < B; ++c) {
    b.active[c] = (active == nullptr || active[c] != 0) ? 1 : 0;
    if (!b.active[c]) continue;
    ++n_active;
    b.tick[c] = ++h->client_tick[c];
    for (int i = 0; i < ns && i < 8; ++i) b.s0[c][i] = s_host[(size_t)c * ns + i];
  }
  if (n_active == 0) return CTK_OK;
  h->tick++;
  NoiseSrc nsrc{};
  int rcn = make_noise(h, STREAM_MPPI, h->n_ind, 0, (size_t)h->NG, &nsrc);
  if (rcn != CTK_OK) return rcn;
  REQ(nsrc.inj == nullptr, "ctk_step_batch draws its noise in-kernel (clear the injected-noise queue)");
  MppiFuse fuse{};
  make_fuse(h, 2, h->d_u_out, &fuse);
  fuse.host = HostMirror{nullptr, 0};
  fuse.handover = nullptr;  // (no chained tick follows a batch launch)
  MppiOdeArgs a = mppi_ode_args(h, S0{}, nsrc, fuse);  // logging is off: no log buffers
  a.trace = nullptr;
  b.stride_unom = (size_t)h->H; b.stride_J = (size_t)h->N; b.stride_partials = h->partials_stride;
  b.stride_record = (size_t)h->n_ind + 2; b.stride_mbox = h->mbox_stride;
  h->launches++;
  cudaError_t e;
  {
    KernelTimer kt(h);
    e = launch_mppi_ode_batch(h->cost.kind, h->ode_period_t, h->ode_grid, B, h->ode_block, h->ode_smem, h->stream, a, b);
  }
  h->last_kernel = "mppi_ode_batch_kernel<" + std::to_string(h->cost.kind) + "," + std::to_string(h->ode_period_t) + ",1024> x " + std::to_string(n_active) + " clients";
  if (e != cudaSuccess) return fail(CTK_ECUDA, std::string("mppi_ode_batch_kernel: ") + cudaGetErrorString(e));
  CU(cudaMemcpyAsync(h->h_batch ? h->h_batch : h->h_pin + 8, h->d_u_out, 2 * (size_t)B * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  const float* res = h->h_batch ? h->h_batch : h->h_pin + 8;
  for (int c = 0; c < B; ++c) {
    if (!b.active[c]) continue;
    if (res[2 * c + 1] != 0.0f) return fail(CTK_ECUDA, "tick finish timed out: a block of client " + std::to_string(c) + "'s grid did not publish its softmin record within 2 s");
    u_out_host[c] = res[2 * c];
  }
  return CTK_OK;
}

extern "C" int ctk_reset_client(ctk_handle* h, int client) {
  REQ(h && client >= 0 && client < h->nclients, "no such client slot");
  REQ(h->cfg.optimizer == CTK_OPT_MPPI, "multi-client handles are MPPI handles");
  CU(cudaSetDevice(h->cfg.device));
  const std::vector<float> tmp = mid_range(h, (size_t)h->H);
  CU(cudaMemcpyAsync(h->d_u_nom + (size_t)client * h->H, tmp.data(), sizeof(float) * h->H, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(h->d_u_prev + client, 0, sizeof(float), h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->client_tick[client] = 0;
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// fused cross-GPU exchange: mailboxes in peer memory (one process per GPU -> CUDA IPC; one process -> peer access)
// ---------------------------------------------------------------------------------------------------------------
extern "C" int ctk_exchange_export(ctk_handle* h, void* ipc_handle_out64) {
  REQ(h && ipc_handle_out64, "null pointer");
  REQ(h->env == 0, "the cross-GPU exchange is implemented for the CartPole environment");
  REQ(h->d_mbox != nullptr, "this optimizer has no exchange mailbox (RPGD is replicas-only)");
  CU(cudaSetDevice(h->cfg.device));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaIpcMemHandle_t hd;
  CU(cudaIpcGetMemHandle(&hd, h->d_mbox));
  memcpy(ipc_handle_out64, &hd, sizeof(hd));
  return CTK_OK;
}
static int exchange_reset(ctk_handle* h, int rank, int world) {
  REQ(world >= 1 && world <= CTK_MAX_PEERS && rank >= 0 && rank < world, "need 0 <= rank < world <= 8");
  REQ(h->cfg.optimizer != CTK_OPT_CEM || (long long)world * h->cfg.cem_best_k <= TOPK_THREADS, "sharded CEM: world x cem_best_k must be <= 1024");
  CU(cudaStreamSynchronize(h->stream));
  h->close_peers();
  h->xworld = world; h->xrank = rank; h->xseq = 0;
  h->bseq = 0;
  CU(cudaMemset(h->d_mbox, 0, sizeof(unsigned long long) * (h->cfg.optimizer == CTK_OPT_CEM ? cem_mbox_slots() : mbox_total_slots(h->n_ind, h->H))));
  return CTK_OK;
}
extern "C" int ctk_exchange_connect(ctk_handle* h, int rank, int world, const void* ipc_handles) {
  REQ(h && ipc_handles, "null pointer");
  REQ(h->d_mbox != nullptr, "this optimizer has no exchange mailbox (RPGD is replicas-only)");
  CU(cudaSetDevice(h->cfg.device));
  int rc = exchange_reset(h, rank, world);
  if (rc != CTK_OK) return rc;
  for (int r = 0; r < world; ++r) {
    if (r == rank) { h->mbox_peer[r] = h->d_mbox; continue; }
    cudaIpcMemHandle_t hd;
    memcpy(&hd, (const char*)ipc_handles + (size_t)r * sizeof(hd), sizeof(hd));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      h->xworld = 1; h->xrank = 0;
      return fail(CTK_ECUDA, std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(r) + "): " + cudaGetErrorString(e));
    }
    h->mbox_peer[r] = (unsigned long long*)p;
    h->mbox_ipc[r] = true;
  }
  return CTK_OK;
}
extern "C" int ctk_exchange_barrier(ctk_handle* h) {
  REQ(h, "null handle");
  REQ(h->d_mbox != nullptr, "this optimizer has no exchange mailbox");
  if (h->xworld <= 1) return CTK_OK;
  CU(cudaSetDevice(h->cfg.device));
  MppiFuse f{};
  f.world = h->xworld; f.rank = h->xrank;
  f.seq = next_seq(h->bseq);
  f.mbox_local = h->d_mbox;
  for (int r = 0; r < CTK_MAX_PEERS; ++r) f.mbox_peer[r] = h->mbox_peer[r];
  h->launches++;
  CU(launch_exchange_barrier(f, h->cfg.optimizer == CTK_OPT_CEM ? cem_mbox_slots() - 2 * CTK_MAX_PEERS : mbox_barrier_offset(h->n_ind), h->stream));
  return CTK_OK;
}
extern "C" int ctk_exchange_mailbox(ctk_handle* h, void** dev_ptr) {
  REQ(h && dev_ptr, "null pointer");
  *dev_ptr = h->d_mbox;
  return CTK_OK;
}
extern "C" int ctk_exchange_connect_ptrs(ctk_handle* h, int rank, int world, void* const* mailboxes, const int* devices) {
  REQ(h && mailboxes && devices, "null pointer");
  REQ(h->d_mbox != nullptr, "this optimizer has no exchange mailbox (RPGD is replicas-only)");
  CU(cudaSetDevice(h->cfg.device));
  int rc = exchange_reset(h, rank, world);
  if (rc != CTK_OK) return rc;
  for (int r = 0; r < world; ++r) {
    if (r != rank && devices[r] != h->cfg.device) {
      cudaError_t e = cudaDeviceEnablePeerAccess(devices[r], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
      if (e != cudaSuccess) { h->xworld = 1; h->xrank = 0; return fail(CTK_ECUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e)); }
    }
    h->mbox_peer[r] = (r == rank) ? h->d_mbox : (unsigned long long*)mailboxes[r];
  }
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// state / counters / logs
// ---------------------------------------------------------------------------------------------------------------
static int transpose_dev(ctk_handle* h, const float* in, float* out, int R, int C) {
  h->launches++;
  CU(launch_transpose(in, out, R, C, h->stream));
  return CTK_OK;
}

static int state_ptr(ctk_handle* h, int which, float** p, size_t* n, bool* tmajor) {
  *tmajor = false;
  const size_t H = h->H, N = h->N;
  switch (which) {
    case CTK_STATE_U_NOM: *p = (h->cfg.optimizer == CTK_OPT_RPGD) ? h->d_unom_log : h->d_u_nom; *n = H * (size_t)h->nclients * h->nu; break;  // RPGD: Q[best] before the shift (:426)
    case CTK_STATE_CEM_MU: *p = h->d_mu; *n = H * h->nu; break;
    case CTK_STATE_CEM_STD: *p = h->d_sd; *n = H * h->nu; break;
    case CTK_STATE_RPGD_Q: *p = h->d_Q[h->cur]; *n = N * H * h->nu; *tmajor = true; break;
    // gradient-assisted CEM keeps its Adam moments attached to the population ROWS (never permuted): buffer 0
    case CTK_STATE_RPGD_M: *p = h->d_m[h->cfg.rpgd_gradient_mode >= 2 ? 0 : h->cur]; *n = N * H * h->nu; *tmajor = true; break;
    case CTK_STATE_RPGD_V: *p = h->d_v[h->cfg.rpgd_gradient_mode >= 2 ? 0 : h->cur]; *n = N * H * h->nu; *tmajor = true; break;
    case CTK_STATE_RPGD_AGES: *p = h->d_ages[h->cur]; *n = N; break;
    case CTK_STATE_U_PREV: *p = h->d_u_prev; *n = (size_t)(h->nclients > h->nu ? h->nclients : h->nu); break;
    case CTK_STATE_RNN_H: *p = h->d_rnn_h; *n = 2 * (size_t)h->mlp.hidden; break;
    default: return fail(CTK_EINVAL, "unknown state id");
  }
  if (*p == nullptr) return fail(CTK_EINVAL, "state not present for this optimizer");
  return CTK_OK;
}

extern "C" int ctk_get_state(ctk_handle* h, int which, float* dst, size_t n) {
  REQ(h && dst, "null pointer");
  CU(cudaSetDevice(h->cfg.device));
  float* p; size_t cnt; bool tm;
  int rc = state_ptr(h, which, &p, &cnt, &tm);
  if (rc != CTK_OK) return rc;
  REQ(n == cnt, "size mismatch");
  if (tm) {
    Owned<float> tmp;
    CU(tmp.alloc(cnt, false));
    rc = transpose_dev(h, p, tmp, h->H * h->nu, h->N);  // [H][nu][N] -> [N][H][nu]
    if (rc != CTK_OK) return rc;
    CU(cudaMemcpyAsync(dst, tmp, cnt * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return CTK_OK;
  }
  CU(cudaMemcpyAsync(dst, p, cnt * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return CTK_OK;
}

extern "C" int ctk_set_state(ctk_handle* h, int which, const float* src, size_t n) {
  REQ(h && src, "null pointer");
  CU(cudaSetDevice(h->cfg.device));
  float* p; size_t cnt; bool tm;
  int rc = state_ptr(h, which, &p, &cnt, &tm);
  if (rc != CTK_OK) return rc;
  REQ(n == cnt, "size mismatch");
  if (tm) {
    Owned<float> tmp;
    CU(tmp.alloc(cnt, false));
    CU(cudaMemcpyAsync(tmp, src, cnt * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    rc = transpose_dev(h, tmp, p, h->N, h->H * h->nu);
    CU(cudaStreamSynchronize(h->stream));
    return rc;
  }
  CU(cudaMemcpyAsync(p, src, cnt * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return CTK_OK;
}

extern "C" int ctk_get_counter(ctk_handle* h, int which, int64_t* v) {
  REQ(h && v, "null pointer");
  switch (which) {
    case CTK_COUNTER_COUNT: *v = h->count; break;
    case CTK_COUNTER_ADAM_STEP: *v = h->adam_step; break;
    case CTK_COUNTER_TICK: *v = h->tick; break;
    default: return fail(CTK_EINVAL, "unknown counter id");
  }
  return CTK_OK;
}
extern "C" int ctk_set_counter(ctk_handle* h, int which, int64_t v) {
  REQ(h, "null pointer");
  switch (which) {
    case CTK_COUNTER_COUNT: h->count = v; break;
    case CTK_COUNTER_ADAM_STEP: h->adam_step = v; break;
    case CTK_COUNTER_TICK: h->tick = v; break;
    default: return fail(CTK_EINVAL, "unknown counter id");
  }
  return CTK_OK;
}
extern "C" int ctk_enable_kernel_timing(ctk_handle* h, int on) {
  REQ(h, "null handle");
  h->timing = on != 0;
  h->ev_used = 0;
  if (on) {  // create the events up front: cudaEventCreate inside a timed multi-GPU loop would skew the ranks
    CU(cudaSetDevice(h->cfg.device));
    while (h->ev.size() < 512) {
      cudaEvent_t e;
      CU(cudaEventCreate(&e));
      h->ev.push_back(e);
    }
  }
  return CTK_OK;
}
extern "C" int ctk_get_kernel_timing(ctk_handle* h, double* ms_sum, int64_t* n) {
  REQ(h && ms_sum && n, "null pointer");
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  double tot = 0.0;
  for (size_t i = 0; i + 1 < h->ev_used; i += 2) {
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]));
    tot += ms;
  }
  *ms_sum = tot;
  *n = (int64_t)(h->ev_used / 2);
  h->ev_used = 0;
  return CTK_OK;
}
// Diagnostics: per-block globaltimer stamps of the ODE rollout kernel's phases (kernel entry, prologue done, rollouts done,
// block reduce done, record stored, tick finished).  enable allocates the buffer; get copies [grid][8] uint64 of the last launch.
extern "C" int ctk_debug_trace(ctk_handle* h, int enable, uint64_t* out_host, size_t n_u64, int* grid_out) {
  REQ(h, "null handle");
  CU(cudaSetDevice(h->cfg.device));
  CU(cudaStreamSynchronize(h->stream));
  const size_t per = (size_t)CTK_MBOX_BLOCKS * 8, n = 4 * per;  // the last 4 launches, slot = launch sequence number & 3
  if (out_host && h->d_trace) {
    if (n_u64 >= n) {  // whole history, oldest first
      std::vector<uint64_t> tmp(n);
      CU(cudaMemcpy(tmp.data(), h->d_trace, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
      for (int i = 0; i < 4; ++i) memcpy(out_host + (size_t)i * per, tmp.data() + (size_t)((h->xseq + 1 + i) & 3u) * per, per * sizeof(uint64_t));
    } else {  // the last launch only
      REQ(n_u64 >= (size_t)(h->num_sms > 0 ? h->num_sms : 148) * 8, "trace buffer too small");
      CU(cudaMemcpy(out_host, h->d_trace + (size_t)(h->xseq & 3u) * per, (size_t)(h->num_sms > 0 ? h->num_sms : 148) * 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    }
  }
  if (grid_out) *grid_out = h->ode_grid;
  if (enable && !h->d_trace) CU(h->d_trace.alloc(n));
  if (!enable) h->d_trace.reset();
  return CTK_OK;
}
// instantiation of the last rollout-kernel launch of this handle, e.g. "mppi_ode_kernel<0,0,10,2,896,0>" (verification: the parity
// tests assert that the kernel they compared with the oracle is the one bench.py times)
extern "C" const char* ctk_last_kernel(ctk_handle* h) { return h ? h->last_kernel.c_str() : ""; }
extern "C" int ctk_get_launch_count(ctk_handle* h, int64_t* v) { REQ(h && v, "null pointer"); *v = h->launches; return CTK_OK; }

// device source (after the layout transpose, if any) and size of one log
static int log_source(ctk_handle* h, int which, const void** src_out, size_t* need_out) {
  const size_t N = h->N, H = h->H;
  const void* src = nullptr;
  size_t need = 0;
  if (h->env != 0 && (which == CTK_LOG_Q || which == CTK_LOG_ROLLOUTS)) {  // written in the reference's layout by the rollout kernel
    REQ(h->cfg.logging, "logging disabled");
    *src_out = which == CTK_LOG_Q ? h->d_log_Q_soa : h->d_log_traj_soa;
    *need_out = which == CTK_LOG_Q ? N * H * h->nu * 4 : N * (H + 1) * h->ns * 4;
    return CTK_OK;
  }
  switch (which) {
    case CTK_LOG_J: src = h->d_J; need = N * 4; break;
    case CTK_LOG_Q:
      REQ(h->cfg.logging, "logging disabled");
      if (h->cfg.optimizer == CTK_OPT_RPGD) { int rc = transpose_dev(h, h->d_Q_log, h->d_log_tmp, (int)H, (int)N); if (rc) return rc; }
      else { int rc = transpose_dev(h, h->d_log_Q_soa, h->d_log_tmp, (int)H, (int)N); if (rc) return rc; }
      src = h->d_log_tmp; need = N * H * 4; break;
    case CTK_LOG_ROLLOUTS: {
      REQ(h->cfg.logging, "logging disabled");
      int rc = transpose_dev(h, h->d_log_traj_soa, h->d_log_tmp, (int)((H + 1) * 6), (int)N);
      if (rc) return rc;
      src = h->d_log_tmp; need = N * (H + 1) * 6 * 4; break;
    }
    case CTK_LOG_ELITE_IDX:
      if (h->cfg.optimizer == CTK_OPT_CEM) { src = h->d_elite_idx; need = (size_t)h->elite_log_rows * h->cfg.cem_best_k * 4; }
      else if (h->cfg.optimizer == CTK_OPT_RPGD && h->cfg.rpgd_gradient_mode >= 2) { src = h->d_elite_idx; need = (size_t)h->elite_log_rows * h->cfg.cem_best_k * 4; }
      else if (h->cfg.optimizer == CTK_OPT_RPGD) { src = h->d_best_idx; need = (size_t)h->cfg.rpgd_keep_k * 4; }
      else return fail(CTK_EINVAL, "no elite log for MPPI");
      break;
    case CTK_LOG_U_NOM:
      REQ(h->cfg.optimizer == CTK_OPT_RPGD, "u_nom log is RPGD only (use CTK_STATE_U_NOM for MPPI)");
      src = h->d_unom_log; need = H * 4; break;
    case CTK_LOG_AGES:
      REQ(h->cfg.optimizer == CTK_OPT_RPGD && h->cfg.logging, "ages log needs RPGD with logging");
      src = h->d_ages_log; need = N * 4; break;
    default: return fail(CTK_EINVAL, "unknown log id");
  }
  *src_out = src;
  *need_out = need;
  return CTK_OK;
}

extern "C" int ctk_get_log(ctk_handle* h, int which, void* dst, size_t nbytes) {
  REQ(h && dst, "null pointer");
  CU(cudaSetDevice(h->cfg.device));
  const void* src = nullptr;
  size_t need = 0;
  int rc = log_source(h, which, &src, &need);
  if (rc != CTK_OK) return rc;
  REQ(nbytes == need, "size mismatch (expected " + std::to_string(need) + " bytes)");
  CU(cudaMemcpyAsync(dst, src, need, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return CTK_OK;
}

extern "C" int ctk_get_log_view(ctk_handle* h, int which, const void** host_ptr, size_t* n_bytes) {
  REQ(h && host_ptr && n_bytes, "null pointer");
  REQ(which >= 0 && which < 8, "unknown log id");
  CU(cudaSetDevice(h->cfg.device));
  const void* src = nullptr;
  size_t need = 0;
  int rc = log_source(h, which, &src, &need);
  if (rc != CTK_OK) return rc;
  if (h->h_log_cap[which] < need) {
    if (h->h_log[which]) CU(cudaStreamSynchronize(h->stream));
    h->h_log_cap[which] = 0;
    CU(h->h_log[which].alloc(need ? need : 4, false));
    h->h_log_cap[which] = need;
  }
  CU(cudaMemcpyAsync(h->h_log[which], src, need, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  *host_ptr = h->h_log[which];
  *n_bytes = need;
  return CTK_OK;
}

// Top-M logging (SURVEY 8f.2; consumer: reference Controllers/__init__.py:159-178, producer optimizer_mppi.py:214-218): the logs of
// the m lowest-cost rollouts of the last tick only -- K4 top-k over J on the device (ties to the lower index, as everywhere), one
// gather launch per log out of the SoA buffers the rollout kernels wrote, ONE device->host copy of m x ((H+1) ns + H nu + 2) floats
// through pinned memory instead of the whole [N, H+1, ns] log (C5: 2.8 GB -> 0.18 MB at m = 64).  Any output pointer may be null.
extern "C" int ctk_get_log_top(ctk_handle* h, int m, int32_t* idx_out, float* J_out, float* Q_out, float* traj_out) {
  REQ(h, "null pointer");
  REQ(m >= 1 && m <= h->N && m <= 512, "need 1 <= m <= min(num_rollouts, 512)");
  REQ(h->cfg.logging || (Q_out == nullptr && traj_out == nullptr), "logging disabled (only the indices and costs are available)");
  CU(cudaSetDevice(h->cfg.device));
  const size_t N = h->N, H = h->H;
  const size_t RQ = H * h->nu, RT = (H + 1) * h->ns;
  const size_t nk = (size_t)((N + TOPK_THREADS - 1) / TOPK_THREADS) * m + TOPK_THREADS;
  if (h->top_keys_cap < nk) {
    h->top_keys_cap = 0;
    CU(h->d_top_keys[0].alloc(nk));
    CU(h->d_top_keys[1].alloc(nk));
    h->top_keys_cap = nk;
  }
  const size_t no = (size_t)m * (RQ + RT + 2);
  if (h->top_out_cap < no) {
    h->top_out_cap = 0;
    CU(h->d_top_out.alloc(no));
    CU(h->h_top.alloc(no, false));
    h->top_out_cap = no;
  }
  // K4 levels over the costs of the last tick (global ids: shard offset + local index)
  int cnt = (int)N;
  const uint64_t* kin = nullptr;
  CU(topk_levels(h->d_J, kin, cnt, 0, h->off, m, true, h->d_top_keys[0], h->d_top_keys[1], h->stream, h->launches));
  float* d_Q = h->d_top_out;                       // [m][H nu]
  float* d_T = d_Q + (size_t)m * RQ;               // [m][(H+1) ns]
  float* d_Jm = d_T + (size_t)m * RT;              // [m]
  int32_t* d_idx = reinterpret_cast<int32_t*>(d_Jm + m);  // [m]
  const int soa = h->env == 0 ? 1 : 0;
  const float* srcQ = nullptr;
  if (Q_out) srcQ = (h->env == 0 && h->cfg.optimizer == CTK_OPT_RPGD) ? h->d_Q_log : h->d_log_Q_soa;
  REQ(!Q_out || srcQ, "no control log for this configuration");
  REQ(!traj_out || h->d_log_traj_soa, "no trajectory log for this configuration");
  h->launches++;
  CU(launch_log_gather(kin, m, h->off, h->d_J, N, srcQ, (int)RQ, soa, d_Q, d_Jm, d_idx, h->stream));
  if (traj_out) {
    h->launches++;
    CU(launch_log_gather(kin, m, h->off, h->d_J, N, h->d_log_traj_soa, (int)RT, soa, d_T, nullptr, nullptr, h->stream));
  }
  CU(cudaMemcpyAsync(h->h_top, h->d_top_out, no * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  const float* hp = h->h_top;
  if (Q_out) memcpy(Q_out, hp, sizeof(float) * m * RQ);
  if (traj_out) memcpy(traj_out, hp + (size_t)m * RQ, sizeof(float) * m * RT);
  if (J_out) memcpy(J_out, hp + (size_t)m * (RQ + RT), sizeof(float) * m);
  if (idx_out) memcpy(idx_out, hp + (size_t)m * (RQ + RT) + m, sizeof(int32_t) * m);
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// nominal single rollout (predict_optimal_trajectory)
// ---------------------------------------------------------------------------------------------------------------
extern "C" int ctk_rollout_single(ctk_handle* h, const float* s_host, const float* Q_host, float* traj_host, float* summed) {
  REQ(h && s_host && Q_host && traj_host, "null pointer");
  REQ(h->env == 0, "the standalone nominal rollout is implemented for the CartPole environment");
  CU(cudaSetDevice(h->cfg.device));
  const int H = h->H;
  Owned<float> d;
  CU(d.alloc(8 + H + (size_t)(H + 1) * 6 + 1, false));
  float *d_s = d, *d_Q = d_s + 8, *d_traj = d_Q + H, *d_sum = d_traj + (size_t)(H + 1) * 6;
  CU(cudaMemcpyAsync(d_s, s_host, 6 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(d_Q, Q_host, H * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  h->launches++;
  CU(launch_single_rollout(pred_kind(h), d_s, d_Q, H, h->d_kc, h->mlp, h->d_u_prev, d_traj, d_sum, h->stream));
  std::vector<float> tmp((size_t)(H + 1) * 6 + 1);
  CU(cudaMemcpyAsync(tmp.data(), d_traj, tmp.size() * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  memcpy(traj_host, tmp.data(), sizeof(float) * (size_t)(H + 1) * 6);
  if (summed) *summed = tmp.back();
  return CTK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// utilities
// ---------------------------------------------------------------------------------------------------------------
extern "C" int ctk_fp32_peak(int device, double* tflops, double* clk_mhz) {
  REQ(tflops, "null pointer");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  Owned<float> d;
  CU(d.alloc((size_t)blocks * threads, false));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 6; ++rep) {
    CU(cudaEventRecord(e0));
    CU(launch_fma_peak(d, blocks, threads, iters, nullptr));
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8 * 16 * (double)iters * blocks * threads;
    if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *tflops = best;
  if (clk_mhz) *clk_mhz = best * 1e12 / (2.0 * 128.0 * prop.multiProcessorCount) / 1e6;  // implied FFMA issue clock
  return CTK_OK;
}

// warp-instructions per second per SMSP-cycle for an FP32 instruction mix (variant: see fp32_micro_kernel)
extern "C" int ctk_fp32_microbench(int device, int variant, double* ginstr_per_s) {
  REQ(ginstr_per_s && variant >= 1 && variant <= 5, "variant in 1..5");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 2048;
  Owned<float> d, seed;
  CU(d.alloc((size_t)blocks * threads, false));
  CU(seed.alloc(64, false));
  float hs[64];
  for (int i = 0; i < 64; ++i) hs[i] = 0.5f + 0.001f * i;
  CU(cudaMemcpy(seed, hs, sizeof(hs), cudaMemcpyHostToDevice));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CU(cudaEventRecord(e0));
    CU(launch_fp32_micro(variant, d, blocks, threads, iters, seed, nullptr));
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    const double ninstr = 64.0 * iters * (double)blocks * threads;  // thread-instructions
    if (rep > 0) best = std::max(best, ninstr / (ms * 1e-3) / 1e9);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *ginstr_per_s = best;
  return CTK_OK;
}

extern "C" int ctk_philox_fill(int device, uint64_t seed, int kind, float* dst, size_t n) {
  REQ(dst, "null pointer");
  CU(cudaSetDevice(device));
  Owned<float> d;
  CU(d.alloc(n, false));
  NoiseSrc ns{};
  ns.inj = nullptr; ns.key0 = (uint32_t)seed; ns.key1 = (uint32_t)(seed >> 32); ns.tick = 1; ns.stream = STREAM_MPPI;
  ns.per_rollout = 16; ns.uniform = kind;
  CU(launch_philox_fill(ns, d, n, nullptr));
  CU(cudaMemcpy(dst, d, sizeof(float) * n, cudaMemcpyDeviceToHost));
  return CTK_OK;
}

static_assert((uint32_t)CTK_STREAM_MPPI == STREAM_MPPI && (uint32_t)CTK_STREAM_CEM == STREAM_CEM && (uint32_t)CTK_STREAM_RPGD_INIT == STREAM_RPGD_INIT &&
                  (uint32_t)CTK_STREAM_RPGD_RESAMPLE == STREAM_RPGD_RESAMPLE, "public stream ids == kernel stream ids");
// The standard draws a consumer of THIS handle generates in Philox mode: same key (seed), same counter words (draw block,
// global rollout id, tick, stream) and the same device function (noise4) as the kernels, so a test can hand the oracle exactly
// the numbers the production (in-kernel noise) instantiations consumed.
extern "C" int ctk_philox_export(ctk_handle* h, uint32_t stream, int64_t tick, int per_rollout, int uniform, size_t row0, size_t rows,
                                 float* dst_host) {
  REQ(h && dst_host, "null pointer");
  REQ(per_rollout >= 1, "per_rollout must be >= 1");
  CU(cudaSetDevice(h->cfg.device));
  const size_t n = rows * (size_t)per_rollout;
  if (n == 0) return CTK_OK;
  NoiseSrc ns{};
  ns.inj = nullptr; ns.key0 = (uint32_t)(h->cfg.seed & 0xffffffffull); ns.key1 = (uint32_t)(h->cfg.seed >> 32);
  ns.tick = (uint32_t)tick; ns.stream = stream; ns.per_rollout = per_rollout; ns.uniform = uniform ? 1 : 0;
  Owned<float> d;
  CU(d.alloc(n, false));
  CU(launch_philox_export(ns, row0, d, n, h->stream));
  CU(cudaMemcpyAsync(dst_host, d, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return CTK_OK;
}

extern "C" int ctk_topk(int device, const float* cost_host, int n, int k, int32_t* idx_out) {
  REQ(cost_host && idx_out && n >= 1 && k >= 1 && k <= n && k <= 512, "need 1 <= k <= min(n, 512)");
  CU(cudaSetDevice(device));
  Owned<float> d_c;
  Owned<uint64_t> d_k0, d_k1;
  const size_t nk = (size_t)((n + 1023) / 1024) * k + 1024;
  CU(d_c.alloc(n, false));
  CU(d_k0.alloc(nk, false));
  CU(d_k1.alloc(nk, false));
  CU(cudaMemcpy(d_c, cost_host, sizeof(float) * n, cudaMemcpyHostToDevice));
  int cnt = n;
  const uint64_t* kin = nullptr;
  int64_t launches = 0;  // no handle to count them on
  CU(topk_levels(d_c, kin, cnt, 0, 0, k, true, d_k0, d_k1, nullptr, launches));
  std::vector<uint64_t> keys((size_t)k);
  CU(cudaMemcpy(keys.data(), kin, sizeof(uint64_t) * k, cudaMemcpyDeviceToHost));
  for (int i = 0; i < k; ++i) idx_out[i] = (int32_t)(keys[i] & 0xffffffffu);
  return CTK_OK;
}
