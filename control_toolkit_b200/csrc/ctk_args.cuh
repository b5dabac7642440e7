// ctk_args.cuh -- plain argument blocks shared by the host-side engine (ctk_engine.cu) and the kernel translation
// units.  No device code here.
#pragma once
#include <stdint.h>
#include <stddef.h>

#include "ctk_math.cuh"

namespace ctk {

enum : uint32_t { STREAM_MPPI = 0, STREAM_CEM = 1, STREAM_RPGD_INIT = 2, STREAM_RPGD_RESAMPLE = 3 };

struct NoiseSrc {
  const float* inj;   // != nullptr: injected standard draws, row-major [N_global, per_rollout]; else Philox
  uint32_t key0, key1;  // seed
  uint32_t tick;        // counter word 2
  uint32_t stream;      // counter word 3 (STREAM_* + sub-iteration << 8)
  int per_rollout;      // draws per rollout in this block of noise
  int uniform;          // 0: N(0,1)  1: U[0,1)
};

// Initial state of a tick: either a device pointer (device-resident callers, ctk_step_device / ctk_step_local) or the six
// values themselves inside the kernel parameters (host callers: ctk_step needs no host->device copy at all).
struct S0 {
  const float* p;  // [6] device, or null -> v
  float v[6];
#if defined(__CUDACC__)
  __device__ __forceinline__ float ld(int i) const { return p != nullptr ? p[i] : v[i]; }
#endif
};

// Result mirror in MAPPED pinned host memory (device view).  The kernel that finishes a tick stores u, the status word and
// (optionally) one [H] state array there as tagged 8-byte slots (value | launch sequence number, ctk_device.cuh host_put): the
// host caller polls the tags instead of enqueueing device->host copies and synchronising the stream.
// Layout (uint64 slots): [4] u  [5] status  [8 .. 8+H) state array;  floats [0..6) carry the state in the other direction.
struct HostMirror {
  float* p;          // null: no mirror (device-resident callers)
  unsigned int seq;  // never 0
};

struct MlpDev {
  int hidden;              // <= 128, multiple of 16
  const float* blob;       // device: W1[6][hid] | b1[hid] | W2[hid][hid] | b2[hid] | W3T[5][hid] | b3[8]
  int blob_floats;
  const void* tc_blob;     // device: tcgen05 engine blob (ctk_mlp_tc.cuh: W2 bf16 split tiles | W1 | b1 | b2 | W3T | b3) or null
  // recurrent predictor (GruSimtPred): blob = Wi1[6][3h] | Wh1[h][3h] | bi1[3h] | bh1[3h] | Wi2[h][3h] | Wh2[h][3h] | bi2[3h] | bh2[3h] |
  // W3T[5][h] | b3[8], gate order [r, z, n]; rnn_h = the SAVED hidden state [2][2h]: row 0 current (every rollout starts from it),
  // row 1 the state before the last predictor.update (nominal rollout of the tick, reference optimizer_mppi.py:199-202)
  const float* rnn_h;
};

CTK_HD int mlp_blob_floats(int hid) { return 6 * hid + hid + hid * hid + hid + 5 * hid + 8; }
CTK_HD int gru_blob_floats(int hid) { return 3 * hid * (6 + hid + 2) + 3 * hid * (2 * hid + 2) + 5 * hid + 8; }

// Loop-invariant constants of the rollout kernels live in DEVICE memory (handle-owned) and are read once per thread
// with volatile loads: sm_100 FP instructions take no constant-bank operands and ptxas re-issues LDC/LDCU inside the
// rollout loop for kernel-parameter constants (18 issue slots per rollout-step, seen in SASS); a volatile global load
// cannot be rematerialised, so the values stay in registers.
struct DevConsts {
  FwdK fwd;
  CostC cost;
  OdeC ode;  // adjoint constants (rpgd_grad_coef_kernel keeps them register-resident the same way)
};

// The 12 constants that appear as the multiplier / addend of an FMA whose other two sources are registers.  They are
// passed as KERNEL PARAMETERS (constant bank -> LDCU -> uniform registers) so those FMAs read only two vector
// registers; an FMA with three distinct vector-register sources issues at ~58 % rate on sm_100 (register-file read
// bandwidth, measured with ctk_fp32_microbench).  The remaining constants only feed 2-operand instructions and live in
// vector registers (DevConsts).
struct alignas(16) HotUK {
  float k_dd, k_bar, k_ep, k_cc;
  float k_ccrc, k_du2, k_udu, cU;
  float kTm, h, hk, K1p;
};

// ----------------------------------------------------------------------------------------------------------------
// In-kernel tick finish (K2 fused into the rollout kernel).  Every block publishes its softmin record [rho_b, a_b, b_z[n_ind]]
// as tagged 8-byte slots (value | sequence number in ONE store: no fence, no flag round trip) into its shard's mailbox; block 0
// of every shard, the finisher, polls the grid's records, rescales them exactly to their minimum, forwards the shard's combined
// record over NVLink peer stores into every shard's mailbox (hops == 2, default), polls the world's shard records and updates
// u_nom / u.  hops == 1 instead stores every BLOCK record straight into every shard's mailbox and lets each finisher combine
// world x grid records: one global hop less on paper, measured slower at 8 GPUs (13 k small NVLink writes per GPU and tick take
// ~6 us to land, a single forwarded record ~2.8 us).  Every shard combines the same records in the same order: the replicated
// optimizer state stays bit-identical.  Replaces reference optimizer_mppi.py:163-168,190-191 (+ the cross-shard
// weighted-sum exchange of SURVEY 8e).
// Mailbox layout (uint64 slots): [2 (sequence parity)][CTK_MAX_PEERS (source shard)][CTK_MBOX_BLOCKS (source block)][record stride],
// then the barrier area [2][CTK_MAX_PEERS] and the hand-over slots.  Double-buffered by parity: a shard can be at most one tick
// ahead of its slowest peer.
// Chained ticks (ctk_step_device_n): the finisher also publishes u_prev and u_nom[H] as tagged slots (handover); the next tick of the
// chain polls them instead of waiting for the previous launch to complete (griddepcontrol.wait), which takes the kernel-completion /
// dependent-release latency off the tick-to-tick critical path.
// ----------------------------------------------------------------------------------------------------------------
constexpr int CTK_MAX_PEERS = 8;
constexpr int CTK_MBOX_BLOCKS = 320;  // >= the grid of any rollout kernel (one or two CTAs per SM: 148 SMs on B200)
CTK_HD int mbox_record_stride(int n_ind) { return (n_ind + 3) & ~1; }  // slots per record: 2 + n_ind padded to even (16-byte polls)
CTK_HD size_t mbox_record_slots(int n_ind) { return (size_t)2 * CTK_MAX_PEERS * CTK_MBOX_BLOCKS * mbox_record_stride(n_ind); }
// + barrier area [2][CTK_MAX_PEERS] + tagged hand-over of the tick's result to the next tick of a chain: u_prev, u_nom[H] (H <= 4096 slots)
CTK_HD size_t mbox_barrier_offset(int n_ind) { return mbox_record_slots(n_ind); }
CTK_HD size_t mbox_handover_offset(int n_ind) { return mbox_record_slots(n_ind) + 2 * CTK_MAX_PEERS; }
CTK_HD size_t mbox_total_slots(int n_ind, int H) { return mbox_handover_offset(n_ind) + 1 + (size_t)H; }
struct MppiFuse {
  int mode;                  // 0: block records only (legacy K2 launch follows)  1: + shard record (staged exchange)  2: + finalize
  int world, rank;           // shards taking part in the exchange (1: no exchange)
  unsigned int seq;          // sequence number of this launch (monotonic, never 0, in lock step on all shards): tag of the records
  float* record_out;         // [2 + n_ind] shard record (mode >= 1)
  unsigned long long* mbox_local;                 // this shard's mailbox
  unsigned long long* mbox_peer[CTK_MAX_PEERS];   // every shard's mailbox (mbox_peer[rank] == mbox_local)
  unsigned long long* handover;                   // [1 + H] tagged u_prev, u_nom[H] of the tick (local); a chained tick READS its predecessor's
  int publish_handover;                           // 1: a chained tick follows this one, publish the hand-over
  unsigned long long* trace; // diagnostics: block 0's row of the phase timeline (slots 6, 7: records polled, records combined) or null
  int hops;                  // cross-GPU exchange: 1 every block stores its record into every shard's mailbox; 2 the finisher forwards the shard record
  int chained;               // 1: the previous launch of the stream is the previous tick of this handle's chain: poll its hand-over
  float* u_nom;              // [H] in/out
  float* u_prev;             // [1] out (unless frozen)
  float* u_out;              // [2] out: u, status (0 ok, 1 a peer's record missing, 2 a local block's record missing)
  int freeze_prev;
  HostMirror host;           // mode 2: u / status / u_nom[H] mirrored to the host caller
};

struct MppiArgs {
  int N, off, H, period, n_ind;  // local rollouts, global id offset, horizon, inducing-point period / count
  S0 s0;                         // initial state
  const float* u_nom;            // [H] device, UNSHIFTED state of the previous tick (shift applied on read, :184)
  const float* u_prev;           // [1] device, previous_input of the cost (self.u, :211)
  NoiseSrc noise;                // per_rollout = n_ind
  float stdev, lo, hi;           // SQRTRHODTINV (:130), control limits
  float k_du2, k_udu, k_uu, neg_inv_lbd;  // :154-155 pre-multiplied by cc_weight; :165
  int stash;                     // 1: keep each rollout's draws in shared memory for the softmin record (else regenerate)
  const DevConsts* kc;           // device: forward ODE + cost constants
  const float* kx;               // device: {lo, hi, k_du2, k_udu}
  HotUK uk;                      // uniform-register constants (see HotUK)
  MlpDev mlp;
  float* J;                      // [N] out: total MPPI cost S
  float* partials;               // [gridDim.x][2 + n_ind] out: rho_b, a_b, b_z[n_ind]
  float* log_traj_soa;           // [(H+1)][6][N] or null
  float* log_Q_soa;              // [H][N] or null
  MppiFuse fuse;                 // in-kernel tick finish (see MppiFuse)
};

// K2: combine `cnt` softmin records [rho, a, b_z[n_ind]] (block partials or per-shard records) into one record;
// if fin.enable, finish the tick: u_nom <- clip(shift(u_nom) + interp(b_z) * stdev / a)  (optimizer_mppi.py:190-191)
struct MppiFinalize {
  int enable;
  int H, period, n_ind;
  float stdev, lo, hi, neg_inv_lbd;
  float* u_nom;   // [H] in/out
  float* u_prev;  // [1] out (unless frozen)
  float* u_out;   // [1] out or null
  int freeze_prev;
};

// Uniform-register constants of the scaled-variable CartPole rollout (K1 for the ODE predictor, ctk_kernels_mppi_ode.cuh).
// State variables carried per rollout:  T = angle/sqrt(2),  W = beta*angleD (beta = sqrt((k+1)L/g)),  c, s,  x,
// V = (cF/g)*positionD.  With them one Euler step is 12 FP32 instructions + wrap (3) + half-angle sincos (14) + 1 MUFU.
struct OdeHot {
  // dynamics
  float cUg, cTl2, kTm2, K1p, h_T, h_W, h_x, h_V;
  // state scaling (prologue / logs / terminal cost)
  float beta, inv_beta, cFg, inv_cFg;
  // stage cost, pre-multiplied by 1/(H+1); kA/kB/kC: u * (kA u + kB u_prev + kC du) merges the cost's cc and ccrc terms
  // with the MPPI correction (optimizer_mppi.py:154-155)
  float k_dd, k_bar, k_ep, k_ekp2, kA, kB, kC, k_du2, k_ccrc;
  float target, thl_095, thl_09, k_border, thl_01, k_term, shift;
  float lo, hi, stdev, neg_inv_lbd;
};

struct MppiOdeArgs {
  int N, off, H, period, n_ind;
  int fshare16;         // share of block 0, the tick's finisher, in sixteenths of an ordinary block's share (16: equal shares)
  double per16;         // N / (fshare16 + 16 (grid - 1)): rollouts per sixteenth of a share (0: the kernel derives it)
  S0 s0;                // initial state
  const float* u_nom;   // [H] unshifted
  const float* u_prev;  // [1]
  NoiseSrc noise;
  OdeHot k;
  float* J;             // [N]
  float* partials;      // [gridDim.x][2 + n_ind]
  float* log_traj_soa;  // [(H+1)][6][N] or null
  float* log_Q_soa;     // [H][N] or null
  unsigned long long* trace;  // [gridDim.x][8] globaltimer stamps per block (diagnostics) or null
  MppiFuse fuse;
};

// Several clients' MPPI ticks in one launch (mppi_ode_batch_kernel, ctk_kernels_mppi_ode.cuh): per-client inputs inside the kernel
// parameters, per-client state behind the pointers of client 0 at fixed strides
constexpr int kMaxBatchClients = 16;
struct MppiBatch {
  int active[kMaxBatchClients];
  uint32_t tick[kMaxBatchClients];   // Philox counter word of the client's tick
  float s0[kMaxBatchClients][8];     // measured states
  size_t stride_unom, stride_J, stride_partials, stride_record, stride_mbox;  // elements between consecutive clients
};

struct CemArgs {
  int N, off, H;
  S0 s0;                // initial state
  const float* mu;      // [H] dist_mue
  const float* sd;      // [H] stdev
  const float* u_prev;  // [1]
  NoiseSrc noise;       // per_rollout = H
  float lo, hi;
  const DevConsts* kc;  // device: forward ODE + cost constants
  MlpDev mlp;
  float* J;             // [N]
  float* log_traj_soa;  // [(H+1)][6][N] or null
  float* log_Q_soa;     // [H][N] or null
};

// K3 for the ODE predictor with intermediate_steps == 1: the scaled-variable step of K1 (ctk_ode_scaled.cuh)
struct CemOdeArgs {
  int N, off, H;
  S0 s0;                // initial state
  const float* mu;      // [H] dist_mue
  const float* sd;      // [H] stdev
  const float* u_prev;  // [1]
  NoiseSrc noise;       // per_rollout = H
  OdeHot k;             // uniform-register constants (derive_ode_hot with a zero MPPI correction; lo / hi = control limits)
  float* J;             // [N]
  float* log_traj_soa;  // [(H+1)][6][N] or null
  float* log_Q_soa;     // [H][N] or null
  uint64_t* cand_out;   // != null: every block (256 rollouts) also sorts its (cost, global id) keys and emits its kk smallest
  int kk;               //          to cand_out[blockIdx.x * kk ..] -- level 0 of the hierarchical top-k without its own launch
};

// The whole CEM tick (all outer iterations) as ONE persistent launch for populations that fit one resident grid
// (ctk_kernels_cem.cuh cem_tick_kernel): blocks exchange their candidate keys and block 0 publishes the refit distribution
// through tagged 8-byte slots, so the iterations need no kernel boundary.
struct CemTickArgs {
  int N, off, H, k, iters;
  S0 s0;
  float *mu, *sd;              // [H] dist_mue / stdev, in/out
  float* u_prev;               // [1] in (cost) / out (unless frozen)
  float* u_out;                // [1] or null
  int freeze_prev;
  NoiseSrc noise;              // iteration 0; iteration it: stream | it << 8, inj + it * inj_stride
  size_t inj_stride;           // draws per iteration (N_global * H)
  OdeHot hot;                  // uniform-register constants (zero MPPI correction; lo / hi = control limits)
  float* J;                    // [N] costs of the LAST iteration
  float* log_traj_soa;         // [(H+1)][6][N] or null
  float* log_Q_soa;            // [H][N] or null
  unsigned long long* cand;    // [gridDim.x][k] tagged candidate keys: ordered cost (32) | id (16) | sequence tag (16)
  int k2, runs_pad, q_cap;     // pow2 >= max(k, 32); pow2 >= gridDim.x; floats of the big shared buffer (>= runs_pad * k2 * 2)
  int rb;                      // rollouts per block (power of two, 32 .. 512; the block has 512 threads)
  unsigned long long* dist;    // [2][H] tagged mu / sd published by block 0 for the next iteration
  unsigned int seq0;           // sequence number of iteration 0 (monotonic across ticks, never 0)
  float sd_min, sd_init;
  int32_t* elite_idx_out;      // [elite_cap][k] global ids, best first, or null
  int elite_cap;
  HostMirror host;
  unsigned long long* trace;   // diagnostics (ctk_debug_trace): block 0's globaltimer stamps [iteration][8], or null
};

struct CemRefitArgs {
  int H, k, cnt;             // cnt candidate keys (num_shards * k, each shard's list sorted or not)
  const uint64_t* cand;      // [cnt] (ordered cost, global id)
  NoiseSrc noise;            // the SAME noise block the rollouts consumed: elite Q rows are regenerated, never stored
  float lo, hi;
  float* mu;                 // [H] in/out
  float* sd;                 // [H] in/out
  int last;                  // 1: apply the post-loop clip/shift of optimizer_cem_tf.py:99-102
  float sd_min, sd_init;
  float* u_prev;             // [1]
  float* u_out;              // [1] or null
  int freeze_prev;
  int32_t* elite_idx_out;    // [k] global ids, best first (log) or null
  HostMirror host;           // last iteration: u mirrored to the host caller
  // Fused cross-GPU candidate exchange (SURVEY 8e, CEM row): world > 1 -> `cand` holds THIS shard's k best keys; the kernel stores
  // them into every shard's mailbox over NVLink (two tagged 8-byte slots per key: high / low word | sequence number), polls the
  // world x k keys of its own mailbox and merges them -- every shard refits the same distribution, no NCCL call, no host round trip.
  // Mailbox layout (uint64 slots): [2 (sequence parity)][CTK_MAX_PEERS][kCemMboxKeys][2], then the barrier area.
  int world, rank;
  unsigned int seq;          // exchange sequence number of this outer iteration (monotonic, never 0, lock step on all shards)
  unsigned long long* mbox_local;
  unsigned long long* mbox_peer[CTK_MAX_PEERS];
};
constexpr int kCemMboxKeys = 512;  // = the largest cem_best_k
CTK_HD size_t cem_mbox_slots() { return (size_t)2 * CTK_MAX_PEERS * kCemMboxKeys * 2 + 2 * CTK_MAX_PEERS; }

struct RpgdGradArgs {
  int N, H, iters;
  S0 s0;                // initial state
  const float* u_prev;  // [1] previous_input (self.u)
  float* Q;             // [H][N] in/out
  float* m;             // [H][N] in/out
  float* v;             // [H][N] in/out
  float lo, hi;
  float lr, gradmax_clip;
  double beta1, beta2, eps;
  long long adam_step0;  // global step counter before this tick's first gradient step
  int adam_form;         // 0 Keras, 1 torch, 2 plain gradient descent q - lr * g (optimizer_cem_naive_grad_tf.py:74)
  const DevConsts* kc;   // device copy of {fwd, cost, ode}: register-resident constants of the coefficient-form kernel
  OdeC ode;              // adjoint constants
  FwdK fwd;              // forward constants
  CostC cost;
  float* J;              // [N] cost of the final (get_action) rollout
  float* log_traj_soa;   // [(H+1)][6][N] or null
  unsigned long long* trace;  // diagnostics (ctk_debug_trace): globaltimer stamps of block 0's phases, or null
  // Adam bias corrections of the first kAdamHostIters gradient steps of this launch, evaluated on the host in float64 and rounded
  // once (1 - beta1^t, 1 - beta2^t, lr sqrt(1 - beta2^t) / (1 - beta1^t)); later steps (warm-up ticks) use the in-kernel pow
  int n_host_adam;
  float bc1_h[8], bc2_h[8], alpha_h[8];
};

constexpr int kEnvMaxStates = 8, kEnvMaxControls = 4;  // states / control inputs of any environment (the CartPole: 6 / 1)

// Population steps of the gradient optimizers (ctk_kernels_rpgd_select.cuh), for the CartPole and every registered environment:
// populations are [H][nu][N] (flat column t * nu + c), limits per input.
struct RpgdSelectArgs {
  int N, H, k, period, n_ind;
  int shift_previous;
  int resample;            // count % resamp_per == 0
  int tail_resample;       // gradient mode: no reordering, the LAST control of every row is redrawn (noise rows 0..N-1, nu draws each)
  const float* J;          // [N]
  const float *Q, *m, *v;  // [H][nu][N] current
  const float* ages;       // [N]
  float *Qn, *mn, *vn;     // [H][nu][N] next
  float* agesn;            // [N]
  NoiseSrc noise;          // resample: per_rollout = n_ind * nu (C order over [n_ind, nu]), rows 0..N-k-1; tail redraw: per_rollout = nu
  int dist;                // 0 normal, 1 uniform
  float s_mean, s_std;
  float s_min[kEnvMaxControls], s_max[kEnvMaxControls], lo[kEnvMaxControls], hi[kEnvMaxControls];
  float* u_nom_out;        // [H][nu] Q[best_idx[0]] BEFORE the shift (optimal_control_sequence, :426)
  float* u_prev;           // [nu]
  float* u_out;            // [nu] or null
  int freeze_prev;
  int32_t* best_idx_out;   // [k]
  HostMirror host;         // u of input 0 and u_nom_out mirrored to the host caller (CartPole host-facing ticks), or null
};

// Gradient-assisted CEM (reference optimizer_cem_naive_grad_tf.py, optimizer_cem_grad_bharadhwaj_tf.py): population stored like RPGD
struct GradCemSampleArgs {
  int H, ld, col0, cnt;    // dst[col * ld + col0 + r] for r < cnt, col < H * nu
  const float *mu, *sd;    // [H][nu]
  NoiseSrc noise;          // rows 0..cnt-1, per_rollout = H * nu, draw index = column
  float lo[kEnvMaxControls], hi[kEnvMaxControls];
  float* dst;              // [H][nu][ld]
};

struct GradCemRefitArgs {
  int N, H, k;
  const float* J;          // [N] costs of the population AFTER its gradient step
  const float* Q;          // [H][nu][N] that population
  float* Q_carry;          // [H][nu][N] next buffer: the k elites are written to columns 0..k-1 (rank order), or null
  float *mu, *sd;          // [H][nu] out
  int last;                // 1: post-loop clip / shift, the vacated last step refilled with mid-range means
  int u_from_mean;         // 1: u = refit mean[0] (naive-grad :105), 0: u = best sample's first control (bharadhwaj :168)
  float sd_min, sd_init;
  float lo[kEnvMaxControls], hi[kEnvMaxControls];
  float* u_prev;           // [nu]
  float* u_out;            // [nu] or null
  int freeze_prev;
  int32_t* elite_idx_out;  // [k] or null
  HostMirror host;         // last iteration: u mirrored to the host caller
};

// ---- environments registered through the functor registry (ctk_kernels_env.cuh) ----------------------------------------------
struct EnvParams { float p[24]; };           // environment-specific constants (layout: the Env struct in ctk_kernels_env.cuh)
struct S0e { const float* p; float v[kEnvMaxStates]; };  // initial state: device pointer, or the values inside the kernel parameters
struct EnvMppiArgs {
  int N, off, H, period, n_ind;
  S0e s0;
  float* u_nom;          // [H][NU] in (unshifted, :184 shift on read) / out (update kernel)
  float* u_prev;         // [NU]
  NoiseSrc noise;        // per_rollout = n_ind * NU, C order over [n_ind, NU]
  float stdev, k_du2, k_udu, k_uu, neg_inv_lbd;
  float lo[kEnvMaxControls], hi[kEnvMaxControls];
  EnvParams env;
  float* J;              // [N] total MPPI cost S
  float* log_traj;       // [N][H+1][NS] or null
  float* log_Q;          // [N][H][NU] or null
  float* u_out;          // [NU] or null
  int freeze_prev;
};
struct EnvCemArgs {
  int N, off, H;
  S0e s0;
  const float* mu;       // [H][NU]
  const float* sd;       // [H][NU]
  const float* u_prev;   // [NU]
  NoiseSrc noise;        // per_rollout = H * NU
  float lo[kEnvMaxControls], hi[kEnvMaxControls];
  EnvParams env;
  float* J;
  float* log_traj;
  float* log_Q;
};
struct EnvCemRefitArgs {
  int H, nu, k, cnt;
  const uint64_t* cand;  // [cnt] (ordered cost, global id)
  NoiseSrc noise;
  float lo[kEnvMaxControls], hi[kEnvMaxControls];
  float *mu, *sd;        // [H][NU] in/out
  int last;
  float sd_min, sd_init;
  float* u_prev;         // [NU]
  float* u_out;          // [NU] or null
  int freeze_prev;
  int32_t* elite_idx_out;
};

// Gradient optimizers on a registered environment (ctk_kernels_env_rpgd.cuh).  Population arrays are [H][NU][N]: flat column
// t * NU + c, one thread per trajectory reads coalesced.
constexpr int kEnvRpgdBlock = 32;  // trajectories per block of the gradient kernel (= the largest population of the one-launch tick)
constexpr size_t kEnvRpgdSmemMax = 227 * 1024 - 1024;  // the tape (dynamic shared memory); the fused select's arrays come on top
struct EnvRpgdGradArgs {
  int N, H, iters;
  S0e s0;
  const float* u_prev;   // [NU]
  float *Q, *m, *v;      // [H][NU][N] in/out
  float lo[kEnvMaxControls], hi[kEnvMaxControls];
  float lr, gradmax_clip;
  double beta1, beta2, eps;
  long long adam_step0;
  int adam_form;         // as RpgdGradArgs
  EnvParams env;
  float* J;              // [N] cost of the updated population
  float* log_traj;       // [N][H+1][NS] or null
  float* log_Q;          // [N][H][NU] or null
  int n_host_adam;
  float bc1_h[8], bc2_h[8], alpha_h[8];
};

constexpr int TOPK_THREADS = 1024;  // keys per top-k block

}  // namespace ctk
