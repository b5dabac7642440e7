/* ctk_b200.h -- C ABI of libctk_b200.so: the B200 (sm_100a) backend for the batched MPC rollout hot path of
 * SensorsINI/Control_Toolkit (MPPI / CEM / RPGD + the predictor and cost they drive).
 *
 * The reference is pure Python; its "FFI" for this path is the Python optimizer plugin interface
 *   template_optimizer.__init__/configure/step/optimizer_reset      (reference Optimizers/__init__.py:13-71)
 * as called by controller_mpc                                          (reference Controllers/controller_mpc.py:56-109).
 * Every entry point below cites the reference call it replaces.  The Python classes in
 * control_toolkit_b200/Optimizers/ bind these symbols with ctypes (the same mechanism the reference itself uses to
 * call C at Controllers/controller_C.py:222-248); INTEGRATION.md shows the binding.
 *
 * Conventions: plain pointers and sizes only; all arrays are fp32 unless stated; "host" pointers are ordinary host
 * memory (pinned or not), "dev" pointers are device memory on the handle's device.  Every function returns 0 on
 * success or a negative CTK_E* code; ctk_last_error() returns a thread-local message.  There is no CPU fallback:
 * if no CUDA device is usable, ctk_create fails.
 */
#ifndef CTK_B200_H
#define CTK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTK_ABI_VERSION 1

/* ---- status codes ------------------------------------------------------------------------------------------- */
#define CTK_OK 0
#define CTK_EINVAL (-1)   /* bad argument / unsupported configuration (Python raises ValueError)                 */
#define CTK_ECUDA (-2)    /* CUDA runtime error (Python raises RuntimeError)                                     */
#define CTK_ESTATE (-3)   /* call made in the wrong state (e.g. step before reset)                               */

/* ---- enums -------------------------------------------------------------------------------------------------- */
enum { CTK_OPT_MPPI = 0, CTK_OPT_CEM = 1, CTK_OPT_RPGD = 2 };            /* optimizer_mppi / optimizer_cem_tf / optimizer_rpgd */
enum { CTK_PRED_ODE = 0, CTK_PRED_MLP = 1, CTK_PRED_GRU = 2 };           /* predictor_specification "ODE" / "Dense-..." / "GRU-..." */
enum { CTK_COST_DEFAULT = 0, CTK_COST_QUADRATIC_BOUNDARY_GRAD = 1 };     /* cost_function_specification                         */
/* environment_name (reference Controllers/__init__.py:33; the cost class is Control_Toolkit_ASF.Cost_Functions.<env>.<name>,
   Cost_Functions/cost_function_wrapper.py:59-66).  CARTPOLE: 6 states, 1 control, every optimizer and predictor, the fused kernels.
   DUBINS_CAR: 3 states [x, y, yaw], 2 controls [throttle, steer]; MPPI and CEM with its ODE and its `default` cost through the
   general-environment kernels (ctk_kernels_env.cuh); parameters by ctk_set_env_params, per-input limits by ctk_set_control_limits. */
enum { CTK_ENV_CARTPOLE = 0, CTK_ENV_DUBINS_CAR = 1 };
enum { CTK_DIST_NORMAL = 0, CTK_DIST_UNIFORM = 1 };                      /* RPGD SAMPLING_DISTRIBUTION                          */
enum { CTK_ADAM_KERAS = 0, CTK_ADAM_TORCH = 1 };                         /* reference optimizer_rpgd.py:34-43 vs :56-82         */
/* MLP predictor engine.  SIMT: FP32 pipe (numerical anchor).  TCGEN05: 128 x 128 layer on the tensor cores as six products of
   three-term bf16 splits (fp32-level accuracy, passes the fp32 reference fixtures).  TCGEN05_BF16 / TCGEN05_FAST: opt-in reduced
   precision -- ONE bf16 product (operands rounded to bfloat16, fp32 accumulation); _FAST additionally evaluates tanh with the
   single-instruction MUFU.TANH (~2^-11 relative).  Parity of _BF16 is defined against an oracle applying the same operand rounding. */
enum { CTK_MLP_SIMT = 0, CTK_MLP_TCGEN05 = 1, CTK_MLP_TCGEN05_BF16 = 2, CTK_MLP_TCGEN05_FAST = 3 };

/* which = state arrays (get/set).  Layouts are the reference's: [1,H,nu] or [N,H,nu] row-major.                 */
enum {
  CTK_STATE_U_NOM = 0,      /* MPPI u_nom [H,nu] ([num_clients][H] for a multi-client handle) (optimizer_mppi.py:227-231); RPGD:
                               Q[best] before the shift [H,nu]                                                      */
  CTK_STATE_CEM_MU = 1,     /* CEM dist_mue [H]          (optimizer_cem_tf.py:114)                                */
  CTK_STATE_CEM_STD = 2,    /* CEM stdev [H]             (optimizer_cem_tf.py:115)                                */
  CTK_STATE_RPGD_Q = 3,     /* RPGD Q_tf [N,H,nu]        (optimizer_rpgd.py:540-544)                              */
  CTK_STATE_RPGD_M = 4,     /* Adam m [N,H,nu]           (optimizer_rpgd.py:84-131)                               */
  CTK_STATE_RPGD_V = 5,     /* Adam v [N,H,nu]                                                                    */
  CTK_STATE_RPGD_AGES = 6,  /* trajectory_ages [N]       (optimizer_rpgd.py:548)                                  */
  CTK_STATE_U_PREV = 7,     /* self.u, the previous_input of the cost [nu] (Optimizers/__init__.py:35)            */
  CTK_STATE_RNN_H = 8       /* saved hidden state of the recurrent predictor [2 * hidden] (layer 1 | layer 2): what every rollout
                               starts from and predictor.update advances (optimizer_mppi.py:195-197)                  */
};
/* which = integer counters */
enum { CTK_COUNTER_COUNT = 0,      /* optimizer.count   (optimizer_cem_tf.py:116, optimizer_rpgd.py:545)          */
       CTK_COUNTER_ADAM_STEP = 1,  /* Adam global step  (optimizer_rpgd.py:59)                                    */
       CTK_COUNTER_TICK = 2 };     /* number of step() calls since create (Philox counter word)                   */
/* which = logs of the LAST tick (only filled when cfg.logging != 0; reference optimizer_mppi.py:214-218)         */
enum {
  CTK_LOG_Q = 0,          /* Q_logged [N,H,nu]                                                                    */
  CTK_LOG_J = 1,          /* J_logged [N]        (always available, logging or not)                               */
  CTK_LOG_ROLLOUTS = 2,   /* rollout_trajectories_logged [N,H+1,ns]                                               */
  CTK_LOG_ELITE_IDX = 3,  /* int32 [iters_of_last_tick, k] global rollout ids of the elites, best first (CEM);
                             [k] best_idx (RPGD)                                                                   */
  CTK_LOG_U_NOM = 4,      /* optimal_control_sequence [H] of the last tick (RPGD u_nom, optimizer_rpgd.py:426)    */
  CTK_LOG_AGES = 5        /* trajectory_ages_logged [N] (RPGD, ages before the update, optimizer_rpgd.py:415)     */
};

/* ---- parameter blocks (compound constants evaluated in float64 on the host, rounded once to fp32) ------------ */
typedef struct ctk_ode_params {   /* CartPole Euler ODE; replaces PredictorWrapper.predict_core for "ODE"        */
  float u_max, kp1_Mm, m, neg_M_fric, neg_J_fric, mg, L, kp1, mL, g, kp1L, h;
  int32_t intermediate_steps;
} ctk_ode_params;

typedef struct ctk_cost_params {  /* CartPole cost classes; replaces CostFunctionWrapper.get_trajectory_cost     */
  int32_t kind;                   /* CTK_COST_*                                                                  */
  float dd_weight, ep_weight, ekp_weight, cc_weight, ccrc_weight, R, MAX_COST;
  float two_thl, thl_095, thl_005, thl_09, thl_01;
  float target_position, target_equilibrium;   /* live environment attributes (controller update_attributes)     */
} ctk_cost_params;

typedef struct ctk_mlp_weights {  /* Dense 6 -> hidden tanh -> hidden tanh -> 5 ; row-major [in,out]; host ptrs  */
  int32_t hidden;
  const float *W1, *b1, *W2, *b2, *W3, *b3;
} ctk_mlp_weights;

typedef struct ctk_gru_weights {  /* 6 -> GRU(hidden) -> GRU(hidden) -> Dense 5; row-major [in, 3*hidden], gate order [r, z, n];
                                     r = sigmoid(gi_r + gh_r), z = sigmoid(gi_z + gh_z), n = tanh(gi_n + r * gh_n), h' = (1-z) n + z h
                                     with gi = x Wi + bi, gh = h Wh + bh (torch.nn.GRU / Keras reset_after cell); host ptrs            */
  int32_t hidden;                 /* multiple of 8, <= 32                                                        */
  const float *Wi1, *Wh1, *bi1, *bh1, *Wi2, *Wh2, *bi2, *bh2, *W3, *b3;
} ctk_gru_weights;

typedef struct ctk_config {
  int32_t abi_version;            /* = CTK_ABI_VERSION                                                           */
  int32_t optimizer;              /* CTK_OPT_*                                                                   */
  int32_t predictor;              /* CTK_PRED_*                                                                  */
  int32_t device;                 /* CUDA device ordinal                                                         */
  /* template_optimizer ctor (reference Optimizers/__init__.py:13-50) */
  int32_t num_rollouts;           /* rollouts evaluated by THIS handle (local shard)                             */
  int32_t num_rollouts_global;    /* total over all shards (== num_rollouts when not sharded)                    */
  int32_t rollout_offset;         /* global id of local rollout 0 (Philox counters use global ids)               */
  int32_t mpc_horizon;
  int32_t num_states;             /* 6                                                                           */
  int32_t num_control_inputs;     /* 1                                                                           */
  float action_low, action_high;
  uint64_t seed;
  int32_t logging;                /* optimizer_logging                                                           */
  int32_t freeze_previous_input;  /* 1: previous_input frozen at 0 (TF graph-trace semantics, SURVEY 8 quirks)   */
  int32_t period_interpolation_inducing_points;  /* MPPI, RPGD                                                   */
  /* MPPI (reference optimizer_mppi.py:16-34,130,154-168); fp32 coefficients precomputed by the host in the
     reference's evaluation order */
  float mppi_coef_du2;            /* fp32(fp32(0.5*(1-1/NU))*R)                                                  */
  float mppi_R;                   /* R                                                                           */
  float mppi_half_R;              /* fp32(0.5*R)                                                                 */
  float mppi_cc_weight;
  float mppi_neg_inv_LBD;         /* fp32(-1.0/LBD)                                                              */
  float mppi_stdev;               /* SQRTRHODTINV = fp32(SQRTRHOINV/sqrt(dt))                                    */
  /* CEM (reference optimizer_cem_tf.py:16-34) */
  int32_t cem_outer_it, cem_best_k, cem_warmup, cem_warmup_iterations;
  float cem_initial_action_stdev, cem_stdev_min;
  /* RPGD (reference optimizer_rpgd.py:148-179) */
  int32_t rpgd_outer_its, rpgd_first_iter_count, rpgd_resamp_per, rpgd_shift_previous, rpgd_keep_k;
  int32_t rpgd_distribution;      /* CTK_DIST_*                                                                  */
  int32_t rpgd_adam_form;         /* CTK_ADAM_*                                                                  */
  float rpgd_sample_mean, rpgd_sample_stdev, rpgd_sample_min, rpgd_sample_max;
  float rpgd_learning_rate, rpgd_gradmax_clip;
  double rpgd_beta_1, rpgd_beta_2, rpgd_epsilon;
  int32_t mlp_engine;             /* CTK_MLP_*                                                                   */
  int32_t cem_uniform_actions;    /* 1: random shooting (reference optimizer_random_action_tf.py:56-68): every tick samples
                                     Q ~ U[action_low, action_high) instead of N(dist_mue, stdev); use cem_outer_it = cem_best_k = 1 */
  int32_t rpgd_gradient_mode;     /* 0: RPGD.  1: population gradient descent (reference optimizer_gradient_tf.py:101-167): no ranking-based
                                     resampling; every tick all rows shift by one step and their last control is redrawn from
                                     U[action_low, action_high) (one draw per row); use period 1, keep_k = num_rollouts.
                                     2: CEM with one clipped gradient-descent step per sample before ranking (reference
                                     optimizer_cem_naive_grad_tf.py:58-114; u = first element of the refit mean).
                                     3: CEM with carried elites and one Keras-Adam step on the population per outer iteration
                                     (reference optimizer_cem_grad_bharadhwaj_tf.py:93-178; moments persist per row).
                                     Modes 2/3 read the cem_* fields (outer_it, best_k, initial_action_stdev, stdev_min, warmup*)
                                     and rpgd_learning_rate / gradmax_clip / beta / epsilon; period must be 1                  */
  int32_t num_clients;            /* 0 / 1: one client (the reference's controller).  2 .. 16: the handle carries that many independent
                                     MPPI clients -- own warm-start sequence, previous input, costs and Philox tick counter each -- whose
                                     ticks ctk_step_batch runs in ONE launch (SURVEY 8f.4; MPPI + ODE predictor, logging off, unsharded) */
  int32_t environment;            /* CTK_ENV_*                                                                    */
  int32_t rpgd_sample_whole_space; /* environments other than the CartPole: 1 = uniform RPGD draws over each input's own [low, high]
                                     (ctk_set_control_limits; reference sample_whole_control_space), 0 = over [rpgd_sample_min,
                                     rpgd_sample_max] for every input.  The CartPole reads rpgd_sample_min / max                  */
  int32_t reserved[2];
} ctk_config;

typedef struct ctk_handle ctk_handle;

/* ---- lifecycle ---------------------------------------------------------------------------------------------- */
/* replaces Optimizer(**kwargs) + optimizer.configure(...)  (controller_mpc.py:56-65,84-89)                       */
int ctk_create(const ctk_config *cfg, const ctk_ode_params *ode, const ctk_cost_params *cost, ctk_handle **out);
int ctk_destroy(ctk_handle *h);
/* replaces optimizer.optimizer_reset()  (controller_mpc.py:108-109; optimizer_mppi.py:227-231,
   optimizer_cem_tf.py:113-117, optimizer_rpgd.py:527-548).  RPGD draws its initial population here.             */
int ctk_reset(ctk_handle *h);
/* live cost / environment parameters (controller update_attributes, Controllers/__init__.py:106-107)            */
int ctk_set_cost_params(ctk_handle *h, const ctk_cost_params *cost);
int ctk_set_ode_params(ctk_handle *h, const ctk_ode_params *ode);
/* environments other than the CartPole: the flat parameter block of the environment's device functors (Dubins car: h, v_max,
   omega_max, dd_weight, obstacle_weight, cc_weight * R, ccrc_weight, terminal_weight, target_x, target_y, obstacle_x, obstacle_y,
   obstacle_r^2, MAX_COST), and the per-input control limits (template_optimizer stores action_low / action_high as [nu] tensors,
   Optimizers/__init__.py:42-44).  The ode / cost blocks of ctk_create are ignored for such handles.                            */
int ctk_set_env_params(ctk_handle *h, const float *p, int n);
int ctk_set_control_limits(ctk_handle *h, const float *low, const float *high, int nu);
int ctk_set_mlp_weights(ctk_handle *h, const ctk_mlp_weights *w);
/* recurrent predictor (CTK_PRED_GRU; MPPI and CEM): weights; the saved hidden state is zeroed.  Every MPPI tick ends with the
   reference's predictor.update(s, Q0 = new u_nom[0]) (optimizer_mppi.py:192,195-197) as one small kernel on the handle's stream;
   CEM never advances the state (optimizer_cem_tf.py has no such call).  CTK_STATE_RNN_H reads / writes the saved state.        */
int ctk_set_gru_weights(ctk_handle *h, const ctk_gru_weights *w);
/* run subsequent work on this cudaStream_t (0 = legacy default stream)                                          */
int ctk_set_stream(ctk_handle *h, void *cuda_stream);

/* ---- noise -------------------------------------------------------------------------------------------------- */
/* Injected-noise mode (verification): queue n standard draws z (N(0,1) or U[0,1), exactly the numbers a replay
   rng hands the reference at optimizer_mppi.py:173 / optimizer_cem_tf.py:64 / optimizer_rpgd.py:277,284), consumed
   in order by the following reset()/step() calls.  The buffer holds the draws of the GLOBAL population
   ([num_rollouts_global, ...]); a shard reads its own rows.  When the queue is empty the kernels generate
   Philox4x32-10 noise in-kernel (counter = draw block, global rollout id, tick, stream id; key = seed).          */
int ctk_push_injected_noise(ctk_handle *h, const float *z_host, size_t n);
int ctk_clear_injected_noise(ctk_handle *h);

/* ---- the hot path ------------------------------------------------------------------------------------------- */
/* replaces optimizer.step(s, time) (controller_mpc.py:104): one full tick, host in / host out.
   s_host [num_states]; u_out_host [num_control_inputs].  (Environments other than the CartPole: a plain launch sequence with one
   device->host copy of u; what follows describes the CartPole ticks.)  The call issues no cudaMemcpy and no stream synchronisation:
   the state travels inside the kernel parameters, the tick's last kernel stores u and a status word as tagged 8-byte
   slots (value | launch sequence number) into mapped pinned host memory, and the call polls the tags (a faulted or
   lost stream is detected through cudaStreamQuery after 50 ms; 60 s hard limit).  MPPI, CEM (unsharded populations up
   to one resident grid) and RPGD with num_rollouts <= 32 run the whole tick as ONE kernel launch.                  */
int ctk_step(ctk_handle *h, const float *s_host, float *u_out_host);
/* ctk_step plus the read-back of one [H] state array: CTK_STATE_U_NOM (MPPI u_nom; RPGD Q[best] before the shift,
   optimizer_rpgd.py:426) comes back through the same host mirror, CTK_STATE_CEM_MU / CEM_STD through one device->host copy.
   The plugin's step() returns u AND refreshes the warm-start sequence every tick
   (optimizer_mppi.py:220 optimal_control_sequence = u_nom).                                                         */
int ctk_step_state(ctk_handle *h, const float *s_host, float *u_out_host, int which, float *state_out_host, size_t n);
/* The same tick split for sharded (multi-GPU) use and for device-resident timing:
   ctk_step_local   : sample + rollout + cost + local reduction; asynchronous on the handle's stream; s_dev [ns].
   ctk_partials     : device pointer / float count of this shard's exchange record
                      (MPPI: [rho, a, b_z[n_ind]];  CEM: k x [cost, global id(as float bits), Q[H]]).
   ctk_step_finish  : combine `num_shards` records (laid out contiguously, device memory) and update the optimizer
                      state identically on every shard; writes u to u_out_dev [nu] (device) if not NULL.
   CEM runs cem_outer_it local/finish pairs per tick: ctk_step_local returns 1 while more iterations remain.      */
int ctk_step_local(ctk_handle *h, const float *s_dev);
int ctk_partials(ctk_handle *h, float **dev_ptr, size_t *n_floats);
int ctk_step_finish(ctk_handle *h, const float *gathered_dev, int num_shards, float *u_out_dev);

/* Asynchronous device-resident tick: s_dev [ns] and u_out_dev [2] (u, exchange status) stay on the device, nothing is
   synchronised.  With a connected exchange (below) every shard calls it once per tick; the whole tick -- rollouts,
   softmin record, NVLink record exchange, u_nom update -- is ONE kernel launch.  The status word (0: ok) is written by the
   CartPole MPPI tick and the one-launch CEM tick; the other ticks write u only (general environments: u_out_dev [nu]). */
int ctk_step_device(ctk_handle *h, const float *s_dev, float *u_out_dev);

/* n ticks back to back (states s_dev + i * s_stride floats, results [u, status] to u_out_dev + i * u_stride floats; u_out_dev may
   be NULL): one call enqueues the whole chain, consecutive ticks overlap through programmatic dependent launch -- the next tick's
   in-kernel noise generation runs underneath the previous tick's finish / exchange / launch gap.                          */
int ctk_step_device_n(ctk_handle *h, const float *s_dev, size_t s_stride, float *u_out_dev, size_t u_stride, int n);

/* ---- multi-client batching behind the serving edge (SURVEY 8f.4) ------------------------------------------------ */
/* replaces num_clients separate optimizer.step(s, time) calls of num_clients controllers (reference
   controller_server/controller_server.py:55-86 serves one ctrl.step per request): s_host [num_clients][num_states]; active
   [num_clients] (NULL: all) selects the clients that tick; u_out_host [num_clients] (entries of inactive clients untouched).  One
   kernel launch (grid.y = client); every client's tick is bit-identical to the tick of a single-client handle with the same
   configuration, seed and tick count.  Cost / ODE parameters are shared by the clients of a handle.                          */
int ctk_step_batch(ctk_handle *h, const float *s_host, const int32_t *active, float *u_out_host);
/* a new client takes over slot `client`: warm-start sequence to mid-range, previous input and tick counter to zero              */
int ctk_reset_client(ctk_handle *h, int client);

/* ---- fused cross-GPU exchange (MPPI, SURVEY 8e) --------------------------------------------------------------- */
/* Each shard owns a mailbox in its HBM; peers store their softmin record (n_ind + 2 values, each packed with the tick's
   sequence number in one 8-byte store) straight into it over NVLink from inside the rollout kernel, and the last block
   of every shard combines the records -- no NCCL call, no extra launch.  One process per GPU: export the local
   mailbox as a 64-byte CUDA IPC handle, all-gather the handles with any host transport, connect.  One process driving
   several GPUs (tests): pass the mailbox pointers and device ordinals directly.  ctk_step / ctk_step_device then
   exchange; every shard must tick in lock step.  A peer that never delivers makes ctk_step fail after 2 s.           */
int ctk_exchange_export(ctk_handle *h, void *ipc_handle_out64);
int ctk_exchange_connect(ctk_handle *h, int rank, int world, const void *ipc_handles /* world x 64 bytes */);
int ctk_exchange_mailbox(ctk_handle *h, void **dev_ptr);
/* device-side barrier across the connected shards on the handle's stream (one tiny kernel: tagged flags through the mailboxes);
   bench.py aligns the shards with it BEFORE a timed tick, so that skew from outside the timed region is not measured inside  */
int ctk_exchange_barrier(ctk_handle *h);
int ctk_exchange_connect_ptrs(ctk_handle *h, int rank, int world, void *const *mailboxes, const int *devices);

/* ---- state / logs ------------------------------------------------------------------------------------------- */
int ctk_get_state(ctk_handle *h, int which, float *dst_host, size_t n);
int ctk_set_state(ctk_handle *h, int which, const float *src_host, size_t n);
int ctk_get_counter(ctk_handle *h, int which, int64_t *value);
int ctk_set_counter(ctk_handle *h, int which, int64_t value);
int ctk_get_log(ctk_handle *h, int which, void *dst_host, size_t n_bytes);
/* The same log, handed out as a VIEW of a handle-owned pinned host buffer (one device->host DMA at PCIe rate, no pageable
   staging, no first-touch page faults on a fresh destination): *host_ptr stays valid until the next ctk_get_log_view of the
   same log id, ctk_step or ctk_destroy.  Replaces the `.numpy()` hand-over of the logged tensors (reference
   optimizer_mppi.py:214-218, Controllers/__init__.py:159-178 copies them into the controller's own history).           */
int ctk_get_log_view(ctk_handle *h, int which, const void **host_ptr, size_t *n_bytes);
/* Optional top-M-only logging (SURVEY 8f.2; the producer it replaces is reference optimizer_mppi.py:214-218 / optimizer_cem_tf.py:
   104-108, the consumer Controllers/__init__.py:159-178): the m lowest-cost rollouts of the last tick, best first, ties to the
   lower index -- selected (K4) and gathered on the device.  idx_out [m] global rollout ids, J_out [m], Q_out [m,H,nu],
   traj_out [m,H+1,ns]; any pointer may be null; Q_out / traj_out need cfg.logging.  1 <= m <= min(num_rollouts, 512).          */
int ctk_get_log_top(ctk_handle *h, int m, int32_t *idx_out_host, float *J_out_host, float *Q_out_host, float *traj_out_host);
/* number of CUDA kernels this handle has launched since create (bench.py "gpu_launches")                         */
int ctk_get_launch_count(ctk_handle *h, int64_t *value);
/* template instantiation of this handle's last rollout-kernel launch, e.g. "mppi_ode_kernel<0,0,10,2,1024,0>" (the parity tests
   assert that the instantiation they pinned to the oracle is the one bench.py times); valid until the next step / destroy      */
const char *ctk_last_kernel(ctk_handle *h);
/* CUDA-event timing of the dominant kernel of a tick (the fused rollout kernel: K1 MPPI, K3 CEM, K6/K7 RPGD), used by
   bench.py for roofline.achieved.  enable(on) resets the accumulator; get() synchronises the stream and returns the
   summed duration and the number of timed launches since enable().                                                */
int ctk_enable_kernel_timing(ctk_handle *h, int on);
int ctk_get_kernel_timing(ctk_handle *h, double *ms_sum, int64_t *n_launches);
/* diagnostics: per-block phase timeline (globaltimer ns) of the last MPPI/ODE rollout-kernel launch, [grid][8] uint64   */
int ctk_debug_trace(ctk_handle *h, int enable, uint64_t *out_host, size_t n_u64, int *grid_out);
/* standalone nominal rollout of one control sequence (reference optimizer_mppi.py:199-202 predict_optimal_trajectory,
   optimizer_rpgd.py:382-386): s_host [ns], Q_host [H] -> traj_host [H+1, ns], summed stage cost (may be NULL).     */
int ctk_rollout_single(ctk_handle *h, const float *s_host, const float *Q_host, float *traj_host, float *summed_stage_cost);

/* ---- utilities ---------------------------------------------------------------------------------------------- */
const char *ctk_last_error(void);
int ctk_abi_version(void);
/* FP32 FMA-chain microbenchmark used as the measured FP32 roofline denominator (TFLOP/s)                         */
int ctk_fp32_peak(int device, double *tflops, double *sm_clock_mhz_est);
/* FP32 issue-rate microbenchmark: G thread-instructions/s for an instruction mix (1 FFMA with three register sources,
   2 FMUL, 3 FADD, 4 FFMA+FMUL alternating, 5 rollout-like mix); ctk_fp32_peak uses the uniform-operand FFMA form.       */
int ctk_fp32_microbench(int device, int variant, double *ginstr_per_s);
/* Philox self-test: fill dst_host with n standard normals (kind 0) / uniforms (kind 1) exactly as the kernels draw */
int ctk_philox_fill(int device, uint64_t seed, int kind, float *dst_host, size_t n);
/* Verification hook for the PRODUCTION (in-kernel noise) instantiations: the standard draws rows [row0, row0 + rows) of the noise
   block (stream, tick) of this handle -- same key, counters and device function as the kernels.  stream = CTK_STREAM_* | (outer
   iteration << 8); tick = CTK_COUNTER_TICK of the step that consumed the block (RPGD's initial population: the counter at
   ctk_reset).  dst_host [rows * per_rollout], row-major.  The oracle replays them through rng.normal / rng.uniform
   (optimizer_mppi.py:173, optimizer_cem_tf.py:64, optimizer_rpgd.py:277,284).                                          */
enum { CTK_STREAM_MPPI = 0, CTK_STREAM_CEM = 1, CTK_STREAM_RPGD_INIT = 2, CTK_STREAM_RPGD_RESAMPLE = 3 };
int ctk_philox_export(ctk_handle *h, uint32_t stream, int64_t tick, int per_rollout, int uniform, size_t row0, size_t rows,
                      float *dst_host);
/* standalone top-k (ties -> lower index), the kernel behind tf.argsort(...)[:k] (optimizer_cem_tf.py:73-74)      */
int ctk_topk(int device, const float *cost_host, int n, int k, int32_t *idx_out_host);

#ifdef __cplusplus
}
#endif
#endif /* CTK_B200_H */
