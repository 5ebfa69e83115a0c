/*
 * dsact.h — C ABI of the B200-native DSAC-T update engine (libdsact.so).
 *
 * Drop-in boundary for ONE path of Jingliang-Duan/DSAC-v2: the per-step
 * critic/actor/temperature update over a replay minibatch,
 *     DSAC_V2.local_update(data, iteration)             reference dsac_v2.py:102-105
 * plus the replay minibatch gather that feeds it,
 *     ReplayBuffer.sample_batch(batch_size)             reference training/replay_buffer.py:85-90
 * called from OffSerialTrainer.step                      reference training/trainer.py:69,82.
 *
 * Conventions
 *  - plain C types only; every function returns 0 on success or a negative
 *    DSACT_E* code, and `dsact_last_error()` holds a message for the caller's thread;
 *  - the CALLER (PyTorch) owns every device allocation; the library borrows
 *    pointers handed over in `dsact_bind*` and never frees them;
 *  - all work is enqueued on the caller's CUDA stream (`cudaStream_t` passed as
 *    `void*`) and is asynchronous with respect to the host;
 *  - one handle per device and per trainer thread (not thread safe);
 *  - all tensors are fp32, row-major, contiguous unless a leading dimension is given.
 *
 * Flat parameter layout (`dsact_layout`): params = [ q1 | q2 | policy | log_alpha ],
 * targets = [ q1_target | q2_target | policy_target ]; each network is the
 * concatenation, in `state_dict` order (reference SURVEY §4 schema), of
 * weight_j [out_j, in_j] then bias_j [out_j].  grads / adam_m / adam_v mirror params.
 */
#ifndef DSACT_H
#define DSACT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSACT_ABI_VERSION 1
#define DSACT_MAX_HIDDEN 6
#define DSACT_NUM_STATS 16

enum {
  DSACT_OK = 0,
  DSACT_EINVAL = -1,   /* bad argument / unsupported configuration */
  DSACT_ECUDA = -2,    /* a CUDA runtime call failed */
  DSACT_ESTATE = -3,   /* call sequence error (e.g. step before bind) */
  DSACT_EARCH = -4     /* device is not sm_100 */
};

/* hidden activations, reference utils/common_utils.py:16-45 */
enum {
  DSACT_ACT_LINEAR = 0, DSACT_ACT_RELU = 1, DSACT_ACT_GELU = 2, DSACT_ACT_TANH = 3,
  DSACT_ACT_SIGMOID = 4, DSACT_ACT_ELU = 5, DSACT_ACT_SELU = 6
};

/* arithmetic of the dense layers */
enum {
  DSACT_GEMM_FP32 = 0,     /* fp32 FFMA, bit-comparable with the reference's fp32 path */
  DSACT_GEMM_BF16X3 = 1,   /* tcgen05 bf16 split-precision (hi*hi + hi*lo + lo*hi), fp32 accumulate */
  DSACT_GEMM_BF16 = 2      /* tcgen05 single-pass bf16, fp32 accumulate (throughput mode) */
};

/* What ApproxContainer.__init__ + DSAC_V2.__init__ read from kwargs
 * (reference dsac_v2.py:25-59,79-90; utils/common_utils.py:48-89). */
typedef struct dsact_config {
  int32_t abi_version;           /* = DSACT_ABI_VERSION */
  int32_t obs_dim;               /* obsv_dim */
  int32_t act_dim;               /* action_dim */
  int32_t n_hidden_q;            /* len(value_hidden_sizes) */
  int32_t n_hidden_pi;           /* len(policy_hidden_sizes) */
  int32_t hidden_q[DSACT_MAX_HIDDEN];
  int32_t hidden_pi[DSACT_MAX_HIDDEN];
  int32_t act_q;                 /* value_hidden_activation  */
  int32_t act_pi;                /* policy_hidden_activation */
  int32_t max_batch;             /* largest minibatch a step will see */
  int32_t auto_alpha;            /* dsac_v2.py:85 */
  int32_t delay_update;          /* dsac_v2.py:87 */
  int32_t gemm_mode;             /* DSACT_GEMM_* */
  int32_t use_graph;             /* replay captured CUDA graphs for repeated identical calls */
  int32_t act_dist;              /* policy_act_distribution: 0 TanhGaussDistribution, 1 GaussDistribution
                                    (utils/act_distribution_cls.py:20-79, 82-116) */
  /* scalars are doubles because the reference holds them as Python floats and forms
   * 1-beta, lr/(1-beta^t) ... in double before they touch an fp32 tensor */
  double gamma, tau, tau_b;       /* dsac_v2.py:82,83,90 */
  double alpha_fixed;             /* dsac_v2.py:86 (used when auto_alpha == 0) */
  double lr_q, lr_pi, lr_alpha;   /* dsac_v2.py:54-59 */
  double min_log_std, max_log_std;/* networks/mlp.py:73-74 */
  double adam_beta1, adam_beta2, adam_eps; /* torch.optim.Adam defaults 0.9 / 0.999 / 1e-8 */
} dsact_config;

typedef struct dsact_layout {
  int64_t n_q;          /* floats in one Q network */
  int64_t n_pi;         /* floats in the policy network */
  int64_t n_params;     /* 2*n_q + n_pi + 1 (log_alpha last) */
  int64_t n_targets;    /* 2*n_q + n_pi */
  int64_t workspace_bytes; /* activation / scratch arena the caller must provide */
  int64_t state_floats; /* persistent device state (EMA, counters, accumulators, stats) */
  int64_t max_batch;
} dsact_layout;

/* Device pointers of caller-owned tensors. */
typedef struct dsact_buffers {
  float *params, *targets, *grads, *adam_m, *adam_v;
  const float *act_high, *act_low;   /* [act_dim], policy.act_high_lim / act_low_lim */
  float *state;                      /* [state_floats], zero-initialised by the caller */
  void *workspace;                   /* [workspace_bytes], 256-byte aligned */
} dsact_buffers;

/* One replay minibatch, device pointers (the dict `data`, dsac_v2.py:219-225). */
typedef struct dsact_batch {
  const float *obs, *act, *rew, *obs2, *done;
  int32_t batch;
  const float *logp;  /* behaviour log-prob; stored and gathered like the reference does, never read by the update */
} dsact_batch;

/* The normal draws that affect an update (SURVEY Appendix B): eps1/eps2 [B,A]
 * for the two rsample() calls, z3/z4 [B] for the two target __q_evaluate calls.
 * Pass NULL instead of the struct to draw them on the device (Philox4x32-10). */
typedef struct dsact_noise {
  const float *eps1, *eps2, *z3, *z4;
} dsact_noise;

typedef struct dsact_handle dsact_handle;

const char *dsact_last_error(void);
int dsact_abi_version(void);

/* sizes implied by a configuration; no device needed */
int dsact_query_layout(const dsact_config *cfg, dsact_layout *out);

/* replaces ApproxContainer/DSAC_V2 construction (dsac_v2.py:25-59,79-90) */
int dsact_create(const dsact_config *cfg, int device, dsact_handle **out);
void dsact_destroy(dsact_handle *h);
int dsact_bind(dsact_handle *h, const dsact_buffers *bufs);

/* seed / counter of the device noise generator and of replay index sampling */
int dsact_seed(dsact_handle *h, uint64_t seed);

/* overwrite the carried scalars: mean_std1/2 (< 0 = "unset", dsac_v2.py:88-89),
 * Adam step counters of the critics and of policy/alpha */
int dsact_set_carry(dsact_handle *h, float mean_std1, float mean_std2,
                    int64_t adam_steps_q, int64_t adam_steps_pi, void *stream);

/* DSAC_V2.local_update (dsac_v2.py:102-105): gradients + Adam + delayed Polyak */
int dsact_step(dsact_handle *h, const dsact_batch *batch, const dsact_noise *noise,
               int64_t iteration, void *stream);

/* The same call with a HOST minibatch — what the reference's trainer hands to local_update (training/trainer.py:69,82:
 * `replay_samples` are CPU tensors): `host` holds host pointers (pinned for full PCIe rate; pageable works).  The five
 * arrays are copied into one of two internal device staging sets on a private copy stream (the copy of call k+1 runs
 * under the kernels of call k), then dsact_step runs on that set.  dsact_stage_host / dsact_stage_release are the two
 * halves for callers that want another entry point (dsact_dp_step, dsact_compute_grads ...) on a host minibatch:
 * stage -> device pointers in `dev` (valid until the second next stage call) -> any step call(s) on `dev` ->
 * release (marks the set reusable once the work enqueued on `stream` so far has finished). */
int dsact_step_host(dsact_handle *h, const dsact_batch *host, const dsact_noise *noise, int64_t iteration, void *stream);
int dsact_stage_host(dsact_handle *h, const dsact_batch *host, dsact_batch *dev, void *stream);
int dsact_stage_release(dsact_handle *h, void *stream);

/* split form = get_remote_update_info / remote_update (dsac_v2.py:107-138).
 * phase1: all forwards up to the per-critic sum of std over the local shard
 *         (state[DSACT_STATE_STDSUM..+1]); phase2: EMA, losses, all backward passes
 *         with loss means taken over `global_batch` rows.  A data-parallel caller
 *         all-reduces the two std sums between the phases and `grads` after phase2. */
int dsact_grad_phase1(dsact_handle *h, const dsact_batch *batch, const dsact_noise *noise, void *stream);
int dsact_grad_phase2(dsact_handle *h, int64_t global_batch, void *stream);
int dsact_compute_grads(dsact_handle *h, const dsact_batch *batch, const dsact_noise *noise, void *stream);
/* DSAC_V2.__update (dsac_v2.py:320-347) on whatever is in `grads` */
int dsact_apply(dsact_handle *h, int64_t iteration, void *stream);

/* tb_info (dsac_v2.py:188-202) of the last step, in this order:
 *  0 q1 mean, 1 q2 mean, 2 std1 mean, 3 std2 mean, 4 min std1, 5 min std2,
 *  6 actor loss, 7 critic loss, 8 mean tanh(policy mean), 9 mean policy std,
 * 10 entropy, 11 alpha (pre-update), 12 mean_std1, 13 mean_std2,
 * 14 data-parallel exchange status (0 = ok, 1 + r = rank r never arrived, see dsact_dp_step), 15 reserved.
 * Finalises the accumulators over `global_batch` rows and copies 16 floats to `host_out`
 * (pinned or pageable) asynchronously on `stream`. */
int dsact_read_stats(dsact_handle *h, int64_t global_batch, float *host_out, void *stream);

/* ---- device replay ring buffer (ReplayBuffer, training/replay_buffer.py:15-90) ---- */
typedef struct dsact_replay {
  float *obs, *obs2, *act, *rew, *done, *logp; /* [capacity, O], [capacity, O], [capacity, A], 3x [capacity] */
  int64_t capacity;
} dsact_replay;

int dsact_replay_bind(dsact_handle *h, const dsact_replay *rb);
/* store(): copy n transitions (rows of the staging arrays; host-pinned, pageable or device)
 * into rows (ptr + i) % capacity */
int dsact_replay_add(dsact_handle *h, const float *obs, const float *obs2, const float *act,
                     const float *rew, const float *done, const float *logp,
                     int64_t n, int64_t ptr, void *stream);
/* sample_batch(): gather rows idx[i] (device int64, or NULL = draw uniformly in [0,size) on
 * the device) into the engine's batch arena; `out` receives the arena's device pointers */
int dsact_replay_sample(dsact_handle *h, int32_t batch, int64_t size, const int64_t *idx,
                        dsact_batch *out, void *stream);
/* sample_batch + local_update in one submission (no host round trip in between) */
int dsact_replay_step(dsact_handle *h, int32_t batch, int64_t size, const int64_t *idx,
                      const dsact_noise *noise, int64_t iteration, void *stream);

/* ---- data-parallel replicas over NVLink peer memory (one process per GPU) ---------------------------------------
 * Replaces, for the same path, what `dsac-v2_b200/dp.py` does with three graph launches and four NCCL all-reduces
 * (reference: the reduction semantics of DSAC_V2.__compute_gradient, dsac_v2.py:150-206/233-241, under data
 * parallelism; the reference itself has no multi-GPU path, SURVEY.md 8e).  Set-up, once, on every rank:
 *   dsact_dp_export  -> allocate this rank's exchange buffer, return its CUDA IPC handle (DSACT_IPC_HANDLE_BYTES);
 *   (exchange the handles between the processes: any host transport, e.g. torch.distributed.all_gather_object)
 *   dsact_dp_connect -> map every peer's buffer (`handles` = world x DSACT_IPC_HANDLE_BYTES, rank order), reset epochs;
 *   (host barrier between the ranks).
 * Then dsact_dp_step / dsact_dp_replay_step = dsact_step / dsact_replay_step on this rank's shard, with the critic-std
 * sums, the gradients and the logged sums reduced over all ranks inside the step's own kernels (rank-ordered sums: the
 * replicas stay bit-identical).  `global_batch` = sum of the ranks' batch sizes.  A peer that never arrives makes
 * tb_info slot 14 non-zero (1 + its rank) after DSACT_DP_TIMEOUT_MS (default 10 s) instead of hanging the GPU. */
#define DSACT_IPC_HANDLE_BYTES 64
#define DSACT_DP_MAX_RANKS 8
int dsact_dp_export(dsact_handle *h, void *handle_out, int64_t *bytes_out);
int dsact_dp_connect(dsact_handle *h, int32_t rank, int32_t world, const void *handles);
int dsact_dp_step(dsact_handle *h, const dsact_batch *batch, const dsact_noise *noise, int64_t global_batch,
                  int64_t iteration, void *stream);
int dsact_dp_replay_step(dsact_handle *h, int32_t batch, int64_t size, const int64_t *idx, const dsact_noise *noise,
                         int64_t global_batch, int64_t iteration, void *stream);

/* ---- CNN approximators (BASELINE config 5, reference networks/cnn.py:30-53,151-240,383-461) --------------------------------
 * The same update path when value_func_type / policy_func_type = "CNN": every network is a private conv encoder
 * (Conv2d + ReLU per layer, no padding) followed by two separate MLP heads `mean` and `log_std` on the flattened
 * feature (the critics append the action to it).  Flat layout per network, in state_dict order: conv.{0,2,..}.weight
 * [Cout,Cin,k,k] / .bias, mean.{0,2,..}.weight / .bias, log_std.{0,2,..}.weight / .bias; params = [q1|q2|policy|log_alpha].
 * fp32 direct convolutions + the fp32 grouped GEMMs for the heads, eager launches.
 * dsact_cnn_step = DSAC_V2.local_update(data, iteration) with data["obs"] / ["obs2"] of shape [B, C, H, W] (contiguous).
 * The same head-wise engine also carries the variants of the reference that keep network outputs in separate heads or
 * need another loss, all in fp32: no encoder (n_conv = 0: the observation vector feeds the heads), one two-output head per
 * critic (q_heads = 1, networks/mlp.py), the policy's std types (pi_std), the plain Gaussian action distribution
 * (act_dist) and DSAC_V1 (algo = 1: ONE critic, flat layout [q | policy | log_alpha], dsac_v1.py). */
#define DSACT_MAX_CONV 8
typedef struct dsact_cnn_config {
  int32_t abi_version;
  int32_t channels, height, width;   /* obsv_dim = (C, H, W) */
  int32_t act_dim;
  int32_t n_conv;                    /* 0: no encoder, the observation (channels = obs_dim, height = width = 1) feeds the heads */
  int32_t conv_kernel[DSACT_MAX_CONV], conv_channels[DSACT_MAX_CONV], conv_stride[DSACT_MAX_CONV];
  int32_t n_hidden;                  /* hidden layers of every head MLP (networks/cnn.py:204 mlp_hidden_layers) */
  int32_t hidden[DSACT_MAX_HIDDEN];
  int32_t act_hidden;                /* DSACT_ACT_* of the head MLPs (the conv stack is ReLU) */
  int32_t max_batch, auto_alpha, delay_update;
  int32_t q_heads;                   /* 2: separate mean and std heads (networks/cnn.py:383-461); 1: one head with both outputs
                                        (networks/mlp.py:113-127, with n_conv = 0) */
  int32_t act_dist;                  /* 0 TanhGaussDistribution, 1 GaussDistribution (as in dsact_config) */
  int32_t pi_std;                    /* 0: log_std from its own head (networks/cnn.py, mlp.py std_type "mlp_separated");
                                        1: learnable row [1, act_dim] (mlp.py std_type "parameter"), laid out BEFORE the mean head;
                                        2: ONE head with 2 * act_dim outputs (mlp.py std_type "mlp_shared") */
  int32_t algo;                      /* 0: DSAC_V2 / DSAC-T (dsac_v2.py); 1: DSAC_V1 (dsac_v1.py:56-273): ONE critic, flat layout
                                        [q | policy | log_alpha], fixed TD bound */
  int32_t v1_bound;                  /* DSAC_V1 `bound` (dsac_v1.py:80): 1 = bounded loss (:219-229), 0 = Gaussian NLL (:231) */
  double gamma, tau, tau_b, alpha_fixed, lr_q, lr_pi, lr_alpha, min_log_std, max_log_std;
  double adam_beta1, adam_beta2, adam_eps;
  double td_bound;                   /* DSAC_V1 `TD_bound` (dsac_v1.py:79, default 20) */
} dsact_cnn_config;
typedef struct dsact_cnn_handle dsact_cnn_handle;
int dsact_cnn_query_layout(const dsact_cnn_config *cfg, dsact_layout *out);
int dsact_cnn_create(const dsact_cnn_config *cfg, int device, dsact_cnn_handle **out);
void dsact_cnn_destroy(dsact_cnn_handle *h);
int dsact_cnn_bind(dsact_cnn_handle *h, const dsact_buffers *bufs);
int dsact_cnn_set_carry(dsact_cnn_handle *h, float mean_std1, float mean_std2, int64_t adam_steps_q, int64_t adam_steps_pi,
                        void *stream);
int dsact_cnn_seed(dsact_cnn_handle *h, uint64_t seed);
int dsact_cnn_step(dsact_cnn_handle *h, const dsact_batch *batch, const dsact_noise *noise, int64_t iteration, void *stream);
/* Split form of dsact_cnn_step, with the contracts of dsact_grad_phase1 / _phase2 / dsact_compute_grads / dsact_apply
 * (get_remote_update_info / remote_update, dsac_v2.py:107-138, and data-parallel updates through torch.distributed):
 *  phase1: clears grads and accumulators, draws the noise on the device if `noise` is NULL, runs every forward; leaves
 *          the LOCAL per-critic sums of std in state[DSACT_STATE_STDSUM..+1].  The handle keeps the batch / noise
 *          pointers until the phase2 that follows, so they must stay valid until then;
 *  phase2: mean_std EMA, losses with means over `global_batch` rows (>= the phase-1 batch, else DSACT_EINVAL), every
 *          backward pass, the log_alpha gradient of the local rows, the EMA / temperature commit.  Without a preceding
 *          phase1: DSACT_ESTATE.  A data-parallel caller all-reduces the two std sums between the phases, and `grads`
 *          + the logged accumulators (16 sums, then 2 minima at DSACT_STATE_ACC + 16) after phase2;
 *  compute_grads = phase1 + phase2 with global_batch = the batch;
 *  apply: Adam on the three networks and log_alpha + delayed Polyak on whatever is in `grads` (it may have been
 *         overwritten by the caller), for `iteration`.
 * dsact_cnn_step = phase1 + phase2(batch) + apply, enqueued by the same code.  On a DSAC_V1 handle (algo = 1) the four
 * return DSACT_EINVAL. */
int dsact_cnn_grad_phase1(dsact_cnn_handle *h, const dsact_batch *batch, const dsact_noise *noise, void *stream);
int dsact_cnn_grad_phase2(dsact_cnn_handle *h, int64_t global_batch, void *stream);
int dsact_cnn_compute_grads(dsact_cnn_handle *h, const dsact_batch *batch, const dsact_noise *noise, void *stream);
int dsact_cnn_apply(dsact_cnn_handle *h, int64_t iteration, void *stream);
int dsact_cnn_read_stats(dsact_cnn_handle *h, int64_t global_batch, float *host_out, void *stream);
/* device replay ring for image transitions: rows of obs / obs2 are the flattened [C*H*W] images (fp32, like the
 * reference's CarRacing data, env_gym/gym_carracing_data.py:19-21); same semantics as dsact_replay_bind / _add / _sample */
int dsact_cnn_replay_bind(dsact_cnn_handle *h, const dsact_replay *rb);
int dsact_cnn_replay_add(dsact_cnn_handle *h, const float *obs, const float *obs2, const float *act, const float *rew,
                         const float *done, const float *logp, int64_t n, int64_t ptr, void *stream);
int dsact_cnn_replay_sample(dsact_cnn_handle *h, int32_t batch, int64_t size, const int64_t *idx, dsact_batch *out, void *stream);
/* The same ring with 8-bit images: obs / obs2 rows hold one uint8 code k per pixel, the pixel being float32(k) / 255.0f
 * (IEEE correctly-rounded division).  That is exact for observations on the 1/255 grid, such as the reference's
 * gym_carracingraw (rgb / 255, env_gym/gym_carracingraw_data.py:66-69), and takes a quarter of the fp32 ring's image bytes.
 * Callers encode k = rint(x * 255) and accept a pixel only if the decoded value equals x bit for bit; values off the
 * grid (e.g. gym_carracing's gray / 128 - 1) have no code and belong in the fp32 ring.  act / rew / done / logp stay fp32.
 *  bind_u8: a handle without a conv encoder (n_conv = 0: vector observations) gets DSACT_EINVAL.  Binding either kind
 *           replaces the ring bound before;
 *  add_u8:  dsact_cnn_replay_add's rows (ptr + i) % capacity with uint8 obs / obs2 staging.  On an fp32 ring it returns
 *           DSACT_ESTATE, and so does dsact_cnn_replay_add on an 8-bit ring;
 *  dsact_cnn_replay_sample gathers from whichever kind was bound last and decodes into the same fp32 minibatch arena.
 *           With idx = NULL it draws the same indices as on an fp32 ring (same seed and counter), so the two kinds of ring
 *           holding the same transitions return identical minibatches. */
typedef struct dsact_replay_u8 {
  uint8_t *obs, *obs2;                         /* [capacity, O] codes */
  float *act, *rew, *done, *logp;              /* [capacity, A], 3x [capacity] */
  int64_t capacity;
} dsact_replay_u8;
int dsact_cnn_replay_bind_u8(dsact_cnn_handle *h, const dsact_replay_u8 *rb);
int dsact_cnn_replay_add_u8(dsact_cnn_handle *h, const uint8_t *obs, const uint8_t *obs2, const float *act, const float *rew,
                            const float *done, const float *logp, int64_t n, int64_t ptr, void *stream);

/* introspection for tests/bench: number of kernel launches (graph nodes included)
 * submitted by this handle so far, and by the most recent entry-point call */
int64_t dsact_launch_count(const dsact_handle *h);
int32_t dsact_last_call_launches(const dsact_handle *h);

/* One eager (un-graphed) dsact_step with a CUDA event after every launch; per kernel class
 * [0 elementwise/other, 1 forward GEMM, 2 dgrad GEMM, 3 wgrad GEMM]: device milliseconds,
 * algorithmic FLOPs (2*M*N*K of every problem) and launch count.  Synchronises the stream. */
typedef struct dsact_profile {
  double ms[4], flops[4];
  int32_t launches[4];
  double total_ms;
} dsact_profile;
int dsact_profile_step(dsact_handle *h, const dsact_batch *batch, const dsact_noise *noise, int64_t iteration,
                       void *stream, dsact_profile *out);

/* raw dense-layer entry for unit tests of the GEMM kernels, in the handle's gemm_mode:
 *  variant 0 (forward): C[M,N]  = A[M,K] * B[N,K]^T (+ bias[N])
 *  variant 1 (dgrad)  : C[M,N]  = A[M,K] * B[K,N]
 *  variant 2 (wgrad)  : C[M,N] += A[K,M]^T * B[K,N]   (split-K, atomic accumulate) */
int dsact_test_gemm(dsact_handle *h, int32_t variant, const float *A, int32_t lda, const float *B, int32_t ldb,
                    const float *bias, float *C, int32_t ldc, int32_t M, int32_t N, int32_t K, void *stream);

#define DSACT_STATE_STDSUM 4   /* state[4], state[5]: local sums of critic std (phase1 -> phase2) */
#define DSACT_STATE_ACC 16     /* state[16..47]: per-step accumulators (sums first, then mins) */
#define DSACT_STATE_STATS 48   /* state[48..63]: finalised tb_info */
#define DSACT_STATE_ADAM 64    /* state[64..68]: Adam step sizes / bias corrections of the running step (internal) */
#define DSACT_STATE_DP_ERR 7    /* int32: 0, or 1 + rank of the peer a dsact_dp_step exchange timed out on */
#define DSACT_STATE_DP_EPOCH 15 /* int32: exchanges opened by dsact_dp_step so far (reset by dsact_dp_connect) */

#ifdef __cplusplus
}
#endif
#endif /* DSACT_H */
