/*
 * dppo_b200.h — C ABI of libdppo_b200.so: the B200-native (sm_100a) implementation of DPPO's
 * data-parallel hot path (DDPM chain sampling + PPO log-prob update + eps-MSE pre-train step).
 *
 * The reference (jamesmshihua/DiffusionPolicyOptimization) has no FFI / plugin layer: its boundary
 * is the Python object surface the agents call.  Each entry point below names the reference
 * method(s) it replaces (file:line relative to the reference root).  TensorFlow's tape + optimizer
 * cannot be kept (TF is not a dependency), so "loss -> gradient -> AdamW" is one entry point.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes.  Unless a parameter is documented as HOST, every
 *     pointer is a DEVICE pointer owned by the caller, row-major contiguous fp32 (int32 indices).
 *   - every call is asynchronous on the passed stream (a cudaStream_t cast to void*; NULL = the
 *     legacy default stream) except the *_host convenience calls, which synchronise that stream.
 *   - return value: 0 = OK, negative = error; dppo_last_error() returns a thread-local message.
 *   - a handle is bound to one GPU and is not thread-safe: one handle per rank / process.
 *   - there is no CPU fallback: without a usable CUDA device dppo_create fails.
 *
 * Shapes: Do = obs_dim*cond_steps, A = horizon_steps*action_dim, T = denoising_steps,
 *         K = ft_denoising_steps, H = actor_hidden, Hc = critic_hidden.
 */
#ifndef DPPO_B200_H
#define DPPO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPPO_ABI_VERSION 1

typedef struct dppo_handle dppo_handle;
typedef void* dppo_stream_t; /* cudaStream_t */

/* network ids for dppo_{set,get}_weights / dppo_actor_forward */
enum { DPPO_NET_ACTOR = 0, DPPO_NET_ACTOR_FT = 1, DPPO_NET_CRITIC = 2, DPPO_NET_ACTOR_EMA = 3 };
/* activation ids: model/common/mlp.py:6-14 (only the two any cfg uses) */
enum { DPPO_ACT_RELU = 0, DPPO_ACT_MISH = 1 };
/* arithmetic of the MLP GEMMs */
enum {
    DPPO_PREC_FP32 = 0, /* CUDA-core FFMA everywhere: the parity mode (1e-4 rel / 1e-3 abs)        */
    DPPO_PREC_BF16 = 1, /* tcgen05 bf16 x bf16 -> fp32 for large row counts; fp32 master weights,
                           fp32 epilogues; looser bound stated in DESIGN.md                         */
    DPPO_PREC_BF16X3 = 2 /* tcgen05, every operand as bf16 hi + lo planes and every product as
                           hi*hi + lo*hi + hi*lo into one fp32 TMEM accumulator: meets the fp32
                           parity tolerance (1e-4 rel / 1e-3 abs) on the tensor pipe.  Covers action
                           chunks A = horizon_steps * action_dim <= 128; a wider chunk runs every
                           call on the FFMA path of DPPO_PREC_FP32                                  */
};
/* optimizer slots */
enum { DPPO_OPT_PRETRAIN = 0 /* actor */, DPPO_OPT_FINETUNE = 1 /* actor_ft ++ critic */ };

/* Hyper-parameters = cfg.model.* / cfg.train.* of cfg/gym/finetune/hopper-v2/ft_ppo_diffusion_mlp.yaml
 * and cfg/gym/pretrain/hopper-medium-v2/pre_diffusion_mlp.yaml.  dppo_cfg_default() fills the
 * hopper fine-tune values.
 * Accepted shapes (dppo_create refuses any other, naming the limit; dppo_num_params returns 0 for it):
 *   obs_dim, action_dim, horizon_steps, cond_steps >= 1;  1 <= denoising_steps <= 255;  0 <= ft_denoising_steps <= denoising_steps;
 *   time_dim even, 4 ... 64;  denoising_steps * time_dim <= 8192 (the time-embedding backward keeps 5 T time_dim floats in
 *   shared memory: 160 KB);  actor_hidden, critic_hidden multiples of 4, 16 ... 1024. */
typedef struct dppo_cfg {
    int32_t obs_dim, action_dim, horizon_steps, cond_steps;   /* yaml:16-22                        */
    int32_t denoising_steps, ft_denoising_steps;              /* yaml:18-19                        */
    int32_t time_dim;                                         /* mlp_diffusion.py:17  (16)         */
    int32_t actor_hidden, critic_hidden;                      /* yaml:93,102 (512 / 256)           */
    int32_t actor_act, critic_act;                            /* yaml:94,103 (ReLU / Mish)         */
    int32_t precision;                                        /* DPPO_PREC_*                       */
    float denoised_clip_value;      /* diffusion.py:28; < 0 = None                                 */
    float randn_clip_value;         /* yaml:83                                                     */
    float final_action_clip_value;  /* diffusion.py:30; < 0 = None                                 */
    float min_sampling_denoising_std, min_logprob_denoising_std; /* yaml:84-85                    */
    float gamma_denoising;          /* yaml:79                                                     */
    float clip_ploss_coef, clip_ploss_coef_base, clip_ploss_coef_rate; /* yaml:80-82             */
    float clip_vloss_coef;          /* diffusion_ppo.py:14; < 0 = None                             */
    int32_t norm_adv;               /* diffusion_ppo.py:17                                         */
    int32_t reward_horizon;         /* train_ppo_diffusion_agent.py:26 (= act_steps)               */
    float vf_coef;                  /* yaml:71                                                     */
    float logprob_clip_lo, logprob_clip_hi; /* diffusion_ppo.py:50-51 (-5, 2)                      */
    /* keras.optimizers.AdamW (Keras 3 semantics; train_ppo_agent.py:45-49, pretrain/train_agent.py:129-132) */
    float adam_beta1, adam_beta2, adam_eps;
    float weight_decay;             /* fine-tune optimizer (Keras default 0.004: `decay=` kwarg is ignored) */
    float pretrain_weight_decay;    /* pre_diffusion_mlp.yaml:29 (1e-6)                            */
} dppo_cfg;

int         dppo_abi_version(void);
const char* dppo_last_error(void);
void        dppo_cfg_default(dppo_cfg* cfg);
size_t      dppo_cfg_size(void); /* sizeof(dppo_cfg), for binding sanity checks */

/* DDPM constants — model/diffusion/sampling.py:7-17 + model/diffusion/diffusion.py:58-73.
 * HOST call, no GPU needed.  out is HOST [9*T]: rows betas, alphas_cumprod, sqrt_alphas_cumprod,
 * sqrt_one_minus_alphas_cumprod, sqrt_recip_alphas_cumprod, sqrt_recipm1_alphas_cumprod,
 * ddpm_logvar_clipped, ddpm_mu_coef1, ddpm_mu_coef2. */
int dppo_ddpm_schedule(int T, float* out);

/* number of fp32 parameters of a network; flat order = Keras variable-creation order:
 * actor  = [time Dense(2td) W[td,2td], b, time Dense(td) W[2td,td], b, input W[Din,H], b,
 *           block.l1 W[H,H], b, block.l2 W[H,H], b, output W[H,A], b]   (mlp_diffusion.py:40-62, mlp.py:117-132,170-171)
 * critic = [input W[Do,Hc], b, l1 W, b, l2 W, b, output W[Hc,1], b]       (critic.py:27-38)
 * Dense kernels are stored [in, out]. */
size_t dppo_num_params(const dppo_cfg* cfg, int net);

/* PPODiffusion.__init__ / VPGDiffusion.__init__ / DiffusionModel.__init__
 * (diffusion_ppo.py:8-30, diffusion_vpg.py:29-110, diffusion.py:19-100).  Weights start at zero. */
int  dppo_create(const dppo_cfg* cfg, int device, dppo_handle** out);
void dppo_destroy(dppo_handle* h);

/* set_weights / get_weights / load_weights / save_weights (diffusion.py:204-208,
 * finetune/train_agent.py:127-142).  `is_device` says whether src/dst is a device pointer;
 * host transfers synchronise the stream. */
int dppo_set_weights(dppo_handle* h, int net, const float* src, size_t n, int is_device, dppo_stream_t s);
int dppo_get_weights(dppo_handle* h, int net, float* dst, size_t n, int is_device, dppo_stream_t s);
/* AdamW moments + step counter of an optimizer slot (n = params covered by that slot). */
int dppo_set_opt_state(dppo_handle* h, int opt, const float* m, const float* v, size_t n, int64_t step, int is_device, dppo_stream_t s);
int dppo_get_opt_state(dppo_handle* h, int opt, float* m, float* v, size_t n, int64_t* step, int is_device, dppo_stream_t s);
/* VPGDiffusion.step(): set the number of fine-tuned denoising steps (diffusion_vpg.py:114-142). */
int dppo_set_ft_denoising_steps(dppo_handle* h, int K);
/* Per-variable gradient clipping of the fine-tuning update, train_ppo_diffusion_agent.py:349-354:
 * `[tf.clip_by_norm(g, clip_norm) for g in gradients]` (each Dense kernel / bias on its own: g * c / max(||g||_2, c)),
 * applied after the data-parallel reduction and before AdamW.  clip_norm <= 0 switches it off (the default; no shipped
 * cfg sets max_grad_norm).  The reference passes the constant 1.0 whatever max_grad_norm is.  `grads_out` of the
 * ppo_step calls keeps returning the unclipped gradient (what tape.gradient returns). */
int dppo_set_grad_clip_norm(dppo_handle* h, float clip_norm);

/* DiffusionMLP.call (mlp_diffusion.py:65-90): eps[N,A] = net(x[N,A], t[N] int32, obs[N,Do]). */
int dppo_actor_forward(dppo_handle* h, int net, const float* x, const int32_t* t, const float* obs,
                       int N, float* eps, dppo_stream_t s);

/* CriticObs.call (critic.py:40-54): v[N] = critic(obs[N,Do]). */
int dppo_value(dppo_handle* h, const float* obs, int N, float* v, dppo_stream_t s);

/* VPGDiffusion.call (diffusion_vpg.py:249-339): the whole T-step chain in one call.
 *   obs[B,Do]; actions[B,A]; chains_or_null[B,K+1,A].
 *   Noise: x_T_or_null[B,A] and noise_or_null[T,B,A] (row i = i-th loop iteration, t = T-1-i)
 *   inject the Gaussian draws (parity mode); when NULL they are drawn in-kernel by Philox4x32-10
 *   from (seed, offset, global row = row_offset + local row), so results do not depend on how
 *   rows are sharded across GPUs.
 *   min_sampling_std < 0 uses cfg.min_sampling_denoising_std. */
int dppo_sample(dppo_handle* h, const float* obs, int B, int deterministic, int use_base_policy,
                float min_sampling_std, uint64_t seed, uint64_t offset, int64_t row_offset,
                const float* x_T_or_null, const float* noise_or_null,
                float* actions, float* chains_or_null, dppo_stream_t s);
/* Env-side glue (SURVEY.md 8f.4).  dppo_set_env_normalization: the four arrays of the task's normalization.npz
 * (obs_min / obs_max [obs_dim], action_min / action_max [action_dim], host fp32), as loaded by
 * env/gym_utils/wrapper/mujoco_locomotion_lowdim.py:21-25.
 * dppo_rollout_step = one rollout step of agent/finetune/train_ppo_diffusion_agent.py:106-132 around RAW env data:
 *   raw_obs [E][cond_steps*obs_dim] float64 (device, or pinned host memory read through UVA) is normalised exactly like
 *   normalize_obs (:57-58) + the agent's fp32 cast (:111-113) into obs_out [E][Do] (device, e.g. obs_trajs[step]);
 *   the chain runs as in dppo_sample (actions [E][A] and chains on the device);
 *   raw_actions [E][act_steps*action_dim] fp32 (device, or pinned host memory) receives trajectories[:, :act_steps] (:121)
 *   un-normalised like unnormalize_action (:60-62) - written by the sampling kernel's own epilogue on the persistent
 *   cluster path (small env batches): two launches, no copy calls; the caller synchronises the stream and steps the envs. */
int dppo_set_env_normalization(dppo_handle* h, const float* obs_min, const float* obs_max, const float* action_min, const float* action_max);
int dppo_rollout_step(dppo_handle* h, const double* raw_obs, int E, int deterministic, int use_base_policy, float min_sampling_std,
                      uint64_t seed, uint64_t offset, int64_t row_offset, const float* xT, const float* noise,
                      float* obs_out, float* actions, float* chains, float* raw_actions, int act_steps, dppo_stream_t s);
/* Same call with HOST buffers (the reference caller passes NumPy and does np.array() on the result:
 * train_ppo_diffusion_agent.py:111-132).  H2D + kernel + D2H + stream sync inside. */
int dppo_sample_host(dppo_handle* h, const float* obs_host, int B, int deterministic, int use_base_policy,
                     float min_sampling_std, uint64_t seed, uint64_t offset, int64_t row_offset,
                     const float* x_T_host_or_null, const float* noise_host_or_null,
                     float* actions_host, float* chains_host_or_null, dppo_stream_t s);

/* VPGDiffusion.get_logprobs (diffusion_vpg.py:343-425): logp[B*K,A], row = b*K + k. */
int dppo_logprobs(dppo_handle* h, const float* obs, const float* chains, int B, int use_base_policy,
                  float* logp, dppo_stream_t s);
/* VPGDiffusion.get_logprobs_subsample (diffusion_vpg.py:427-481): logp[N,A]. */
int dppo_logprobs_subsample(dppo_handle* h, const float* obs, const float* chains_prev, const float* chains_next,
                            const int32_t* denoising_inds, int N, int use_base_policy, float* logp, dppo_stream_t s);

/* PPODiffusion.c_loss (diffusion_ppo.py:32-132) + tape.gradient + AdamW.apply_gradients
 * (train_ppo_diffusion_agent.py:340-356) in one call, on this rank's N_local rows.
 *   N_global   : rows of the whole (un-sharded) minibatch; all means divide by it.
 *   adv_mean/adv_std : population mean / std of `advantages` over the GLOBAL minibatch
 *                (diffusion_ppo.py:74-75); pass adv_std < 0 to have them computed on device from
 *                the local rows (valid only when N_local == N_global).
 *   apply      : 0 = loss + gradients only, 1 = also all-reduce (if a communicator is attached)
 *                and take the AdamW step with learning rate lr.
 *   metrics8   : DEVICE [8] = (pg_loss, entropy_loss, v_loss, clipfrac, approx_kl, ratio, bc_loss, eta)
 *   grads_or_null : DEVICE [n_actor + n_critic] flat gradient (after the all-reduce when apply=1). */
int dppo_ppo_step(dppo_handle* h, const float* obs, const float* chains_prev, const float* chains_next,
                  const int32_t* denoising_inds, const float* returns, const float* oldvalues,
                  const float* advantages, const float* oldlogprobs, int N_local, int64_t N_global,
                  float adv_mean, float adv_std, float lr, int apply,
                  float* metrics8, float* grads_or_null, dppo_stream_t s);
/* Same with HOST buffers; metrics8_host is HOST [8].  Synchronises the stream. */
int dppo_ppo_step_host(dppo_handle* h, const float* obs, const float* chains_prev, const float* chains_next,
                       const int32_t* denoising_inds, const float* returns, const float* oldvalues,
                       const float* advantages, const float* oldlogprobs, int N_local, int64_t N_global,
                       float adv_mean, float adv_std, float lr, int apply, float* metrics8_host, dppo_stream_t s);

/* Index-driven PPO update (SURVEY.md 8f.1).  The reference keeps one iteration's rollout as device tensors
 * (obs_k, chains_k, returns_k, values_k, advantages_k, logprobs_k: train_ppo_diffusion_agent.py:266-279) and assembles every
 * minibatch on the device from a shuffled flat index (tf.random.shuffle / unravel_index / gather / gather_nd, :287-312).
 * Here the rollout buffers stay resident in HBM (DEVICE pointers owned by the caller):
 *   obs_buf[P][Do], chains_buf[P][K+1][A] (the sampler's `chains` output), oldlogp_buf[P][K][A] (dppo_logprobs output),
 *   returns_buf[P], values_buf[P], adv_buf[P];  P = n_steps * n_envs.
 * inds_k[N] (DEVICE int32) holds flat (b * K + k) indices exactly like the reference's inds_k slice; row r of the
 * minibatch is (obs[b], chains[b][k], chains[b][k+1], k, returns[b], values[b], adv[b], oldlogp[b][k]).  The gather
 * runs in one kernel in front of dppo_ppo_step; everything else (N_global, adv_mean/adv_std, lr, apply, outputs) is as
 * for dppo_ppo_step (adv_std < 0: the statistics are computed over the gathered minibatch). */
int dppo_ppo_step_indexed(dppo_handle* h, const float* obs_buf, const float* chains_buf, const float* oldlogp_buf,
                          const float* returns_buf, const float* values_buf, const float* adv_buf, int64_t P,
                          const int32_t* inds_k, int N_local, int64_t N_global, float adv_mean, float adv_std, float lr, int apply,
                          float* metrics8, float* grads_or_null, dppo_stream_t s);
/* Same with the index list and the metrics in HOST memory (the only per-minibatch host traffic). */
int dppo_ppo_step_indexed_host(dppo_handle* h, const float* obs_buf, const float* chains_buf, const float* oldlogp_buf,
                               const float* returns_buf, const float* values_buf, const float* adv_buf, int64_t P,
                               const int32_t* inds_k_host, int N_local, int64_t N_global, float adv_mean, float adv_std, float lr, int apply,
                               float* metrics8_host, dppo_stream_t s);

/* GAE on the device (SURVEY.md 8f.2; agent/finetune/train_ppo_diffusion_agent.py:242-263): float64 backward scan per env,
 *   delta_t = r_t * reward_scale_const + gamma * V_{t+1} * (1 - terminated_t) - V_t
 *   A_t = delta_t + gamma * gae_lambda * (1 - terminated_t) * A_{t+1};   returns = A + V.
 * DEVICE pointers: rewards[S][E] float64 (env rewards are float64 NumPy in the reference), terminated[S][E] fp32 (0/1),
 * values[S][E] fp32 (dppo_value over the rollout observations), next_values[E] fp32 (dppo_value of the last observation);
 * advantages / returns [S][E] fp32, i.e. already in the flat (step, env) order the update indexes. */
int dppo_gae(dppo_handle* h, const double* rewards, const float* terminated, const float* values, const float* next_values,
             int n_steps, int n_envs, double reward_scale_const, double gamma, double gae_lambda,
             float* advantages, float* returns, dppo_stream_t s);

/* DiffusionModel.c_loss / p_losses / q_sample (diffusion.py:179-202) + tape.gradient + AdamW
 * (train_diffusion_agent.py:63-69) on net DPPO_NET_ACTOR.  t_or_null[N] int32 and
 * noise_or_null[N,A] inject the draws at diffusion.py:183,187; NULL = Philox(seed, offset, row).
 *   loss : DEVICE [1];  grads_or_null : DEVICE [n_actor]. */
int dppo_pretrain_step(dppo_handle* h, const float* actions, const float* obs, int N_local, int64_t N_global,
                       int64_t row_offset, const int32_t* t_or_null, const float* noise_or_null,
                       uint64_t seed, uint64_t offset, float lr, int apply,
                       float* loss, float* grads_or_null, dppo_stream_t s);
/* EMA.update_model_average (pretrain/train_agent.py:53-58): ema <- decay*ema + (1-decay)*actor. */
int dppo_ema_update(dppo_handle* h, float decay, dppo_stream_t s);

/* Multi-GPU (absent in the reference; SURVEY.md §8e): one handle per rank, weights replicated,
 * rows sharded by the caller, ONE sum all-reduce of [grads ++ metric partial sums] per step.
 * dppo_comm_unique_id fills HOST id[128] on rank 0; the caller broadcasts it (any transport) and
 * every rank calls dppo_comm_init.  NCCL is loaded with dlopen("libnccl.so.2"). */
int dppo_comm_unique_id(char* id128);
int dppo_comm_init(dppo_handle* h, const char* id128, int rank, int world);
/* Peer-memory path of that all-reduce (single node, NVLink / NVSwitch P2P): every rank exports CUDA IPC handles of its
 * two gradient buffers and of a flag array (dppo_comm_ipc_export fills HOST out[DPPO_IPC_BYTES]); the caller gathers the
 * blobs of all ranks (any transport) and hands the concatenation [world][DPPO_IPC_BYTES] to dppo_comm_ipc_attach.  From
 * then on `apply = 1` steps use ONE fused kernel instead of ncclAllReduce + AdamW: after a flag barrier over peer memory
 * every rank reads all ranks' gradients through P2P loads in the same rank order (bit-identical sums everywhere), applies
 * AdamW to its replica of the weights and keeps the reduced gradient / metrics.  Gradient buffers alternate between
 * steps, so the barrier of the next step also protects the buffer peers may still be reading.  world <= 8. */
#define DPPO_IPC_BYTES 192
int dppo_comm_ipc_export(dppo_handle* h, char* out);
int dppo_comm_ipc_attach(dppo_handle* h, const char* all_blobs, int rank, int world);

/* Count of kernel launches issued by this handle since creation (bench `gpu_launches`). */
int64_t dppo_launch_count(dppo_handle* h);
/* Health of the peer-memory gradient exchange (dppo_comm_ipc_attach): 0, or an error once a flag barrier timed out
 * (DPPO_PEER_TIMEOUT_S seconds, default 600): from then on the updates are skipped on the device, nothing traps. */
int dppo_comm_status(dppo_handle* h);
/* Of those, the tcgen05 GEMM launches (0 in DPPO_PREC_FP32 mode and below the row threshold). */
int64_t dppo_tc_launch_count(dppo_handle* h);
/* Of those, launches of the fused layer-chain kernel (whole MLP forward / backward / T-step sampler per launch). */
int64_t dppo_fused_launch_count(dppo_handle* h);
/* Which sampler the last dppo_sample used: 1 = persistent cluster kernel (one launch, T steps on
 * chip, fp32 FFMA; ReLU actors of width 256, 512, 768 or 1024 with chunks A <= 128 - other widths,
 * a Mish actor and wider chunks take 2), 2 = layer-by-layer fp32, 3 = layer-by-layer tcgen05,
 * 4 = fused tcgen05 chain (one launch, T steps on chip).  Test / bench introspection. */
int dppo_last_path(dppo_handle* h);
/* Test hook: 0 = automatic dispatch, 1 = force the cluster sampler, 2 = forbid it,
 * 3 = forbid the fused tcgen05 chain (the tensor path then runs one GEMM launch per layer). */
int dppo_force_path(dppo_handle* h, int path);
/* Live kernel timing for the roofline: when enabled, every GEMM-class launch (the MLP layers and
 * their gradients: >97% of the path's flops) is bracketed by CUDA events on the launching stream.
 * dppo_profile_read synchronises the device and returns the accumulated device time, launch count
 * and algorithmic flops (2*M*N*K per GEMM) since the last enable/reset. */
/* Test hook: one tcgen05 GEMM  out[M,N] = act(A*B + bias)  on bf16 device operands.
 * a_mn / b_mn = 0: operand is K-major (A stored [M][K], B stored [N][K]); 1: MN-major (A stored
 * [K][M], B stored [K][N]).  A2 (optional, same major as A, K2 columns) is K-concatenated to A.
 * out_f32 is [splits][M][N] partial sums (no bias/act when splits > 1); out_bf16 optional [M][N]. */
int dppo_debug_tc_gemm(dppo_handle* h, const void* A, int a_mn, int64_t lda, const void* A2, int64_t lda2, int K2,
                       const void* B, int b_mn, int64_t ldb, int M, int N, int K, int splits,
                       const float* bias, int act, float* out_f32, void* out_bf16, dppo_stream_t s);
/* Test hook: one split-precision tcgen05 GEMM (DPPO_PREC_BF16X3 arithmetic)  out[M,N] = A*B  on FP32 device operands:
 * each operand is split into `planes` (2 or 3) bf16 planes on the fly and the product is the sum of the plane products
 * (3 for two planes, 6 for three) with fp32 accumulation in tensor memory.
 * Majorness flags as in dppo_debug_tc_gemm; out_f32 is [splits][M][N] partial sums (splits is clamped to the k-blocks). */
int dppo_debug_split_gemm(dppo_handle* h, const float* A, int a_mn, int64_t lda, const float* B, int b_mn, int64_t ldb,
                          int M, int N, int K, int splits, int planes, float* out_f32, dppo_stream_t s);
/* Test hook: the CTA-pair plane GEMM (ts_path.cuh)  out = act(A*B + bias)  on FP32 device operands: A [M][K] K-major, B as
 * in dppo_debug_split_gemm, N a multiple of 64.  The kernel writes `planes` bf16 planes by TMA; out_f32 [M][N] receives
 * their sum, mask_out (optional, act == 1) the ReLU bit masks [M][N/32]. */
int dppo_debug_pair_gemm(dppo_handle* h, const float* A, int64_t lda, const float* B, int b_mn, int64_t ldb,
                         int M, int N, int K, int planes, const float* bias, int act, float* out_f32, uint32_t* mask_out, dppo_stream_t s);
/* Dev tool: per-CTA cycle counters of the fused chain kernel.  enable != 0 allocates them; out_host (optional)
 * receives HOST [16 launch slots][sm_count][8] (slot = chain launches since the last read, round robin) = {producer wait w_empty, mma wait x_full, mma wait w_full, mma total,
 * epilogue wait acc_full, epilogue generic layers, epilogue final layer, 0} of the last launch. */
int dppo_debug_chain_timing(dppo_handle* h, int enable, long long* out_host, int* sm_count);
/* Dev probe: tcgen05.mma issue cost, TMA round trip and TMA throughput per SM; see tools/mma_probe.py. */
int dppo_debug_mma_probe(dppo_handle* h, int grid, int mode, int iters, int N, int depth, long long* out_host);
/* Measurement aid for bench.py (the strict-fp32 mode's roofline denominator): sustained CUDA-core FFMA rate of this GPU in TFLOP/s -
 * 16 independent fmaf chains per thread, 2048 threads per SM, timed with CUDA events after a warm-up launch. */
int dppo_debug_ffma_peak(dppo_handle* h, double* tflops);
int dppo_profile_enable(dppo_handle* h, int on);
int dppo_profile_read(dppo_handle* h, double* gemm_ms, int64_t* gemm_launches, double* gemm_flops);
/* Tensor-pipe flops the launches of a class actually ISSUED (padded tiles; the plane modes issue 3 or 6 products per algorithmic
 * multiply-add), accumulated like the algorithmic count; call after dppo_profile_read_class (which synchronises). */
int dppo_profile_read_exec(dppo_handle* h, int cls, double* exec_flops);
/* Same, per kernel: 0 = fc::chain_kernel<512> (fused tcgen05 layer chain, actor width), 1 = tcgen05 GEMMs (grouped weight
 * gradients, per-layer fallback), 2 = FFMA SGEMM (fp32 parity mode), 3 = fc::chain_kernel<256> (Mish critic width).  flops are ALGORITHMIC (un-padded dims, SURVEY.md 8d). */
int dppo_profile_read_class(dppo_handle* h, int cls, double* ms, int64_t* launches, double* flops);

#ifdef __cplusplus
}
#endif
#endif /* DPPO_B200_H */
