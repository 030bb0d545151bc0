/*
 * b200rl.h -- C ABI of libb200rl.so: the PPO rollout -> GAE -> minibatch-update hot path of
 * Denys88/rl_games as hand-written sm_100a CUDA kernels.
 *
 * The reference (100% Python) has no FFI; this header is the boundary a maintainer would bind with
 * ctypes (see INTEGRATION.md).  Each entry point cites the reference code it replaces
 * (paths relative to the rl_games repo @ 262cf20).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns all memory,
 *     kernels never allocate or free;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), CUDA-graph capturable;
 *   - return value: 0 = OK, <0 = argument error (B200RL_E*), >0 = cudaError_t of the launch;
 *   - row-major tensors; "rows" of the experience arena are time-major: row(t, env) = t*N + env.
 *     The reference's flat sample index env*H + t (a2c_common.py:33-40 swap_and_flatten01) is
 *     preserved as an index MAPPING, never materialised: minibatch i = envs [i*mb/H, (i+1)*mb/H) x all t
 *     (datasets.py:75-82).
 */
#ifndef B200RL_H
#define B200RL_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RL_OK 0
#define B200RL_EINVAL (-1)
#define B200RL_EUNSUPPORTED (-2)
#define B200RL_ENOTBUILT (-3)

/* activation ids (network_builder.py:52-60 activations_factory) */
#define B200RL_ACT_NONE 0
#define B200RL_ACT_ELU 1
#define B200RL_ACT_RELU 2
#define B200RL_ACT_TANH 3

int b200rl_version(void);
/* compute capability the library was built for (100 => sm_100a) */
int b200rl_built_arch(void);
/* Programmatic dependent launch for the kernels of the per-minibatch chain (forward, backward 1/2, optimiser, post-step):
 * their CTAs may be scheduled while the predecessor kernel drains; each waits (griddepcontrol.wait) before touching any
 * memory of the chain.  Default off (measured slower than plain stream order on the c2 workload); returns the previous
 * setting.  Process-wide. */
int b200rl_set_pdl(int enable);

/* ---------------------------------------------------------------------------------------------
 * GAE.  Replaces rl_games/triton_kernels/gae_kernel.py:16-59 (_gae_kernel), :82-118 (_triton_gae)
 * and the eager loop :62-79; called from a2c_common.py:729-734 (discount_values).
 *   A_t = d_t + g*l*(1-done_{t+1})*A_{t+1},  d_t = r_t + g*V_{t+1}*(1-done_{t+1}) - V_t
 * rewards/values/advs: [H,N,V] with element strides (st_t, st_e, st_v); dones: [H,N] strides (st_t, st_e),
 * u8 (as stored by ExperienceBuffer, experience.py:392) or f32 (as the reference passes after .float()).
 * returns (optional, may be NULL): advs + values, same strides as advs (a2c_common.py:1060).
 * ------------------------------------------------------------------------------------------- */
int b200rl_gae_f32(const float* rewards, const float* values, const void* dones, int dones_is_u8,
                   const float* last_values, const void* last_dones, int last_dones_is_u8,
                   float* advs, float* returns,
                   int H, int N, int V,
                   int64_t r_st_t, int64_t r_st_e, int64_t r_st_v,
                   int64_t v_st_t, int64_t v_st_e, int64_t v_st_v,
                   int64_t d_st_t, int64_t d_st_e,
                   int64_t a_st_t, int64_t a_st_e, int64_t a_st_v,
                   double gamma, double tau, void* stream);

/* Kernel selection for dense [H,N] inputs with N % 16 == 0: 1 (default) = TMA-staged kernel (bulk copies of the tile into shared
 * memory, scan out of shared memory, bulk stores), 0 = register-chunk kernel.  Same results bit for bit.  Returns the previous value. */
int b200rl_gae_set_tma(int enable);

/* Fused GAE + returns + per-block moment partials for prepare_dataset (V == 1, contiguous [H,N]).
 * mask (optional f32 [H,N]) = autoreset validity (a2c_common.py:1002-1006).
 * partials: [gridDim][8] doubles {n, Sv, Sv2, Sr, Sr2, Sa, Sa2, pad}; *n_blocks_out_host receives grid size
 * (at most ceil(N / 64); ceil(N / 128) when max_partials is smaller than that). */
int b200rl_gae_fused_f32(const float* rewards, const float* values, const uint8_t* dones,
                         const float* last_values, const uint8_t* last_dones, const float* mask,
                         float* advs, float* returns, double* partials, int max_partials,
                         int H, int N, double gamma, double tau, int* n_blocks_out_host, void* stream);

/* ---------------------------------------------------------------------------------------------
 * prepare_dataset (a2c_common.py:1586-1660): value normaliser update (values THEN returns,
 * RunningMeanStd Chan merge running_mean_std.py:55-67, fp64 state + int64 count), normalise+clamp
 * values/returns (:69-114), advantage normalisation (A-mean)/(std_unbiased+1e-8) (:1634) or the masked
 * variant (torch_ext.py:172-191), advantages = returns - values (:1598).  Consumes the partials of
 * b200rl_gae_fused_f32 (or b200rl_batch_moments_f64 when the batch was materialised/edited by a caller).
 * vms_mean/vms_var: double[1], vms_count: int64[1] (updated in place unless freeze_stats).
 * ------------------------------------------------------------------------------------------- */
int b200rl_prepare_batch_f32(const float* values, const float* returns, const float* mask,
                             const double* partials, int n_partials,
                             double* vms_mean, double* vms_var, int64_t* vms_count,
                             float* old_values_n, float* returns_n, float* advs_n,
                             int B, int normalize_value, int normalize_advantage, int freeze_stats,
                             void* stream);

/* EMA advantage normaliser (GeneralizedMovingStats 'mean_std', moving_mean_std.py:84-150; a2c_common.py:473-475, :1622-1632):
 * advs holds the RAW advantages of all B rows (b200rl_prepare_batch_f32 with normalize_advantage = 0) and is normalised in place
 * with the updated state, clamped to [-5, 5].  partials: the same batch partial sums prepare_batch consumes.  ema_state: float[2]
 * {mean, mean of squares} (zeros initially), ema_step: int32[1] (1 initially).  training = 0: normalise only. */
int b200rl_adv_ema_normalize_f32(float* advs, int B, const double* partials, int n_partials, float* ema_state,
                                 int* ema_step, float decay, int training, void* stream);
int b200rl_batch_moments_f64(const float* values, const float* returns, const float* mask, double* partials,
                             int max_partials, int B, int* n_blocks_out_host, void* stream);

/* ---------------------------------------------------------------------------------------------
 * RunningMeanStd (running_mean_std.py:19-114) as standalone ops.
 * x: [R, D] rows given as n_chunks chunks of rows_per_chunk rows, chunk c starting at row c*chunk_stride.
 * moments_update: batch mean / biased var per feature merged into (mean f64[D], var f64[D], count i64[1])
 * (the training-mode forward of the obs normaliser never passes a mask: models.py:54-56); also refreshes
 * mean_f32[D] and std_f32[D] = sqrt(var_f32+eps).
 * scratch: double[scratch_blocks*2*D] work area, counter: int32[1] zero-initialised once.
 * ------------------------------------------------------------------------------------------- */
int b200rl_moments_update_f64(const float* x, int D, int rows_per_chunk, int n_chunks,
                              int64_t chunk_stride, double* mean, double* var, int64_t* count,
                              float* mean_f32, float* std_f32, float eps,
                              double* scratch, int scratch_blocks, int* counter, void* stream);
/* Observations do not change across mini-epochs, so the (shifted) batch sums of EVERY minibatch are computed once per
 * epoch in one pass over the arena (x: [H,N,D]); the per-minibatch training-mode update is then only the Chan merge.
 *  mbmom: double[n_mb][2*D]; mb_shift: float[D] (the running mean at call time); counters: int32[n_mb] zeroed once;
 *  scratch: double[scratch_blocks*2*D].  Requires D % 4 == 0 (else use b200rl_moments_update_f64 per minibatch). */
int b200rl_obs_mb_moments_f64(const float* x, int D, int H, int N, int envs_per_mb, const double* run_mean,
                              double* mbmom, float* mb_shift, double* scratch, int scratch_blocks, int* counters, void* stream);
int b200rl_obs_stats_merge_f64(const double* mbmom_i, const float* mb_shift, int D, int n_rows, double* mean, double* var,
                               int64_t* count, float* mean_f32, float* std_f32, float eps, void* stream);
/* mean_f32 = (float)mean, std_f32 = sqrt((float)var + eps): the fp32 copies the fused kernels consume */
int b200rl_refresh_norm_f32(const double* mean, const double* var, float* mean_f32, float* std_f32,
                            float eps, int D, void* stream);
/* y = clamp((x-mean)/sqrt(var+eps), -5, 5)  (denorm=0)   |   y = sqrt(var+eps)*clamp(x,-5,5)+mean  (denorm=1) */
int b200rl_normalize_f32(const float* x, float* y, const double* mean, const double* var, float eps,
                         int64_t rows, int D, int denorm, void* stream);

/* ---------------------------------------------------------------------------------------------
 * fp32 MLP building blocks (mixed_precision: False path).  network_builder.py:494-512.
 *   linear_fwd:  Y[M,Nout] = act( norm(X)[M,K] . W[Nout,K]^T + b )      (norm optional: models.py:54-56)
 *   linear_bwd_data:   dX[M,K] = (dY[M,Nout] . W[Nout,K]) * act'(A_prev)    (A_prev = activation output)
 *   linear_bwd_weight: dW_part[s*split_stride + ..][Nout,K] = dY_s^T . X_s ; db_part[s*split_stride + ..][Nout] = colsum(dY_s)
 * X rows may be chunked like in moments_update (arena, time-major); all other operands are dense.
 * ------------------------------------------------------------------------------------------- */
int b200rl_linear_fwd_f32(const float* X, int rows_per_chunk, int64_t chunk_stride, int64_t x_ld,
                          const float* norm_mean, const float* norm_std,
                          const float* W, const float* b, float* Y, int M, int K, int Nout, int act,
                          int accumulate /* Y = act(XW^T + b + Y) */, void* stream);
int b200rl_linear_bwd_data_f32(const float* dY, const float* W, const float* A_prev, float* dX,
                               int M, int K, int Nout, int act_prev, void* stream);
int b200rl_linear_bwd_weight_f32(const float* dY, const float* X, int rows_per_chunk, int64_t chunk_stride,
                                 int64_t x_ld, const float* norm_mean, const float* norm_std,
                                 float* dW_part, float* db_part, int64_t split_stride, int M, int K, int Nout,
                                 int n_splits, void* stream);
/* out[i] = sum_s part[s*split_stride + i]  (deterministic, fixed order) */
/* The same three building blocks on the 5th-gen tensor cores (tcgen05, bf16 operands rounded while they are staged, fp32 accumulate in
 * TMEM, fp32 bias / activation / outputs) for ANY layer width: the mixed_precision path of LSTM gate GEMMs and of MLPs the fused
 * kernels (b200rl_tc_mlp_*) have no geometry for.  Same arguments, same row / split semantics as the _f32 functions, plus W_bf16
 * (optional): a bf16 copy of W, same [Nout, K] row-major layout (b200rl_cast_bf16 of the flat parameter arena), staged without
 * conversion instead of the fp32 weights. */
int b200rl_cast_bf16(const float* src, void* dst_bf16, int64_t n, void* stream);
int b200rl_linear_fwd_tc(const float* X, int rows_per_chunk, int64_t chunk_stride, int64_t x_ld,
                         const float* norm_mean, const float* norm_std,
                         const float* W, const void* W_bf16, const float* b, float* Y, int M, int K, int Nout, int act,
                         int accumulate, void* stream);
int b200rl_linear_bwd_data_tc(const float* dY, const float* W, const void* W_bf16, const float* A_prev, float* dX,
                              int M, int K, int Nout, int act_prev, void* stream);
int b200rl_linear_bwd_weight_tc(const float* dY, const float* X, int rows_per_chunk, int64_t chunk_stride,
                                int64_t x_ld, const float* norm_mean, const float* norm_std,
                                float* dW_part, float* db_part, int64_t split_stride, int M, int K, int Nout,
                                int n_splits, void* stream);
int b200rl_reduce_splits_f32(const float* part, float* out, int n, int n_splits, int64_t split_stride, void* stream);

/* ---------------------------------------------------------------------------------------------
 * LSTM-with-dones cell (common/layers/recurrent.py:20-80 LSTMWithDones; gate order i,f,g,o; fp32).  The GEMM halves
 * run on b200rl_linear_*; these are the pointwise halves of the forward step and of its BPTT.
 *  cell_fwd: gates [S,4Hd] pre-activations -> activations in place; cin = already-masked c_{t-1}; writes c_out, h_out,
 *            optionally scatters h into an MLP-order buffer (row s -> (s/scatter_rpc)*scatter_stride + s%scatter_rpc) and the
 *            masked carries (h,c)*(1-done_next) for the next step (done_next rows chunk-mapped).
 *  cell_bwd: dh = dH[scatter row] + dhin_next*(1-done_next), dc = dcin_next*(1-done_next) -> dgates [S,4Hd], dcin [S,Hd].
 *  mask_rows: out[s] = in[chunk row s] * (1 - done[chunk row s])  (window-initial states; zeroing after episode ends,
 *             a2c_common.py:1150-1153)
 * ------------------------------------------------------------------------------------------- */
int b200rl_lstm_cell_fwd_f32(float* gates, const float* cin, float* c_out, float* h_out, float* h_scatter, int scatter_rpc,
                             int64_t scatter_stride, float* hin_next, float* cin_next, const uint8_t* done_next,
                             int done_rpc, int64_t done_stride, int S, int Hd, void* stream);
int b200rl_lstm_cell_bwd_f32(const float* gates_act, const float* c_t, const float* cin, const float* dH, int scatter_rpc,
                             int64_t scatter_stride, const float* dhin_next, const float* dcin_next, const uint8_t* done_next,
                             int done_rpc, int64_t done_stride, float* dgates, float* dcin, int S, int Hd, void* stream);
/* train-time reset flags of an RNN policy on a next_step-autoreset env (a2c_common.py:1180-1191):
 * out[t, n] = dones[t, n] | (t > 0 && valid[t - 1, n] == 0)   ([H, N] contiguous) */
int b200rl_rnn_train_dones_u8(const uint8_t* dones, const float* valid, uint8_t* out, int H, int N, void* stream);
int b200rl_rnn_mask_rows_f32(const float* in, int in_rpc, int64_t in_stride, float* out, const uint8_t* done, int done_rpc,
                             int64_t done_stride, int S, int Hd, void* stream);

/* ---------------------------------------------------------------------------------------------
 * PPO loss head.  Replaces a2c_continuous.py:97-134 (calc_losses), :241-257 (bound/reg loss),
 * common_losses.py:16-82, torch_ext.py:27-36 (policy_kl), :157-170 (apply_masks), models.py:335-364
 * (sigma=exp(logstd), neglogp, entropy) and the autograd of all of it w.r.t. mu, value, logstd and the
 * last hidden activation.  Rows are minibatch-local m in [0,M); arena tensors use the chunk mapping.
 * ------------------------------------------------------------------------------------------- */
typedef struct b200rl_loss_cfg {
    float e_clip;            /* config e_clip */
    float critic_coef;       /* config critic_coef */
    float bounds_loss_coef;  /* config bounds_loss_coef (0 if None) */
    int has_bounds_loss;     /* bounds_loss_coef is not None */
    int bound_loss_type;     /* 0 = none, 1 = 'bound', 2 = 'regularisation' */
    int clip_value;          /* config clip_value */
    int use_smooth_clamp;    /* config use_smooth_clamp */
    int ppo;                 /* config ppo (True) */
} b200rl_loss_cfg;

/* per-minibatch scalar outputs (f32 stats[B200RL_NSTATS]) */
#define B200RL_STAT_ALOSS 0
#define B200RL_STAT_CLOSS 1
#define B200RL_STAT_ENTROPY 2
#define B200RL_STAT_BLOSS 3
#define B200RL_STAT_KL 4
#define B200RL_STAT_SUMMASK 5
#define B200RL_STAT_CLIPFRAC 6
#define B200RL_STAT_LR 7      /* lr used for this minibatch's Adam step (written by adam) */
#define B200RL_STAT_GNORM 8   /* global grad norm before clipping (written by adam) */
#define B200RL_NSTATS 16

/* Head GEMM + loss forward + backward down to d(a_last).
 *  a_last [M,Hl] last hidden activation (output of act_last); W_head [A+1,Hl] (row 0 = value head,
 *  rows 1..A = mu head), b_head [A+1], logstd [A] (fixed sigma parameter).
 *  arena tensors (chunk-mapped rows): actions, old_mu, old_sigma [.,A]; old_values_n, returns_n,
 *  old_neglogp, advs_n, mask(optional) [.]
 *  inv_count_dev: device float = 1/max(sum(mask),1) for this minibatch (NULL => 1/M, unmasked).
 *  outputs: d_head [M, A+1] = (dL/dvalue, dL/dmu_0..A-1); d_alast [M,Hl]; new mu/sigma overwrite
 *  old_mu/old_sigma (datasets.py:33-43 update_mu_sigma); optional mu_out [M,A], value_out [M], neglogp_out [M];
 *  block partials [n_blocks][b200rl_loss_partial_stride()] doubles for b200rl_ppo_loss_finalize. */
int b200rl_ppo_head_loss_f32(const float* a_last, int Hl, const float* W_head, const float* b_head,
                             const float* logstd, const float* actions, float* old_mu, float* old_sigma,
                             const float* old_values_n, const float* returns_n, const float* old_neglogp,
                             const float* advs_n, const float* mask,
                             int rows_per_chunk, int64_t chunk_stride, int M, int A,
                             const b200rl_loss_cfg* cfg_host, const float* inv_count_dev,
                             float* d_head, float* d_alast, int act_last,
                             float* mu_out, float* value_out, float* neglogp_out,
                             double* partials, int max_partials, int* n_blocks_out_host, void* stream);
/* partials -> stats[] (means; masked means when inv_count was used) and d_logstd[A]
 * (includes the -entropy_coef * d(entropy)/d(logstd) term; entropy_coef read from device). */
int b200rl_ppo_loss_finalize(const double* partials, int n_partials, int A, const float* entropy_coef_dev,
                             float* stats, float* d_logstd, float* kl_out, void* stream);
/* b200rl_reduce_splits_f32 + b200rl_ppo_loss_finalize in one launch (the two tiny steps between backward and the
 * gradient all-reduce) */
int b200rl_reduce_finalize(const float* part, float* out, int n, int n_splits, int64_t split_stride,
                           const double* partials, int n_partials, int A, const float* entropy_coef_dev,
                           float* stats, float* d_logstd, float* kl_out, void* stream);
/* inv_count[i] = 1/max(sum_{t, e in minibatch i} mask[t,e], 1)  (torch_ext.py:157-170) */
int b200rl_mask_inv_counts_f32(const float* mask, int H, int N, int envs_per_mb, float* inv_count, void* stream);
int b200rl_loss_partial_stride(void);

/* ---------------------------------------------------------------------------------------------
 * Categorical (discrete-action) policy head -- SURVEY 8a row a15.  NOT YET RUN ON HARDWARE (see csrc/discrete.cu): the CPU
 * oracle (oracle/ppo_discrete_oracle.py) is pinned to the reference; these kernels are validated in the next round.
 *  b200rl_categorical_sample_f32: rollout head (models.py:95-125 eval branch; CategoricalMasked distributions.py:23-44):
 *    logits [N, ld] (K used), value_raw [N*value_ld], optional action_masks uint8 [N, K], one uniform per row from u_tape [N] or
 *    Philox(seed, *rng_epoch_dev, step_index, row); action = #{k : cdf_k <= u} clamped to the last action with p > 0;
 *    outputs actions int64 [N, n_heads], neglogp [N], values [N] (de-normalised when normalize_value), dones_out / valid_out
 *    bookkeeping as in b200rl_policy_head_sample_f32.  Multi-discrete (Tuple) spaces: the K logits / masks of a row are the
 *    concatenation of n_heads heads of head_sizes_host[j] actions (sum = K; n_heads = 0 or NULL: one head), one categorical and
 *    one uniform per head (u_tape [n_heads, N]), neglogp and entropy are sums over the heads (models.py:128-206).
 *  b200rl_categorical_loss_f32: training head (a2c_discrete.py:121-209): per-row neglogp / entropy / actor + critic loss,
 *    kl = 0.5 (old_neglogp - neglogp)^2, gradients d_logits [M, d_ld], d_value [M*dv_ld] of
 *    mean(a) + 0.5 critic_coef mean(c) - entropy_coef mean(H) (masked means when mask / inv_count_dev are given), and
 *    per-block partial rows of 8 doubles {w*a, w*c, w*H, w*kl, mask, mask*clipped, w, 0}.  Arena tensors (actions, action_masks,
 *    old_values_n, returns_n, old_neglogp, advs_n, mask) are addressed as chunk_row(m, rows_per_chunk, chunk_stride).
 * ------------------------------------------------------------------------------------------- */
typedef struct b200rl_cat_loss_cfg {
    float e_clip, critic_coef, entropy_coef;
    int clip_value, use_smooth_clamp, ppo;
} b200rl_cat_loss_cfg;
int b200rl_categorical_sample_f32(const float* logits, int ld, int K, int n_heads, const int* head_sizes_host,
                                  const float* value_raw, int value_ld,
                                  const uint8_t* action_masks, const float* u_tape, uint64_t seed,
                                  const uint64_t* rng_epoch_dev, uint32_t step_index, const double* vms_mean,
                                  const double* vms_var, int normalize_value, int64_t* actions, float* neglogp,
                                  float* values, const uint8_t* dones_cur, uint8_t* dones_out, const float* prev_dones,
                                  float* valid_out, int N, int values_only, void* stream);
int b200rl_categorical_loss_f32(const float* logits, int ld, int K, int n_heads, const int* head_sizes_host,
                                const float* values, int value_ld,
                                const int64_t* actions, const uint8_t* action_masks, const float* old_values_n,
                                const float* returns_n, const float* old_neglogp, const float* advs_n, const float* mask,
                                int rows_per_chunk, int64_t chunk_stride, int M, const b200rl_cat_loss_cfg* cfg_host,
                                const float* inv_count_dev, float* d_logits, int d_ld, float* d_value, int dv_ld,
                                double* partials, int max_partials, int* n_blocks_out_host, void* stream);

/* Value-only loss head of the central value network (central_value.py:276-301).  NOT YET RUN ON HARDWARE (see csrc/critic.cu).
 * loss = (masked) mean of critic_loss(old_values_n, values, e_clip, returns_n, clip_value); d_value[m*dv_ld] = its gradient;
 * arena tensors addressed as chunk_row(m, rows_per_chunk, chunk_stride); partial rows of 8 doubles {w*loss, mask, w, 0...}. */
int b200rl_value_loss_f32(const float* values, int value_ld, const float* old_values_n, const float* returns_n,
                          const float* mask, int rows_per_chunk, int64_t chunk_stride, int M, float e_clip, int clip_value,
                          const float* inv_count_dev, float* d_value, int dv_ld, double* partials, int max_partials,
                          int* n_blocks_out_host, void* stream);

/* Fused value head of the tensor-core critic (mixed_precision: True in central_value_config).
 *  b200rl_value_head_loss_f32 (training): a_last [M, Hl] (output of act_last), W_v [Hl], b_v [1], all fp32.
 *    v = W_v . a_last + b_v in fp32, then b200rl_value_loss_f32's loss, weights, chunk mapping and partial rows (one per 256 rows:
 *    {w*loss, mask, w, 0...}); d_alast [M, Hl] = dL/dv * W_v * act'(a_last); the head gradient goes into the split-partial arena
 *    (dW_part + s*split_stride [Hl], db_part + s*split_stride [1] for s < n_splits; sum with b200rl_reduce_splits_f32).  Optional
 *    value_out [M] receives v.  Deterministic (fixed-order sums, no atomics).  Hl <= B200RL_VALUE_HEAD_MAX_HL (else
 *    B200RL_EUNSUPPORTED).  Outputs need no initialisation.
 *  b200rl_value_head_fwd_f32 (rollout): values [N] = v of each row, de-normalised as b200rl_normalize_f32(denorm = 1, eps = 1e-5)
 *    when normalize_value; the dot product has the training kernel's summation order. */
#define B200RL_VALUE_HEAD_MAX_HL 4096
int b200rl_value_head_loss_f32(const float* a_last, int Hl, const float* W_v, const float* b_v, const float* old_values_n,
                               const float* returns_n, const float* mask, int rows_per_chunk, int64_t chunk_stride, int M,
                               float e_clip, int clip_value, const float* inv_count_dev, int act_last, float* d_alast,
                               float* value_out, float* dW_part, float* db_part, int64_t split_stride, int n_splits,
                               double* partials, int max_partials, int* n_blocks_out_host, void* stream);
int b200rl_value_head_fwd_f32(const float* a_last, int Hl, const float* W_v, const float* b_v, const double* vms_mean,
                              const double* vms_var, int normalize_value, float* values, int N, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimiser step.  Replaces a2c_common.py:493-514 (trancate_gradients_and_step: /world_size,
 * clip_grad_norm_, optimizer.step) + torch.optim.Adam(eps=1e-8, weight_decay, fused=True)
 * (a2c_continuous.py:44-48) + the adaptive-KL scheduler (schedulers.py:19-33, a2c_common.py:1557-1563)
 * with lr living in DEVICE memory so no .item() sync is needed per minibatch.
 *  state_d: double[4] = {lr, step, beta1^step, beta2^step} (zeros for the last two mean 'fresh'); double[6] when
 *    cfg->adaptive_lr is 2 or 3: [4], [5] = running KL sum / count of the current mini-epoch (zero-initialised);
 *  kl_dev: device f32 (summed over ranks; scaled by grad_scale inside), may be NULL.
 *  counter: int32[1] zero-initialised once.
 * ------------------------------------------------------------------------------------------- */
typedef struct b200rl_opt_cfg {
    double beta1, beta2, eps, weight_decay;
    double grad_norm;        /* config grad_norm (max norm) */
    double kl_threshold, min_lr, max_lr, lr_multiplier;
    double grad_scale;       /* 1/world_size applied to the (summed) gradient */
    int truncate_grads;      /* config truncate_grads */
    int adaptive_lr;         /* adaptive-KL schedule (schedulers.py:19-33) stepped on the device: 0 = off; 1 = after every
                              * optimiser step on this minibatch's KL (schedule_type 'per_minibatch'); schedule_type 'standard'
                              * (a2c_common.py:1565-1571, one step per mini-epoch on the mean KL): 2 = accumulate this KL,
                              * 3 = last minibatch of the mini-epoch: accumulate, step on the mean, reset */
} b200rl_opt_cfg;

/* optional fused refresh of the packed bf16 weight copy used by the tcgen05 kernels (b200rl_tc_pack_table) */
typedef struct b200rl_pack_table {
    int n_seg;
    int flat_off[4]; int rows[4]; int cols[4];
    uint32_t cs_bytes[4]; uint32_t dst_off[4];
} b200rl_pack_table;

/* optional tail of the optimiser kernels: training-mode obs-normaliser update for the NEXT minibatch from its precomputed
 * batch sums (== b200rl_obs_stats_merge_f64, folded into the last CTA to save a launch); mbmom == NULL or a NULL struct: off */
typedef struct b200rl_obs_merge {
    const double* mbmom; const float* shift; int D; int n_rows;
    double* mean; double* var; int64_t* count; float* mean_f32; float* std_f32; float eps;
} b200rl_obs_merge;

int b200rl_adam_step_f32(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int n,
                         double* state_d, const float* kl_dev, const b200rl_opt_cfg* cfg_host,
                         float* stats_out, int* counter, void* wpack, const b200rl_pack_table* tab_host,
                         const b200rl_obs_merge* merge_next_host, void* stream);

/* state_d[0] = adaptive-KL schedule(base_lr, *kl_dev * kl_scale): one scheduler step outside an optimiser launch (used once after a
 * checkpoint restore, where the reference's first step runs on the checkpoint's optimizer LR while its scheduler continues from the
 * agent's own last_lr: a2c_common.py:852-866) */
int b200rl_lr_schedule_apply(double* state_d, const float* kl_dev, double kl_scale, double base_lr,
                             const b200rl_opt_cfg* cfg_host, void* stream);

/* Single-GPU fused tail of one minibatch: b200rl_reduce_finalize + b200rl_adam_step_f32 in ONE launch (no second trip of
 * the reduced gradient through memory; one grid barrier, grid <= 148 co-resident CTAs).
 *  part: split partial gradients, entry i of split k at part[k*split_stride + i], valid for i in [A, n);
 *  entries [0, A) of the flat gradient (d_logstd) come from the loss partials.  grads[n] receives the reduced gradient.
 *  nrm_part: double[>= 148] scratch; grid_bar: uint64[1] zero-initialised once (monotonic 64-bit arrival counter: never reset, cannot wrap). */
int b200rl_reduce_adam_f32(const float* part, int n_splits, int64_t split_stride, const double* loss_partials,
                           int n_loss_partials, int A, const float* entropy_coef_dev, float* stats, float* kl_out,
                           float* grads, float* params, float* exp_avg, float* exp_avg_sq, int n, double* state_d,
                           const b200rl_opt_cfg* cfg_host, int* counter, double* nrm_part, int nrm_part_len, void* grid_bar,
                           void* wpack, const b200rl_pack_table* tab_host, const b200rl_obs_merge* merge_next_host,
                           void* stream);

/* Multi-GPU edition of b200rl_reduce_adam_f32: split reduction + gradient all-reduce over NVLink peer memory + clip + Adam in
 * ONE launch.  Each CTA publishes its slice of this rank's exchange buffer to the same CTA index on every peer through
 * per-CTA flags (peer_cta_flags_host[r]: rank r's uint64[world][160] flag array, my_cta_flags: this rank's, zero-initialised
 * once) and sums the slice over all ranks in fixed rank order.  peer_grads_host[r]: rank r's exchange buffer of THIS update's
 * parity (float[n + 1]: gradient + KL slot; the caller alternates two buffers by update parity).  red: float[n + 1] local. */
#define B200RL_PEER_FLAG_STRIDE 160
int b200rl_reduce_allreduce_adam_f32(const float* part, int n_splits, int64_t split_stride, const double* loss_partials,
                                     int n_loss_partials, int A, const float* entropy_coef_dev, float* stats,
                                     const void* const* peer_grads_host, void* const* peer_cta_flags_host, int world, int rank,
                                     void* my_cta_flags, void* seq_ptr, float* red, float* params, float* exp_avg,
                                     float* exp_avg_sq, int n, double* state_d, const b200rl_opt_cfg* cfg_host, int* counter,
                                     double* nrm_part, int nrm_part_len, void* grid_bar, void* wpack,
                                     const b200rl_pack_table* tab_host, const b200rl_obs_merge* merge_next_host, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU: fused gradient all-reduce + clip + Adam over NVLink peer memory (one launch per minibatch).
 * Replaces a2c_common.py:493-509 (cat -> all_reduce -> /world -> scatter), :1559-1561 (KL all-reduce) and the
 * optimiser step above.  Every rank's gradient arena (n floats + 1 KL slot) lives in a buffer obtained with
 * b200rl_ipc_alloc and mapped into every peer with b200rl_ipc_open (handles exchanged by the host, e.g. through
 * torch.distributed.all_gather_object).  peer_grads_host[r] / peer_flags_host[r]: device addresses (valid in THIS
 * process) of rank r's gradient buffer for this step's parity and of rank r's flag array (u64[world]);
 * my_flags == peer_flags_host[rank].  seq_ptr: u64[1] step counter, red: float[n+1] local reduced copy,
 * nrm_part: double[>= grid], grid_bar: u64[1] (zeroed once).  Gradient buffers must be double-buffered by step parity.
 * ------------------------------------------------------------------------------------------- */
int b200rl_ipc_alloc(int64_t bytes, void** dev_ptr_out_host, void* handle64_out_host);
int b200rl_ipc_open(const void* handle64_host, void** dev_ptr_out_host);
int b200rl_ipc_close(void* p);
int b200rl_ipc_free(void* p);
int b200rl_allreduce_adam_f32(const void* const* peer_grads_host, void* const* peer_flags_host, int world, int rank,
                              void* my_flags, void* seq_ptr, float* red, double* nrm_part, int nrm_part_len, void* grid_bar,
                              float* params, float* exp_avg, float* exp_avg_sq, int n, double* state_d,
                              const b200rl_opt_cfg* cfg_host, float* stats_out, int* counter, void* wpack,
                              const b200rl_pack_table* tab_host, const b200rl_obs_merge* merge_next_host, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Rollout.  a2c_common.py:985-1069 (play_steps) per-step pieces.
 * policy_head_sample: heads + sigma=exp(logstd) + a = mu + sigma*eps + neglogp + denorm value
 *   (models.py:329-364, :58-60) written straight into arena time-step t (experience.py:433-456).
 *   noise: optional [N,A] standard-normal draws; if NULL, Philox4x32-10 keyed by (seed, *rng_epoch_dev,
 *   step_index, env) is used (counter based => CUDA-graph replayable; bump *rng_epoch_dev once per epoch).
 *   env_actions (optional): clamp(a,-1,1) rescaled to [low,high] (a2c_common.py:1500-1510, :144-148).
 *   dones_out[e] = dones_cur[e] (a2c_common.py:1001); valid_out[e] = 1 - prev_dones[e] (:1002-1006).
 *   values_only != 0: just the (denormalised) value (get_values, a2c_common.py:603-626).
 * ------------------------------------------------------------------------------------------- */
int b200rl_policy_head_sample_f32(const float* a_last, int Hl, const float* W_head, const float* b_head,
                                  const float* logstd, const double* vms_mean, const double* vms_var,
                                  int normalize_value, const float* noise, uint64_t seed,
                                  const uint64_t* rng_epoch_dev, uint32_t step_index,
                                  float* actions, float* mus, float* sigmas, float* neglogp, float* values,
                                  float* env_actions, int clip_actions, const float* act_low, const float* act_high,
                                  const uint8_t* dones_cur, uint8_t* dones_out, const float* prev_dones,
                                  float* valid_out, int N, int A, int values_only, void* stream);

typedef struct b200rl_shaper_cfg {
    float scale_value, shift_value, min_val, max_val;  /* tr_helpers.py:16-42 */
    float gamma;
    int log_val;
    int value_bootstrap;     /* config value_bootstrap && 'time_outs' in infos */
} b200rl_shaper_cfg;

/* post env-step bookkeeping: shaped reward (+ gamma*V*timeout) stored at arena step t, self.dones,
 * episode accumulators and finished-episode means for the AverageMeters (torch_ext.py:326-352).
 *  ep_state: float[3][N] = current_rewards, current_shaped_rewards, current_lengths
 *  meter: double[8] = {mean_reward, mean_shaped_reward, mean_length, current_size, total_done, ...}
 *  valid_t (optional [N]): next_step-autoreset live rows (a2c_common.py:1027-1033)
 *  time_outs_kind: 0 none, 1 u8/bool, 2 f32.  scratch: double[scratch_blocks*4]; counter int32[1] zeroed once. */
int b200rl_post_step_f32(const float* rewards, const void* dones, int dones_is_u8, const void* time_outs,
                         int time_outs_kind, const float* values_t, const float* valid_t,
                         float* rewards_out_t, uint8_t* dones_cur, float* prev_dones_f32,
                         float* ep_state, double* meter, int games_to_track,
                         double* scratch, int scratch_blocks, int* counter, int N,
                         const b200rl_shaper_cfg* cfg_host, void* stream);

/* Synthetic on-GPU measurement env (SURVEY.md 8d; not part of the reference): obs ~ N(0,1) (Philox),
 * reward = -||a||^2, done = (t >= max_len) | Bernoulli(p_done), time_out = (t>=max_len) & !terminated. */
int b200rl_synth_env_step(const float* actions, float* obs, float* rewards, uint8_t* dones, uint8_t* time_outs,
                          int* ep_t, int N, int D, int A, int max_len, float p_done,
                          uint64_t seed, const uint64_t* rng_epoch_dev, uint32_t step_index, void* stream);
int b200rl_bump_u64(uint64_t* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * bf16 tensor-core MLP path (`mixed_precision: True`, the reference's default on bf16-capable GPUs:
 * a2c_common.py:429, a2c_continuous.py:173).  tcgen05.mma + TMEM accumulators + cp.async.bulk tile moves.
 * Network geometry supported by this build: MLP [256,128,64], A <= 15, and either obs dim <= 64 (BASELINE configs[1..2]: all
 * weights resident, b200rl_tc_supported() == 1) or 64 < obs dim <= 256 (BASELINE configs[4]; == 2: layer 1 runs in kernels of its
 * own -- the training forward / backward calls launch them internally, the rollout forward needs `l1_scratch`, a tiled bf16
 * buffer of n_tiles(N_rows) * tile_bytes[0]; xtile must be NULL).  0 = unsupported.  Weights are consumed from ONE packed bf16 copy (b200rl_tc_pack_weights) that
 * serves the forward (K-major view) and the dgrad (MN-major view).  act1/act2/act3/dhead/delta1/delta2 are
 * opaque tiled bf16 buffers: n_tiles(M) = ceil(M/128) tiles of b200rl_tc_tile_bytes() bytes each.  They, xtile and l1_scratch need no
 * initialisation: what they hold before the kernel that fills them runs (NaN included) reaches no result -- padded rows, padded units
 * and the d_head columns past the last action are written as zeros.
 *   fwd_train : trunk + heads + PPO loss fwd/bwd (same semantics / partial format as b200rl_ppo_head_loss_f32,
 *               finalise with b200rl_ppo_loss_finalize)
 *   fwd_rollout: trunk + heads + sample/neglogp/denorm-value epilogue (same semantics as b200rl_policy_head_sample_f32)
 *   bwd       : delta chain + all weight/bias gradients into part[n_parts][P] at the given flat offsets
 *               (sum with b200rl_reduce_splits_f32)
 * Geometry: three hidden layers u1 <= 256, u2 <= 128, u3 <= 64 (zero-padded to the compiled tile widths [256,128,64]; e.g.
 * [128,64,32]), observations D <= 64 (kind 1) or 64 < D <= 256 (kind 2: layer 1 in kernels of its own), up to 15 actions;
 * `activation` = B200RL_ACT_ELU / _RELU / _TANH, one for the whole MLP (network_builder.py:132 _build_mlp); each has its own
 * set of kernels (the activation is a compile-time constant of the epilogues).
 * ------------------------------------------------------------------------------------------- */
int b200rl_tc_supported(int D, int u1, int u2, int u3, int A);
int64_t b200rl_tc_pack_bytes(int D, int u1, int u2, int u3, int A);
int b200rl_tc_tile_bytes(int D, int u1, int u2, int u3, int A, int64_t* out4_host);
/* bytes of one 128-row tile of the normalised bf16 observation buffer (xtile) the training forward emits for the backward kernel
 * (the weight-gradient MMAs of layer 1 TMA-load it instead of re-deriving it from the fp32 observations; obs <= 64 only: with
 * pipelined_wgrad != 0 the two-stage-ring edition of the weight-gradient kernel runs instead); -1 if the geometry is unsupported */
int64_t b200rl_tc_xtile_bytes(int D, int u1, int u2, int u3, int A);
int b200rl_tc_pack_table(int D, int u1, int u2, int u3, int A, int off_W1, int off_W2, int off_W3, int off_Wh,
                         b200rl_pack_table* out_host);
int b200rl_tc_pack_weights(const float* W1, const float* W2, const float* W3, const float* W_head,
                           int D, int u1, int u2, int u3, int A, void* wpack, void* stream);
int b200rl_tc_mlp_fwd_train(const float* obs, int rows_per_chunk, int64_t chunk_stride, int D,
                            const float* norm_mean, const float* norm_std, const void* wpack,
                            const float* b1, const float* b2, const float* b3, const float* b_head, const float* logstd,
                            int u1, int u2, int u3, int activation, int M, int A,
                            const float* actions, float* old_mu, float* old_sigma, const float* old_values_n,
                            const float* returns_n, const float* old_neglogp, const float* advs_n, const float* mask,
                            const b200rl_loss_cfg* cfg_host, const float* inv_count_dev,
                            void* act1, void* act2, void* act3, void* dhead, void* xtile,
                            double* partials, int max_partials, int* n_blocks_out_host, void* stream);
int b200rl_tc_mlp_fwd_rollout(const float* obs, int D, const float* norm_mean, const float* norm_std, const void* wpack,
                              const float* b1, const float* b2, const float* b3, const float* b_head, const float* logstd,
                              int u1, int u2, int u3, int activation, int N_rows, int A,
                              const double* vms_mean, const double* vms_var, int normalize_value,
                              const float* noise, uint64_t seed, const uint64_t* rng_epoch_dev, uint32_t step_index,
                              float* actions, float* mus, float* sigmas, float* neglogp, float* values,
                              float* env_actions, int clip_actions, const float* act_low, const float* act_high,
                              const uint8_t* dones_cur, uint8_t* dones_out, const float* prev_dones, float* valid_out,
                              int values_only, void* l1_scratch, void* stream);
int b200rl_tc_mlp_bwd(const float* obs, int rows_per_chunk, int64_t chunk_stride, int D,
                      const float* norm_mean, const float* norm_std, const void* wpack,
                      int u1, int u2, int u3, int activation, int M, int A,
                      const void* act1, const void* act2, const void* act3, const void* dhead, const void* xtile,
                      int pipelined_wgrad, void* delta2, void* delta1, float* part, int max_parts, int P,
                      int off_W1, int off_b1, int off_W2, int off_b2, int off_W3, int off_b3, int off_Wh, int off_bh,
                      int* n_parts_out_host, void* stream);

/* tcgen05 bring-up / regression: D[128,N] = A[128,K] . B[N,K]^T (bf16 in, fp32 out) on the 5th-gen tensor cores.
 * a_mn / b_mn != 0: that operand is supplied transposed ([K,128] / [K,N]) and consumed through an MN-major
 * shared-memory descriptor (the view the weight-gradient MMAs use). */
int b200rl_tc_gemm_test(const void* A_bf16, const void* B_bf16, float* D, int N, int K, int a_mn, int b_mn, void* stream);

/* L2 flush helper for benchmarking: writes n u32 words. */
int b200rl_fill_u32(uint32_t* p, int64_t n, uint32_t v, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200RL_H */
