/*
 * mjrl_b200 -- C ABI of the B200-native NPG/TRPO/DAPG post-rollout update engine.
 *
 * The reference (aravindr93/mjrl) is pure Python and has no FFI of its own; the boundary it exposes
 * is Python duck-typing (SURVEY.md section 8b).  This header is the C ABI that sits *underneath*
 * the Python classes in mjrl_b200/ (which keep the reference signatures).  Every entry point below
 * cites the reference function(s) it replaces, relative to /root/reference/mjrl/.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types;
 *   - every call returns 0 on success, <0 on error (mjb_last_error() gives the text);
 *   - "host-or-device" float vectors go through cudaMemcpyDefault (UVA), either kind is accepted;
 *   - one engine per device; calls on one engine must not be concurrent (mjrl is single-threaded);
 *   - calls are asynchronous on the engine's stream unless they return host scalars/arrays
 *     (those synchronise the stream before returning);
 *   - no CPU fallback anywhere: a missing GPU / failed launch is an error code.
 */
#ifndef MJRL_B200_H
#define MJRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MJB_VERSION 1

typedef struct mjb_engine mjb_engine;

typedef struct mjb_config {
    int32_t device;          /* CUDA ordinal */
    int32_t obs_dim;         /* env_spec.observation_dim            (utils/gym_env.py:9-13)            */
    int32_t act_dim;         /* env_spec.action_dim  (<= 32)                                            */
    int32_t n_hidden;        /* 0 = LinearPolicy (policies/gaussian_linear.py:32), 2 = MLP              */
    int32_t hidden[2];       /* MLP hidden sizes (policies/gaussian_mlp.py:9), each <= 256              */
    int32_t vf_hidden[2];    /* MLPBaseline hidden sizes (baselines/mlp_baseline.py:12), each <= 256    */
    float   min_log_std;     /* policies/gaussian_mlp.py:10                                             */
    int64_t max_samples;     /* capacity: rollout + demo timesteps held by this rank                    */
    int32_t max_paths;       /* capacity: trajectories held by this rank                                */
    int32_t world_size;      /* data-parallel ranks (1 = single GPU)                                    */
    int32_t rank;
} mjb_config;

/* Scalars the reference logs after train_from_paths (algos/npg_cg.py:145-151, algos/trpo.py:129-135). */
typedef struct mjb_step_stats {
    double alpha, delta, kl_dist, surr_before, surr_after;
    double vpg_dot_npg;      /* g . x                                                                   */
    int32_t backtracks;      /* TRPO line-search shrinks (algos/trpo.py:108-120)                             */
    int32_t cg_iters_run;    /* FVPs actually evaluated (early exit of utils/cg_solve.py:19-20)         */
    float time_vpg_ms, time_npg_ms, time_eval_ms;   /* CUDA-event timings of the phases                */
    float fvp_kernel_ms_sum;  /* sum of CUDA-event durations of the FVP tile kernel launches of this step     */
    int32_t fvp_launches;
} mjb_step_stats;

/* Return statistics of the rollout batch (algos/batch_reinforce.py:188-195). */
typedef struct mjb_batch_stats {
    double mean_return, std_return, min_return, max_return;
    double adv_mean, adv_std;   /* pre-whitening advantage moments (population std)                     */
    int64_t n_samples_global;
} mjb_batch_stats;

enum { MJB_ALGO_NPG = 0, MJB_ALGO_TRPO = 1, MJB_ALGO_DAPG = 2 };
enum { MJB_BATCH_ROLLOUT = 0, MJB_BATCH_DEMO = 1 };

int  mjb_version(void);
const char* mjb_last_error(const mjb_engine* e);   /* e may be NULL: error of the last failed create  */

int  mjb_create(const mjb_config* cfg, mjb_engine** out);
void mjb_destroy(mjb_engine* e);
int  mjb_synchronize(mjb_engine* e);

/* ---- multi-GPU: one process per GPU; NCCL communicator owned by the engine -------------------- */
/* rank 0 obtains a 128-byte NCCL unique id, the host side broadcasts it (torch.distributed), every
 * rank calls mjb_comm_init.  All reductions below then all-reduce across ranks (SURVEY 8e).         */
int  mjb_comm_unique_id(void* id128);
int  mjb_comm_init(mjb_engine* e, const void* id128);
/* All-reduce over NVLink peer memory for the Fisher-vector products (one fused kernel: partial reduction + scatter to the
 * peers + rank-ordered sum; replaces reduce kernel + ncclAllReduce, SURVEY 8e collective (3)).  Every rank exports the
 * CUDA IPC handle (64 bytes) of its exchange buffer, the host side all-gathers them in rank order, every rank imports
 * the world x 64 bytes; mjb_p2p_enable(e, 1) must only be called once EVERY rank imported successfully (returns the
 * resulting state, 0 = NCCL path).  mjb_p2p_calls: fused all-reduces executed so far.                          */
int  mjb_p2p_export(mjb_engine* e, void* handle64);
int  mjb_p2p_import(mjb_engine* e, const void* handles);
int  mjb_p2p_enable(mjb_engine* e, int on);
long long mjb_p2p_calls(mjb_engine* e);

/* ---- trajectories in (samplers/core.py:85-92 path dicts; algos/batch_reinforce.py:180-182 concat) */
/* Per-path HOST pointers to float64 arrays exactly as the sampler delivers them: obs[i] -> (len[i],
 * obs_dim), act[i] -> (len[i], act_dim), rew[i] -> (len[i]).  rew may be NULL (demo paths).  Packs
 * path-order/time-order into device fp32 [N,obs]/[N,act] + fp64 rew through pinned staging.          */
int  mjb_batch_upload(mjb_engine* e, int which, int32_t n_paths, const double* const* obs,
                      const double* const* act, const double* const* rew, const int32_t* len,
                      const uint8_t* terminated);
/* Same, from already-concatenated host-or-device arrays (fp64 host layout of np.concatenate). */
int  mjb_batch_upload_flat(mjb_engine* e, int which, int32_t n_paths, const double* obs, const double* act,
                           const double* rew, const int32_t* len, const uint8_t* terminated);
/* Rollouts that already live on the device as batched arrays obs [n_traj][horizon][obs_dim], act [..][act_dim], rew
 * [n_traj][horizon] (float32, or float64 when is_f64) -- what the learned-model rollouts of
 * algos/model_accel/sampling.py:16-90 produce and algos/model_accel/model_accel_npg.py:107-127 would otherwise slice
 * into host path dicts.  len[i] <= horizon (NULL = all full) keeps a prefix of trajectory i (termination / truncation,
 * model_accel_npg.py:129-158).  Packed device-to-device into the rollout batch; no host copy of the samples. */
int  mjb_batch_upload_rollouts(mjb_engine* e, int32_t n_traj, int32_t horizon, const void* obs, const void* act,
                               const void* rew, int is_f64, const int32_t* len, const uint8_t* terminated);
/* Advantages computed elsewhere (callers of train_from_paths that bring path["advantages"]). */
int  mjb_batch_set_advantages(mjb_engine* e, const double* adv_concat);
/* Already-whitened advantages as the reference's CPI_surrogate / flat_vpg take them (fp32 after .float(),
 * algos/batch_reinforce.py:41); replaces the output of mjb_process_paths. */
int  mjb_batch_set_adv_white(mjb_engine* e, const float* adv_white);
/* Baseline predictions computed elsewhere (non-MLP baselines keep working on the host: their
 * predict(path) output, concatenated, fp32) -- consumed by mjb_compute_advantages. */
int  mjb_batch_set_baseline(mjb_engine* e, const float* base_concat);
/* Returns computed elsewhere (path["returns"], concatenated fp64) -- consumed by mjb_vf_fit. */
int  mjb_batch_set_returns(mjb_engine* e, const double* ret_concat);
/* which: MJB_BATCH_ROLLOUT / MJB_BATCH_DEMO = samples on this rank; 2 = rollout samples over all ranks */
int64_t mjb_batch_size(const mjb_engine* e, int which);

/* ---- returns / advantages (utils/process_samples.py:3-35) ----------------------------------- */
int  mjb_compute_returns(mjb_engine* e, double gamma);                 /* compute_returns :3-5        */
int  mjb_vf_predict(mjb_engine* e);                                    /* MLPBaseline.predict, all paths (baselines/mlp_baseline.py:97-105) */
/* Same, evaluated with the baseline as of the last COMPLETED fit and without joining a fit in flight: the reference
 * computes the advantages with the pre-fit baseline (batch_reinforce.py:98 runs before :108), so the agents may start
 * this step's fit (mjb_vf_fit_begin) first and call this afterwards. */
int  mjb_vf_predict_prefit(mjb_engine* e);
int  mjb_compute_advantages(mjb_engine* e, double gamma, double gae_lambda, int use_gae); /* :7-35    */
int  mjb_get_returns(mjb_engine* e, double* out);                      /* host-or-device, N doubles   */
int  mjb_get_baseline(mjb_engine* e, float* out);                      /* N floats                    */
int  mjb_get_advantages(mjb_engine* e, double* out);                   /* un-whitened, N doubles      */
int  mjb_get_adv_white(mjb_engine* e, float* out);                     /* after mjb_process_paths     */
/* concat + whitening + return statistics (algos/batch_reinforce.py:178-197) */
int  mjb_process_paths(mjb_engine* e, mjb_batch_stats* out);

/* ---- policy parameters (policies/gaussian_mlp.py:60-87; utils/fc_network.py:27-37) ---------- */
int  mjb_policy_dim(const mjb_engine* e);
int  mjb_policy_set_params(mjb_engine* e, const float* theta, int set_new, int set_old);   /* clamps log_std */
int  mjb_policy_get_params(mjb_engine* e, float* theta_out, int which_old);
int  mjb_policy_set_transforms(mjb_engine* e, const float* in_shift, const float* in_scale,
                               const float* out_shift, const float* out_scale, int which_old);

/* ---- the differentiable pieces -------------------------------------------------------------- */
/* CPI_surrogate + kl_old_new fused (algos/batch_reinforce.py:40-52, policies/gaussian_mlp.py:99-145);
 * out[0] = surrogate, out[1] = mean KL(old||new as the reference defines it). */
int  mjb_policy_eval(mjb_engine* e, double out[2]);
/* flat_vpg (algos/batch_reinforce.py:54-58); include_demo: DAPG gradient over rollout+demo with the
 * weights of algos/dapg.py:62-74 (lam = lam_0*lam_1^iter), already multiplied by sample_coef (:97-98). */
int  mjb_policy_vpg(mjb_engine* e, int include_demo, double demo_lam, float* g_out);
/* NPG.HVP (algos/npg_cg.py:62-81): F v + damping v.  idx (device-or-host int32, n_idx entries, global
 * sample indices) reproduces hvp_sample_frac<0.99 (:65-69); NULL = all samples. */
int  mjb_policy_fvp(mjb_engine* e, const float* v, float damping, const int32_t* idx, int64_t n_idx,
                    float* out);
/* cg_solve (utils/cg_solve.py:3-22) with the FVP above, entirely on device; b = last mjb_policy_vpg
 * result if b == NULL.  idx: optional [iters][n_idx] subsample indices. */
int  mjb_policy_cg(mjb_engine* e, const float* b, int iters, float damping, float residual_tol,
                   const int32_t* idx, int64_t n_idx, float* x_out);
/* One whole train_from_paths after process_paths: surrogate, VPG, CG, step size, update (+TRPO line
 * search), re-evaluation, old <- new (algos/npg_cg.py:109-142, algos/trpo.py:83-126, algos/dapg.py:92-121). */
int  mjb_policy_step(mjb_engine* e, int algo, double step_size_or_kl, double const_learn_rate,
                     int cg_iters, float damping, double demo_lam, const int32_t* hvp_idx, int64_t n_idx,
                     mjb_step_stats* out);
int  mjb_policy_last_vectors(mjb_engine* e, float* vpg_out, float* npg_out);   /* g and x of the last step */
/* hvp_sample_frac < 1 under data parallelism (algos/npg_cg.py:65-69, SURVEY 8e): the host draws GLOBAL sample indices,
 * every rank keeps the ones inside its own row range, so the per-iteration lists differ in length between ranks and
 * between iterations.  The index block of the NEXT mjb_policy_cg / mjb_policy_step call stays [iters][n_idx] (n_idx = the
 * row stride); n_each[i] <= n_idx says how many entries of row i are valid.  One-shot: consumed by that call. */
int  mjb_policy_set_hvp_lengths(mjb_engine* e, const int64_t* n_each, int iters);

/* ---- minibatch-Adam policy training: PPO-clip and behaviour cloning -------------------------- */
/* loss_kind: MJB_LOSS_PPO = -mean(min(LR A, clip(LR, 1-clip_coef, 1+clip_coef) A)) with LR = exp(LL - LL_old) on the whitened
 * advantages of mjb_process_paths and LL_old of the old parameters and transforms (algos/ppo_clip.py:48-55,88-97);
 * MJB_LOSS_BC_MLE = -mean(LL), MJB_LOSS_BC_MSE = mean((mu - a)^2) on the resident batch's actions
 * (algos/behavior_cloning.py:83-105,120-127).  Runs `steps` sequential torch.optim.Adam steps (lr, betas 0.9/0.999,
 * eps 1e-8, no weight decay) on theta_new, one minibatch of `batch` (<= 64) resident rows per step, rows idx[step][0..batch)
 * (host-or-device int32 [steps][batch]).  The whole chain is one kernel launch on one SM.  log_std is not clamped inside
 * the chain (the reference clamps in set_param_values after it); MSE leaves log_std and its Adam moments untouched (it has
 * no gradient, so torch's Adam skips it).  Afterwards mjb_policy_eval reports surr_after / kl_dist of the unclamped
 * parameters.  loss_out / clip_frac_out (nullable, host-or-device, steps floats): every step's minibatch loss and the
 * fraction of its rows whose gradient the PPO clip zeroed (0 for the BC losses).  Single GPU, MLP policy only. */
enum { MJB_LOSS_PPO = 0, MJB_LOSS_BC_MLE = 1, MJB_LOSS_BC_MSE = 2 };
int  mjb_policy_sgd(mjb_engine* e, int loss_kind, const int32_t* idx, int64_t steps, int batch, float lr, float clip_coef,
                    float* loss_out, float* clip_frac_out);
/* Adam state of the policy optimizer (torch.optim.Adam(policy.trainable_params), ppo_clip.py:46, behavior_cloning.py:42):
 * moments in the flat theta layout (d floats each, host-or-device) and the step count; it lives on the device and
 * persists across mjb_policy_sgd calls.  NULL / step < 0 leave that part unchanged. */
int  mjb_policy_adam_set(mjb_engine* e, const float* m, const float* v, int64_t step);
int  mjb_policy_adam_get(mjb_engine* e, float* m, float* v, int64_t* step);
/* Full-batch BC loss of theta_new over the resident batch (behavior_cloning.py:115-118,132-135: loss_before / loss_after);
 * loss_kind MJB_LOSS_BC_MLE or MJB_LOSS_BC_MSE.  Uses the old-policy cache buffers as scratch (the cache is rebuilt when
 * next needed). */
int  mjb_policy_bc_loss(mjb_engine* e, int loss_kind, double* out);
/* CUDA-event time of the last mjb_policy_sgd kernel (the whole chain). */
int  mjb_policy_sgd_timing(mjb_engine* e, float* last_ms);

/* FVP arithmetic: 1 (default where supported: 128x128 MLP, obs < 32, act <= 8) = tcgen05 tensor cores with two-term
 * fp16 operand splitting (hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM); 0 = the fp32 FMA tile kernel.
 * Returns 1 (not an error) when tensor cores were requested for a shape that only has the FMA kernel. */
int  mjb_policy_set_tensor_cores(mjb_engine* e, int on);

/* ---- MLP baseline (baselines/mlp_baseline.py, utils/optimize_model.py) ---------------------- */
int  mjb_vf_dim(const mjb_engine* e);
/* weights / Adam moments in nn.Sequential.parameters() order; step = optimizer step count. */
int  mjb_vf_set_state(mjb_engine* e, const float* w, const float* m, const float* v, int64_t step);
int  mjb_vf_get_state(mjb_engine* e, float* w, float* m, float* v, int64_t* step);
/* MLPBaseline.fit (mlp_baseline.py:61-95): epochs x (int(N/bs)-1) sequential Adam steps on MSE with
 * L2-in-gradient weight decay; perms = [epochs][N] host int32 permutations (np.random.permutation).
 * err_out (nullable) = {error_before, error_after} of return_errors=True (:74-83,:87-94). */
int  mjb_vf_fit(mjb_engine* e, const int32_t* perms, int epochs, int batch_size, float lr, float reg_coef,
                double err_out[2]);

/* The same fit, asynchronous: _begin launches the sequential chain on the engine's side stream (it only depends on
 * the returns, so it can run concurrently with mjb_policy_step on the remaining SMs); _end joins, refreshes the
 * predict weights and optionally evaluates error_after.  Any call that needs the baseline state joins implicitly. */
int  mjb_vf_fit_begin(mjb_engine* e, const int32_t* perms, int epochs, int batch_size, float lr, float reg_coef,
                      double* err_before);
int  mjb_vf_fit_end(mjb_engine* e, double* err_after);
/* Fit arithmetic: 1 (default) = the single-SM tcgen05 kernel where the shape allows (128x128 hidden, batch 64, input
 * features within the kernel's shared-memory budget); 0 = the single-CTA fp32-FMA kernel, which is also the fallback
 * for every shape the tensor-core kernel does not cover (utils/optimize_model.py:7-36 semantics in both). */
int  mjb_vf_set_tensor_cores(mjb_engine* e, int on);

/* ---- host helper ---------------------------------------------------------------------------- */
/* np.random.permutation(n) of numpy's global legacy RandomState, bit for bit: the minibatch order MLPBaseline.fit
 * draws per epoch (utils/optimize_model.py:22).  mt_key624 / mt_pos are numpy's MT19937 state
 * (np.random.get_state()[1:3]); they are advanced in place exactly as numpy would, so the caller writes them back
 * with np.random.set_state and every later draw of the program is unchanged.  Pure host code (no device needed);
 * 2-3x faster than numpy's element-wise loop, which sits on the critical path of the fit.  out: n int32. */
int  mjb_host_permutation(uint32_t* mt_key624, int32_t* mt_pos, int64_t n, int32_t* out);

/* ---- introspection for benchmarks ------------------------------------------------------------ */
/* CUDA events on the engine's stream (slots 0..7) so callers time on the device, not by wall clock. */
int  mjb_event_record(mjb_engine* e, int slot);
int  mjb_event_elapsed_ms(mjb_engine* e, int slot_a, int slot_b, float* ms);   /* synchronises on slot_b */
int64_t mjb_kernel_launches(const mjb_engine* e);        /* kernels launched by this engine so far    */
/* Host<->device traffic this engine has issued so far: bytes copied from host memory into the engine (trajectory
 * uploads, parameters, permutations ...), bytes copied back to host memory, and the number of trajectory uploads
 * (mjb_batch_upload / _flat calls that completed).  Benchmarks report per-step deltas of these counters. */
typedef struct mjb_transfer_stats_t { int64_t h2d_bytes, d2h_bytes, uploads; } mjb_transfer_stats_t;
int  mjb_transfer_stats(const mjb_engine* e, mjb_transfer_stats_t* out);
int  mjb_fvp_timing(mjb_engine* e, float* last_ms);       /* CUDA-event time of the last FVP kernel    */
/* CUDA-event time of the sequential Adam kernels of the last fit (all epochs), on the stream they ran on; joins a fit
 * in flight.  Divided by epochs x (N/batch - 1) it is the per-Adam-step latency of utils/optimize_model.py:24-35. */
int  mjb_vf_fit_timing(mjb_engine* e, float* last_ms);


/* ---- developer aids (used by tools/, not by the Python mirror) ---------------------------------- */
/* per-phase clock64 counters of the tensor-core fit kernel / of the linear-policy FVP kernel: enable = 1 arms the
 * counters, enable = 0 reads them back (16 values each) and disarms. */
/* ---- ridge-regression baselines on the resident batch (replaces the N-dependent part of LinearBaseline / QuadraticBaseline:
 * baselines/linear_baseline.py:11-60, baselines/quadratic_baseline.py:11-68).  kind 0 = linear features
 * [clip(o)/10 | 1 | al..al^4] (K = obs_dim + 5), kind 1 = linear + all products o_i o_j, i <= j (K = n + n(n+1)/2 + 5), al =
 * time step / 1000; float64 arithmetic on the fp32-resident observations.
 *   mjb_ridge_features : K.
 *   mjb_ridge_gram     : out[(K+1) x (K+1)] (host doubles, row-major) = Gram matrix of [F | returns], summed over the ranks:
 *                        F^T F = out[:K,:K], F^T y = out[:K,K], y^T y = out[K,K].  The K x K solve stays with the caller
 *                        (the reference's np.linalg.lstsq retry loop).
 *   mjb_ridge_predict  : F c for every resident sample into the baseline buffer (read by mjb_compute_advantages, returned by
 *                        mjb_batch_get); sq_err (nullable) = sum over all ranks of (returns - F c)^2.                       */
int  mjb_ridge_features(const mjb_engine* e, int kind);
int  mjb_ridge_gram(mjb_engine* e, int kind, double* out);
int  mjb_ridge_predict(mjb_engine* e, int kind, const double* coeffs, double* sq_err);

int  mjb_dev_vf_profile(mjb_engine* e, long long* out16, int enable);   /* enable: 1 arm, 0 read head CTA + disarm, 2 read K-split helper 0 */
int  mjb_dev_lin_profile(mjb_engine* e, long long* out8, int enable);

#ifdef __cplusplus
}
#endif
#endif /* MJRL_B200_H */
