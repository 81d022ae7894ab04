// Host-visible declarations of every kernel launcher in the engine (one CUDA TU each).
#pragma once
#include "mlp_kernel.cuh"

namespace mjb {

// Prepped layout for the linear policy: WT [K0P][AP] (transposed, zero padded), b [AP], log_std [AP].
struct LinLayout {
    int K0, K0P, A, AP;
    int oWT, ob, oLS, total;
    int tW, tb, tLS, d;
};

struct LinArgs {
    LinLayout L;
    const float* P;
    const float* T;
    const float* in_shift; const float* in_scale; const float* out_shift; const float* out_scale;
    const float* obs; const float* act; const int* idx; long long n;
    const float* weight; float* ll_old; float* mu_old; const float* old_log_std; int old_flags;
    double* eval_partial; float* gpartial; long long gstride;
};


inline LinLayout make_lin_layout(int K0, int A) {
    LinLayout L;
    L.K0 = K0; L.K0P = round_up(K0, kChunk); L.A = A; L.AP = round_up(A, 8);
    int o = 0;
    L.oWT = o; o += L.K0P * L.AP;
    L.ob = o;  o += L.AP;
    L.oLS = o; o += L.AP;
    L.total = round_up(o, 4);
    L.tW = 0; L.tb = A * K0; L.tLS = L.tb + A; L.d = L.tLS + A;
    return L;
}

// ---- mlp_h*.cu
cudaError_t launch_mlp_h32(int mode, const MlpArgs& args, int grid, cudaStream_t stream);
cudaError_t launch_mlp_h64(int mode, const MlpArgs& args, int grid, cudaStream_t stream);
cudaError_t launch_mlp_h128(int mode, const MlpArgs& args, int grid, cudaStream_t stream);
cudaError_t launch_mlp_h256(int mode, const MlpArgs& args, int grid, cudaStream_t stream);
int occupancy_mlp_h32(int mode, int YR);
int occupancy_mlp_h64(int mode, int YR);
int occupancy_mlp_h128(int mode, int YR);
int occupancy_mlp_h256(int mode, int YR);
inline int mlp_tile_rows_for(int H) { return H == 32 ? 256 : (H == 256 ? 64 : 128); }

// ---- linear_kernel.cu
cudaError_t launch_linear(int mode, const LinArgs& args, int grid, cudaStream_t s);

// ---- scan.cu : returns / GAE / whitening / packing helpers
void launch_f64_to_f32(const double* src, float* dst, long long n, cudaStream_t s);
void launch_tstep(const int* path_off, int n_paths, int* tstep, cudaStream_t s);
// device [n_traj][H][width] (float32 or float64) -> packed valid prefixes (float32 or float64) at row offsets path_off
void launch_pack_rollouts(const void* src, int is_f64, int H, int width, const int* path_off, int n_traj, void* dst, int dst_f64,
                          cudaStream_t s);
void launch_returns(const double* rew, const int* path_off, int n_paths, double gamma, double* ret, cudaStream_t s);
void launch_path_sums(const double* rew, const int* path_off, int n_paths, double* path_ret, cudaStream_t s);
void launch_advantages(const double* rew, const float* base, const double* ret, const int* path_off,
                       const unsigned char* terminated, int n_paths, double gamma, double gamma_lam,
                       int use_gae, double* adv, cudaStream_t s);
// out[0] = sum(x - shift), out[1] = sum((x - shift)^2) over n doubles (deterministic two-stage)
void launch_moments(const double* x, long long n, const double* shift_dev, double* scratch, double* out2,
                    cudaStream_t s);
// device-side finalisation of the statistics (no host round trip between the passes)
void launch_stats_finalize(const double* mom2, double inv_n, double* stats2, int mode, cudaStream_t s);
void launch_path_stats(const double* path_ret, int n_paths, double inv_paths_global, double* out4, int pass, cudaStream_t s);
// white[i] = float((adv[i]-mean)/(std+1e-6)); stats = {mean, std} on device
void launch_whiten(const double* adv, long long n, const double* stats, float* white, cudaStream_t s);
// DAPG weights (dapg.py:62-74): rollout w = 1e-2*white/(std(white)+1e-8), demo w = 1e-2*lam
void launch_dapg_weights(const double* adv, long long n, long long n_demo, const double* stats, double lam,
                         float* w, cudaStream_t s);

// ---- vecops.cu : parameter prep, partial reduction, CG vector updates
void launch_prep_mlp(const float* theta, const PrepLayout& L, float* out, cudaStream_t s);
void launch_prep_linear(const float* theta, const LinLayout& L, float* out, cudaStream_t s);
void launch_clamp_tail(float* theta, int d, int A, float lo, cudaStream_t s);
// out[i] = scale * sum_c partial[c][i]  (+ log_std block of the FVP: c(sigma) * v for i >= tLS)
void launch_reduce_partials(const float* partial, int grid, long long stride, int d, const double* scale_dev,
                            float* out, const float* theta, const float* v, int tLS, int fvp_ls_block,
                            const float* vscale2, cudaStream_t s);
void launch_reduce_eval(const double* partial, int grid, double* out2, cudaStream_t s);

// ---- p2p.cu : the same reduction fused with the all-reduce over NVLink peer memory (one kernel, no NCCL call)
struct P2PReduceArgs {
    const float* partial; int grid; long long stride; int d;      // as launch_reduce_partials
    const double* scale_dev; const float* theta; const float* v; int tLS; int fvp_ls_block; const float* vscale;
    float* out;
    unsigned long long* const* peers;   // device array [world]: exchange buffer of every rank (own one included), peer-mapped:
    int world, rank;                    //   64-bit words {call number : value} [2 parities][world][slot_words]
    int* cta_seq;                       // [ceil(d / 128)] per-CTA call counters (own memory)
    long long slot_words;
};
cudaError_t launch_reduce_allreduce_p2p(const P2PReduceArgs& a, cudaStream_t s);

// ---- ridge.cu : Gram matrix / predictions of the ridge-regression baselines (Linear, Quadratic) on the resident batch
struct RidgeArgs {
    const float* obs; const int* tstep; const double* ret; long long n; int obs_dim;
    int K;                        // features of the launch (Gram: the augmented count, features + returns column)
    const short2* ab;             // [K] per feature: the two tile columns whose product it is
    int tile_cols;                // obs_dim + 7: clip(o)/10 .., 1, al, al^2, al^3, al^4, y, 0
    double* partial; int splits; int nb;   // Gram only: block partials [splits][nb (nb + 1) / 2][64][64], nb = ceil(K / 64)
};
int ridge_blocks(int K);
cudaError_t launch_ridge_scale(const RidgeArgs& a, double* T, cudaStream_t s);      // T [n][tile_cols] float64
cudaError_t launch_ridge_gram(const RidgeArgs& a, const double* T, double* G, cudaStream_t s);
cudaError_t launch_ridge_predict(const RidgeArgs& a, const double* T, const double* coeff, int Kfeat, float* base,
                                 double* err_partial, int grid, cudaStream_t s);
// CG state lives on device: st = {rdotr, done_flag(as double), iters_run, g.x}
// vscale2 (nullable): also emit the power-of-two scale {s, 1/s} of the new search direction p (tensor-core FVP)
void launch_cg_init(const float* b, float* x, float* r, float* p, int d, double* st, float* vscale2, cudaStream_t s);
void launch_cg_update(const float* Fp, float damping, float tol, float* x, float* r, float* p, int d,
                      double* st, float* vscale2, cudaStream_t s);
void launch_dot(const float* a, const float* b, int d, double* out, cudaStream_t s);
void launch_axpy_clamp(const float* theta, const float* x, const double* alpha_dev, double alpha_scale,
                       int d, int A, float lo, float* out, cudaStream_t s);
void launch_scale(float* x, int d, float s_, cudaStream_t s);

// ---- fvp_tc.cu : tcgen05 / TMEM Fisher-vector product for the 128x128 MLP
size_t fvp_tc_prep_bytes();
bool fvp_tc_supported(const PrepLayout& L);
void launch_tc_prep(const float* theta, const PrepLayout& L, const float* scale_dev, unsigned char* out, cudaStream_t s);
void launch_tc_vscale(const float* v, int d, float* out2, cudaStream_t s);
cudaError_t launch_fvp_tc(const PrepLayout& L, const unsigned char* P, const unsigned char* T, const float* in_shift,
                          const float* in_scale, const float* out_scale, const float* obs, const int* idx, long long n,
                          float* gpartial, long long gstride, int grid, cudaStream_t s);

// ---- linear_tc.cu : tcgen05 Fisher-vector product of the linear policy (HBM-bound path)
size_t lin_tc_prep_bytes();
bool lin_tc_supported(int K0, int A);
void lin_tc_set_prof(unsigned long long* p);
// has_idx: the product will gather a subsample (selects the tangent layout of the kernel that will run)
void launch_lin_tc_prep(const float* v, int K0, int A, bool has_idx, const float* scale_dev, unsigned char* out, cudaStream_t s);
cudaError_t launch_linear_tc(const unsigned char* T, const float* theta, const float* in_shift, const float* in_scale,
                             const float* out_scale, bool identity_in, const float* obs, int K0, int A, const int* idx,
                             long long n, float* gpartial, long long gstride, int tW, int tb, int tLS, int grid, cudaStream_t s);

// ---- vf_fit.cu : sequential minibatch Adam of the value net
struct VfFitArgs {
    int K, H1, H2, obs_dim;           // K = obs_dim + 4
    const float* obs; const int* tstep; const double* returns; long long n;
    const int* perm;                  // [n] device permutation of this epoch
    int steps, batch;
    float lr, reg, beta1, beta2, eps;
    long long step0;                  // optimizer steps taken before this launch
    float* w; float* m; float* v;     // flat nn.Sequential order
    float* wT;                        // scratch: transposed copies W1T [K][H1], W2T [H1][H2]
    float* loss_out;                  // [steps] (optional)
};
cudaError_t launch_vf_fit(const VfFitArgs& a, cudaStream_t s);
// vf_fit_tc.cu : fp32 feature matrix + targets of the whole batch (built once per fit)
cudaError_t vf_build_features(const VfFitArgs& a, float* feat, float* ret32, cudaStream_t s);
// consts: caller-owned scratch of >= a.steps float4 (per-step Adam bias-correction constants, filled by the launcher)
// vf_fit_tc.cu : same chain on one SM with tcgen05 (units on the M axis, Adam moments of W2 in TMEM)
bool vf_tc_supported(int K, int H1, int H2, int batch);
void vf_tc_set_prof(long long* dev16);
int vf_tc_feat_pitch(int K);             // row pitch (floats) of the feature matrix vf_build_features writes
int vf_tc_sms(int K);                    // SMs (cluster CTAs) the tensor-core fit occupies: 1 + layer-1 K-split helpers
size_t vf_tc_scratch_bytes();            // global scratch of the K-split hand-offs
cudaError_t launch_vf_fit_tc(const VfFitArgs& a, const float* feat, const float* ret32, float4* consts, void* scratch, cudaStream_t s);
// err = sum((ret - pred)^2) / (sum(ret^2) + 1e-8) pieces: out = {sum err^2, sum ret^2} (fp32 casts like the reference)
void launch_vf_error(const double* ret, const float* pred, long long n, double* scratch, double* out2, cudaStream_t s);

// ---- policy_sgd.cu : sequential minibatch Adam of the Gaussian-MLP policy (PPO-clip, behaviour cloning)
enum { SGD_PPO = 0, SGD_BC_MLE = 1, SGD_BC_MSE = 2 };
struct PolicySgdArgs {
    int K0, h1, h2, A;                // real widths (K0 = obs_dim)
    int loss_kind;                    // SGD_*
    const float* obs; const float* act;            // resident batch rows
    const float* adv; const float* ll_old;         // PPO: whitened advantages, log-likelihood under the old policy
    const float* in_shift; const float* in_scale; const float* out_shift; const float* out_scale;
    const int* idx;                   // [steps][batch] rows of every minibatch
    long long steps; int batch;
    float lr, beta1, beta2, eps;
    float clip_lo, clip_hi;           // PPO: 1 - clip_coef, 1 + clip_coef
    long long step0;                  // optimizer steps taken before this launch
    float* theta; float* m; float* v; // flat reference layout, updated in place
    float* wT;                        // scratch: W1T [K0][h1], W2T [h1][h2], new W3 / b3 [A (h2 + 1)]
    float* loss_out;                  // [steps] minibatch loss (optional)
    float* clip_out;                  // [steps] fraction of rows whose gradient the clip zeroed (optional, PPO)
};
inline size_t policy_sgd_max_smem() { return 226 * 1024; }
size_t policy_sgd_smem_bytes(int K0, int h1, int h2, int A);
size_t policy_sgd_scratch_floats(int K0, int h1, int h2, int A);
cudaError_t launch_policy_sgd(const PolicySgdArgs& a, cudaStream_t s);
// out = sum over rows of ll (SGD_BC_MLE) or sum over rows x A of (mu - act)^2 (SGD_BC_MSE); scratch >= 128 doubles
cudaError_t launch_bc_loss_sum(const float* ll, const float* mu, const float* act, long long n, int A, int kind,
                               double* scratch, double* out, cudaStream_t s);

}  // namespace mjb
