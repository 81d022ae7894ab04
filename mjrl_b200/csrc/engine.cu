// C-ABI implementation (include/mjrl_b200.h): device state, packing, orchestration of the tile kernels,
// device-resident CG, NPG/TRPO/DAPG step, baseline predict/fit, NCCL data parallelism.
// No CPU fallback: every entry point needs a CUDA device and returns <0 on failure.
#include <dlfcn.h>
#include <nccl.h>
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/mjrl_b200.h"
#include "kernels.h"

using namespace mjb;

namespace {

std::string g_create_error;

// ---- NCCL resolved at run time from the library torch already loaded (no link-time dependency) ----
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool load(std::string& err) {
        if (lib) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            lib = dlopen(n, RTLD_NOW | RTLD_NOLOAD);
            if (!lib) lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (lib) break;
        }
        if (!lib) { err = "cannot dlopen libnccl.so.2"; return false; }
#define MJB_SYM(field, name) \
    field = reinterpret_cast<decltype(field)>(dlsym(lib, name)); \
    if (!field) { err = std::string("missing NCCL symbol ") + name; return false; }
        MJB_SYM(GetUniqueId, "ncclGetUniqueId") MJB_SYM(CommInitRank, "ncclCommInitRank")
        MJB_SYM(CommDestroy, "ncclCommDestroy") MJB_SYM(AllReduce, "ncclAllReduce")
        MJB_SYM(Broadcast, "ncclBroadcast") MJB_SYM(GroupStart, "ncclGroupStart")
        MJB_SYM(GroupEnd, "ncclGroupEnd") MJB_SYM(GetErrorString, "ncclGetErrorString")
#undef MJB_SYM
        return true;
    }
};
NcclApi g_nccl;

struct ParamSet {           // one policy parameter set on device
    float* theta = nullptr;       // flat, reference layout
    float* prep = nullptr;        // kernel layout
    float* in_shift = nullptr; float* in_scale = nullptr; float* out_shift = nullptr; float* out_scale = nullptr;
    bool in_ident = true;         // in_shift == 0 and in_scale == 1 (the reference's default): kernels may skip the transform
};

}  // namespace

struct mjb_engine {
    mjb_config cfg;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream_vf = nullptr;      // side stream of the asynchronous baseline fit
    bool fit_in_flight = false;
    bool fit_reads_batch = false;          // the fit in flight reads obs / tstep / returns in place (FMA fallback kernel)
    std::string err;
    long long launches = 0;
    long long h2d_bytes = 0, d2h_bytes = 0, uploads = 0;   // host<->device traffic actually issued (mjb_transfer_stats)
    // ---- policy
    bool linear = false;
    int H = 0;
    PrepLayout PL;
    LinLayout LL;
    int d = 0, prep_total = 0, A = 0, tLS = 0;
    ParamSet pnew, pold;
    float* prep_tan = nullptr;
    // tensor-core FVP path (fvp_tc.cu): fp16 hi/lo pre-tiled copies of theta_new and of the tangent
    bool tc_ok = false, tc_on = true;
    unsigned char* tc_prep_new = nullptr; unsigned char* tc_prep_tan = nullptr; float* tc_vscale = nullptr;
    bool old_equals_new = true, old_cache_valid = false, transforms_equal = true;
    long long cache_rows = 0;
    // ---- batch
    long long cap = 0;
    float* obs = nullptr; float* act = nullptr; double* rew = nullptr;
    int* path_off = nullptr; unsigned char* term = nullptr; int* tstep = nullptr;
    long long n_roll = 0, n_demo = 0, n_glob_roll = 0;
    int n_paths = 0, n_glob_paths = 0;
    std::vector<int> h_path_off;
    double* ret = nullptr; double* adv = nullptr; float* base = nullptr; float* adv_white = nullptr;
    float* weights = nullptr; double* path_ret = nullptr;
    float* ll_old = nullptr; float* mu_old = nullptr;
    bool have_adv = false, have_white = false;
    // ---- scratch
    float* gpartial = nullptr; long long gstride = 0; int max_grid = 0;
    double* eval_partial = nullptr; double* mom_scratch = nullptr;
    double* dsc = nullptr;        // small device doubles, see enum below
    double* h_dsc = nullptr;      // pinned mirror
    float *g = nullptr, *x = nullptr, *r = nullptr, *p = nullptr, *Fp = nullptr, *tmpv = nullptr;
    int* idx_dev = nullptr; long long idx_cap = 0;
    void* pinned = nullptr; size_t pinned_bytes = 0;
    double* stage64 = nullptr; size_t stage64_elems = 0;
    int occ[4] = {0, 0, 0, 0};
    // ---- value net
    int vfH = 0; PrepLayout VPL; int vf_d = 0;
    float *vf_w = nullptr, *vf_m = nullptr, *vf_v = nullptr, *vf_wT = nullptr, *vf_prep = nullptr;
    long long vf_step = 0;
    float* vf_feat = nullptr; float* vf_ret32 = nullptr; long long vf_feat_cap = 0;   // fp32 features / targets of the fit
    int vf_tc_on = 1;         // fit kernel: 1 = single-SM tensor-core kernel where the shape allows, 0 = single-CTA FMA kernel
    int vf_sms = 1;           // SMs the fit kernel in flight occupies
    float4* vf_consts = nullptr; int vf_consts_cap = 0;   // per-step Adam constants of the fit kernels
    void* vf_ks = nullptr;    // hand-off scratch of the K-split tensor-core fit (obs_dim + 4 > 32)
    // ---- all-reduce over NVLink peer memory (p2p.cu): exchange buffer of this rank, peers' buffers opened through CUDA IPC
    unsigned long long* p2p_buf = nullptr; size_t p2p_bytes = 0;
    std::vector<void*> p2p_peer;              // [world] mapped base pointers (own buffer at [rank])
    unsigned long long** p2p_peer_dev = nullptr; int* p2p_seq = nullptr;
    long long p2p_slot = 0;
    bool p2p_ready = false, p2p_on = false;
    // ---- ridge baselines (ridge.cu)
    short2* ridge_ab = nullptr; int ridge_ab_kind = -1, ridge_K = 0;
    double* ridge_partial = nullptr; size_t ridge_partial_cap = 0;
    double* ridge_G = nullptr; size_t ridge_G_cap = 0;
    double* ridge_coeff = nullptr; double* ridge_err = nullptr;
    double* ridge_T = nullptr; size_t ridge_T_cap = 0;
    long long p2p_calls = 0;
    int* perm_dev = nullptr; long long perm_cap = 0;
    // global (all-rank) copies used by the replicated fit when world_size > 1
    float* fit_obs = nullptr; int* fit_tstep = nullptr; double* fit_ret = nullptr; long long fit_cap = 0;
    // ---- comm
    ncclComm_t comm = nullptr;
    // ---- timing
    cudaEvent_t ev[6];
    cudaEvent_t user_ev[8];
    static constexpr int kFvpRing = 128;
    cudaEvent_t fvp_ev[kFvpRing][2];
    long long fvp_count = 0;
    float last_fvp_ms = 0.f;
    // ---- CUDA graphs of the device-resident CG loop (one per distinct launch shape)
    struct CgGraph {
        long long n = 0; const int* idx = nullptr; long long n_idx = 0; int iters = 0; float damping = 0.f, tol = 0.f;
        int sms = 0; bool tc = false, p2p = false; cudaGraphExec_t exec = nullptr;
        std::vector<cudaEvent_t> ev;              // 2 per iteration: around the FVP tile kernel
    };
    std::vector<CgGraph> cg_graphs;
    std::vector<long long> hvp_len;               // per-iteration subsample lengths of the NEXT cg / step call (ragged, multi-GPU)
    bool graphs_on = true;
    const CgGraph* last_cg_graph = nullptr;       // set when the last CG ran as a graph (its events time the FVP launches)
    cudaEvent_t fit_ev[2] = {nullptr, nullptr};     // around the sequential Adam kernels of the last fit (on its stream)
    bool fit_timed = false;
    // ---- minibatch-Adam policy training (policy_sgd.cu): Adam moments / step count, index block, per-step outputs
    float *sgd_m = nullptr, *sgd_v = nullptr, *sgd_wT = nullptr;
    long long sgd_step = 0;
    int* sgd_idx = nullptr; long long sgd_idx_cap = 0;
    float* sgd_out = nullptr; long long sgd_out_cap = 0;  // [2][cap]: per-step loss, clip fraction
    cudaEvent_t sgd_ev[2] = {nullptr, nullptr};     // around the last policy_sgd kernel
    bool sgd_timed = false;
};

enum {  // slots in dsc
    DS_STATS = 0,      // adv mean, adv std
    DS_MOM = 2,        // moments scratch out (2)
    DS_SCALE = 4,      // 1/N_global_rollout, 1/world
    DS_SCALE_SUB = 6,  // 1/n_idx_global, 1/world
    DS_CG = 8,         // rdotr, done, iters, -
    DS_EVAL = 12,      // surr sum, kl sum
    DS_DOT = 14,       // g.x
    DS_ALPHA = 15,
    DS_CNT = 16,       // counts for all-reduce (4)
    DS_RET = 20,       // path-return stats: sum, sumsq, min, max, n
    DS_VF = 26,        // vf error sums (2)
    DS_TCSCALE = 28,   // FVP scale with the tangent's power-of-two pre-scale undone (2)
    DS_BCLOSS = 30,    // full-batch behaviour-cloning loss sum
    DS_TOTAL = 32
};

#define FAIL(e, msg) do { (e)->err = (msg); return -1; } while (0)
#define CK(e, call) do { cudaError_t _c = (call); if (_c != cudaSuccess) { \
    (e)->err = std::string(#call) + ": " + cudaGetErrorString(_c); return -1; } } while (0)
#define NK(e, call) do { ncclResult_t _c = (call); if (_c != ncclSuccess) { \
    (e)->err = std::string(#call) + ": " + g_nccl.GetErrorString(_c); return -1; } } while (0)

namespace {

int pad_hidden(int h) { return h <= 32 ? 32 : h <= 64 ? 64 : h <= 128 ? 128 : 256; }

cudaError_t launch_mlp_any(int H, int mode, const MlpArgs& a, int grid, cudaStream_t s) {
    switch (H) {
        case 32: return launch_mlp_h32(mode, a, grid, s);
        case 64: return launch_mlp_h64(mode, a, grid, s);
        case 128: return launch_mlp_h128(mode, a, grid, s);
        case 256: return launch_mlp_h256(mode, a, grid, s);
    }
    return cudaErrorInvalidValue;
}
int occupancy_any(int H, int mode, int YR) {
    switch (H) {
        case 32: return occupancy_mlp_h32(mode, YR);
        case 64: return occupancy_mlp_h64(mode, YR);
        case 128: return occupancy_mlp_h128(mode, YR);
        case 256: return occupancy_mlp_h256(mode, YR);
    }
    return 0;
}

template <typename T>
int dalloc(mjb_engine* e, T** p, size_t n) {
    CK(e, cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(n, 1) * sizeof(T)));
    CK(e, cudaMemsetAsync(*p, 0, std::max<size_t>(n, 1) * sizeof(T), e->stream));
    return 0;
}

bool is_host_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged;
}
// user pointer -> engine buffer ("host-or-device" arguments of the C ABI); host sources are counted as H2D traffic
int copy_in(mjb_engine* e, void* dst, const void* src, size_t bytes) {
    if (is_host_ptr(src)) e->h2d_bytes += (long long)bytes;
    CK(e, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, e->stream));
    return 0;
}

int allreduce(mjb_engine* e, void* buf, size_t count, ncclDataType_t dt, ncclRedOp_t op = ncclSum) {
    if (!e->comm) return 0;
    NK(e, g_nccl.AllReduce(buf, buf, count, dt, op, e->comm, e->stream));
    return 0;
}

int set_params(mjb_engine* e, ParamSet& ps, const float* theta_src) {
    if (theta_src && copy_in(e, ps.theta, theta_src, sizeof(float) * e->d)) return -1;
    launch_clamp_tail(ps.theta, e->d, e->A, e->cfg.min_log_std, e->stream);
    if (e->linear) launch_prep_linear(ps.theta, e->LL, ps.prep, e->stream);
    else launch_prep_mlp(ps.theta, e->PL, ps.prep, e->stream);
    e->launches += 2;
    if (e->tc_ok && !e->linear && &ps == &e->pnew) { launch_tc_prep(ps.theta, e->PL, nullptr, e->tc_prep_new, e->stream); e->launches += 1; }
    CK(e, cudaGetLastError());
    return 0;
}

int ensure_idx(mjb_engine* e, long long n) {
    if (n <= e->idx_cap) return 0;
    if (e->idx_dev) cudaFree(e->idx_dev);
    e->idx_cap = n;
    CK(e, cudaMalloc(&e->idx_dev, sizeof(int) * n));
    return 0;
}

// Launch one policy tile kernel over rows [0, n).
int run_policy(mjb_engine* e, int mode, const ParamSet& ps, const float* tangent_prep, long long n,
               const int* idx, const float* weight, int old_flags) {
    const bool bwd = (mode == MODE_VPG || mode == MODE_FVP);
    if (e->occ[mode] == 0) {
        e->occ[mode] = e->linear ? 2 : occupancy_any(e->H, mode, e->PL.YR);
        if (e->occ[mode] <= 0) FAIL(e, "kernel does not fit on this device (occupancy 0)");
    }
    const int MT = e->linear ? 128 : mlp_tile_rows_for(e->H);
    const long long tiles = (n + MT - 1) / MT;
    // while the fit is running on its own stream it owns vf_sms SMs: size the persistent grid for the rest
    const int sms = e->num_sms - (e->fit_in_flight ? e->vf_sms : 0);
    int grid = (int)std::max<long long>(1, std::min<long long>(tiles, (long long)e->occ[mode] * sms));
    grid = std::min(grid, e->max_grid);
    if (bwd) CK(e, cudaMemsetAsync(e->gpartial, 0, sizeof(float) * (size_t)grid * e->gstride, e->stream));
    cudaError_t ce;
    if (e->linear) {
        LinArgs a;
        a.L = e->LL; a.P = ps.prep; a.T = tangent_prep;
        a.in_shift = ps.in_shift; a.in_scale = ps.in_scale; a.out_shift = ps.out_shift; a.out_scale = ps.out_scale;
        a.obs = e->obs; a.act = e->act; a.idx = idx; a.n = n; a.weight = weight;
        a.ll_old = e->ll_old; a.mu_old = e->mu_old; a.old_log_std = e->pold.prep + e->LL.oLS; a.old_flags = old_flags;
        a.eval_partial = e->eval_partial; a.gpartial = e->gpartial; a.gstride = e->gstride;
        ce = launch_linear(mode, a, grid, e->stream);
    } else {
        MlpArgs a;
        memset(&a, 0, sizeof(a));
        a.L = e->PL; a.P = ps.prep; a.T = tangent_prep;
        a.in_shift = ps.in_shift; a.in_scale = ps.in_scale; a.out_shift = ps.out_shift; a.out_scale = ps.out_scale;
        a.obs = e->obs; a.obs_dim = e->cfg.obs_dim; a.act = e->act; a.idx = idx; a.n = n; a.weight = weight;
        a.ll_old = e->ll_old; a.mu_old = e->mu_old; a.old_log_std = e->pold.prep + e->PL.oLS; a.old_flags = old_flags;
        a.eval_partial = e->eval_partial; a.gpartial = e->gpartial; a.gstride = e->gstride;
        ce = launch_mlp_any(e->H, mode, a, grid, e->stream);
    }
    if (ce != cudaSuccess) FAIL(e, std::string("policy kernel launch: ") + cudaGetErrorString(ce));
    e->launches += 1;
    return grid;
}

// Make ll_old / mu_old valid for `rows` rows (forward with the OLD parameters and transforms).
int ensure_old_cache(mjb_engine* e, long long rows) {
    if (e->old_cache_valid && e->cache_rows >= rows) return 0;
    int g = run_policy(e, MODE_EVAL, e->pold, nullptr, rows, nullptr, nullptr, OLD_WRITE);
    if (g < 0) return -1;
    e->old_cache_valid = true;
    e->cache_rows = rows;
    return 0;
}

// Tail of every Fisher-vector product: sum of the per-CTA partials (+ the data-free log_std block), summed over the ranks.
// With peer memory set up (mjb_p2p_import) this is ONE kernel -- partial reduction, NVLink scatter, flag exchange, rank-
// ordered sum (p2p.cu); otherwise the reduction kernel followed by ncclAllReduce.
int fvp_reduce(mjb_engine* e, int grid, bool subsample, const float* v, float* out, const float* vscale) {
    const double* scale = e->dsc + (subsample ? DS_SCALE_SUB : DS_SCALE);
    if (e->comm && e->p2p_on) {
        P2PReduceArgs a;
        a.partial = e->gpartial; a.grid = grid; a.stride = e->gstride; a.d = e->d;
        a.scale_dev = scale; a.theta = e->pnew.theta; a.v = v; a.tLS = e->tLS; a.fvp_ls_block = 1; a.vscale = vscale;
        a.out = out; a.peers = e->p2p_peer_dev; a.world = e->cfg.world_size; a.rank = e->cfg.rank;
        a.cta_seq = e->p2p_seq; a.slot_words = e->p2p_slot;
        if (launch_reduce_allreduce_p2p(a, e->stream) != cudaSuccess) FAIL(e, "p2p reduce launch failed");
        e->launches += 1;
        e->p2p_calls += 1;
        return 0;
    }
    launch_reduce_partials(e->gpartial, grid, e->gstride, e->d, scale, out, e->pnew.theta, v, e->tLS, 1, vscale, e->stream);
    e->launches += 1;
    CK(e, cudaGetLastError());
    return allreduce(e, out, e->d, ncclFloat);
}

// F v (undamped, all-reduced) into out.  v, out: device pointers of d floats.
// have_vscale: e->tc_vscale already holds the power-of-two scale of v (written by cg_init / cg_update).
// ev0/ev1: events recorded around the tile kernel (the FVP ring slot, or a graph's own pair while capturing).
int fvp_device(mjb_engine* e, const float* v, const int* idx, long long n_idx, float* out, bool have_vscale = false,
               cudaEvent_t ev0 = nullptr, cudaEvent_t ev1 = nullptr) {
    const long long n = idx ? n_idx : e->n_roll;
    // events handed in belong to a graph being captured: they become EXTERNAL event-record nodes, which is what makes
    // cudaEventElapsedTime on them legal after a replay
    const unsigned evflag = ev0 ? cudaEventRecordExternal : cudaEventRecordDefault;
    if (!ev0) {
        const int slot = (int)(e->fvp_count % mjb_engine::kFvpRing);
        ev0 = e->fvp_ev[slot][0]; ev1 = e->fvp_ev[slot][1];
        e->fvp_count += 1;
    }
    if (e->tc_ok && e->tc_on) {
        // tensor-core path: scale v to O(1) (exact power of two), split to fp16 hi/lo, tcgen05 tile kernel
        if (!have_vscale) { launch_tc_vscale(v, e->d, e->tc_vscale, e->stream); e->launches += 1; }
        if (e->linear) launch_lin_tc_prep(v, e->cfg.obs_dim, e->A, idx != nullptr, e->tc_vscale, e->tc_prep_tan, e->stream);
        else launch_tc_prep(v, e->PL, e->tc_vscale, e->tc_prep_tan, e->stream);
        const int sms = e->num_sms - (e->fit_in_flight ? e->vf_sms : 0);
        const int tile_rows = e->linear ? 64 : 128;
        const long long tiles = (n + tile_rows - 1) / tile_rows;
        const int grid = (int)std::max<long long>(1, std::min<long long>(tiles, sms));
        CK(e, cudaEventRecordWithFlags(ev0, e->stream, evflag));   // (the kernels zero their own gradient partials)
        cudaError_t ce = e->linear
            ? launch_linear_tc(e->tc_prep_tan, e->pnew.theta, e->pnew.in_shift, e->pnew.in_scale, e->pnew.out_scale,
                               e->pnew.in_ident, e->obs, e->cfg.obs_dim, e->A, idx, n, e->gpartial, e->gstride, e->LL.tW, e->LL.tb, e->LL.tLS, grid, e->stream)
            : launch_fvp_tc(e->PL, e->tc_prep_new, e->tc_prep_tan, e->pnew.in_shift, e->pnew.in_scale,
                            e->pnew.out_scale, e->obs, idx, n, e->gpartial, e->gstride, grid, e->stream);
        if (ce != cudaSuccess) FAIL(e, std::string("fvp_tc launch: ") + cudaGetErrorString(ce));
        CK(e, cudaEventRecordWithFlags(ev1, e->stream, evflag));
        e->launches += 2;
        return fvp_reduce(e, grid, idx != nullptr, v, out, e->tc_vscale);
    }
    if (e->linear) launch_prep_linear(v, e->LL, e->prep_tan, e->stream);
    else launch_prep_mlp(v, e->PL, e->prep_tan, e->stream);
    e->launches += 1;
    // the memset of the gradient partials belongs to the FVP; the event pair brackets memset + tile kernel
    CK(e, cudaEventRecordWithFlags(ev0, e->stream, evflag));
    int grid = run_policy(e, MODE_FVP, e->pnew, e->prep_tan, n, idx, nullptr, 0);
    if (grid < 0) return -1;
    CK(e, cudaEventRecordWithFlags(ev1, e->stream, evflag));
    return fvp_reduce(e, grid, idx != nullptr, v, out, nullptr);
}

int set_subsample_scale(mjb_engine* e, long long n_idx_local) {
    e->h_dsc[DS_CNT] = (double)n_idx_local;
    CK(e, cudaMemcpyAsync(e->dsc + DS_CNT, e->h_dsc + DS_CNT, sizeof(double), cudaMemcpyHostToDevice, e->stream));
    if (allreduce(e, e->dsc + DS_CNT, 1, ncclDouble)) return -1;
    CK(e, cudaMemcpyAsync(e->h_dsc + DS_CNT, e->dsc + DS_CNT, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    e->h_dsc[DS_SCALE_SUB] = 1.0 / e->h_dsc[DS_CNT];
    e->h_dsc[DS_SCALE_SUB + 1] = 1.0 / (double)e->cfg.world_size;
    CK(e, cudaMemcpyAsync(e->dsc + DS_SCALE_SUB, e->h_dsc + DS_SCALE_SUB, 2 * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    return 0;
}

int eval_device(mjb_engine* e, double out[2]) {
    if (!e->have_white) FAIL(e, "mjb_policy_eval: call mjb_process_paths first");
    if (ensure_old_cache(e, e->n_roll)) return -1;
    int grid = run_policy(e, MODE_EVAL, e->pnew, nullptr, e->n_roll, nullptr, e->adv_white, OLD_READ);
    if (grid < 0) return -1;
    launch_reduce_eval(e->eval_partial, grid, e->dsc + DS_EVAL, e->stream);
    e->launches += 1;
    if (allreduce(e, e->dsc + DS_EVAL, 2, ncclDouble)) return -1;
    CK(e, cudaMemcpyAsync(e->h_dsc + DS_EVAL, e->dsc + DS_EVAL, 2 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    // torch.mean in fp32: round the mean to fp32 like the reference's scalar
    out[0] = (double)(float)(e->h_dsc[DS_EVAL] / (double)e->n_glob_roll);
    out[1] = (double)(float)(e->h_dsc[DS_EVAL + 1] / (double)e->n_glob_roll);
    return 0;
}

// VPG into e->g (all-reduced).  Returns surr_before through *surr when non-null.
int vpg_device(mjb_engine* e, int include_demo, double demo_lam, double* surr) {
    if (!e->have_white) FAIL(e, "mjb_policy_vpg: call mjb_process_paths first");
    long long n = e->n_roll;
    const float* w = e->adv_white;
    if (include_demo && e->n_demo > 0) {
        launch_dapg_weights(e->adv, e->n_roll, e->n_demo, e->dsc + DS_STATS, demo_lam, e->weights, e->stream);
        e->launches += 1;
        n = e->n_roll + e->n_demo;
        w = e->weights;
    }
    int flags;
    if (e->old_equals_new) {
        flags = OLD_WRITE;                 // LR == 1 exactly; cache mu/LL of the old policy on the way
    } else {
        if (ensure_old_cache(e, n)) return -1;
        flags = OLD_READ;
    }
    int grid = run_policy(e, MODE_VPG, e->pnew, nullptr, n, nullptr, w, flags);
    if (grid < 0) return -1;
    if (flags == OLD_WRITE) { e->old_cache_valid = true; e->cache_rows = n; }
    launch_reduce_partials(e->gpartial, grid, e->gstride, e->d, e->dsc + DS_SCALE, e->g, nullptr, nullptr, e->tLS, 0, nullptr, e->stream);
    e->launches += 1;
    if (allreduce(e, e->g, e->d, ncclFloat)) return -1;
    if (surr) {
        if (n == e->n_roll) {
            launch_reduce_eval(e->eval_partial, grid, e->dsc + DS_EVAL, e->stream);
            e->launches += 1;
            if (allreduce(e, e->dsc + DS_EVAL, 2, ncclDouble)) return -1;
            CK(e, cudaMemcpyAsync(e->h_dsc + DS_EVAL, e->dsc + DS_EVAL, 2 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            CK(e, cudaStreamSynchronize(e->stream));
            *surr = (double)(float)(e->h_dsc[DS_EVAL] / (double)e->n_glob_roll);
        } else {
            double o[2];
            if (eval_device(e, o)) return -1;
            *surr = o[0];
        }
    }
    CK(e, cudaGetLastError());
    return 0;
}

// The launches of one cg_solve (utils/cg_solve.py:3-22): init, then per iteration {tangent prep, FVP tile kernel,
// partial reduce, all-reduce, fused update (which also emits the next tangent's scale)}.
int cg_body(mjb_engine* e, const float* b, int iters, float damping, float tol, const int* idx_dev, long long n_idx,
            const std::vector<cudaEvent_t>* evs, const std::vector<long long>* len_each = nullptr) {
    const bool tc = e->tc_ok && e->tc_on;
    launch_cg_init(b, e->x, e->r, e->p, e->d, e->dsc + DS_CG, tc ? e->tc_vscale : nullptr, e->stream);
    e->launches += 1;
    for (int i = 0; i < iters; ++i) {
        const int* idx = idx_dev ? idx_dev + (size_t)i * n_idx : nullptr;
        const long long n_i = (idx && len_each) ? (*len_each)[i] : n_idx;      // rows of iteration i ([i][0 .. n_i) of the index block)
        if (fvp_device(e, e->p, idx, n_i, e->Fp, tc, evs ? (*evs)[2 * i] : nullptr, evs ? (*evs)[2 * i + 1] : nullptr)) return -1;
        launch_cg_update(e->Fp, damping, tol, e->x, e->r, e->p, e->d, e->dsc + DS_CG, tc ? e->tc_vscale : nullptr, e->stream);
        e->launches += 1;
    }
    CK(e, cudaGetLastError());
    return 0;
}

// cg_solve as ONE graph launch: the loop is launch-bound (d <= 83 k floats per vector op, ~50 nodes), so it is captured
// once per distinct shape and replayed; anything that prevents the capture falls back to plain stream launches.
int cg_device(mjb_engine* e, const float* b, int iters, float damping, float tol, const int* idx_dev, long long n_idx) {
    e->last_cg_graph = nullptr;
    if (idx_dev && !e->hvp_len.empty()) {                     // ragged per-iteration subsamples: plain stream launches
        std::vector<long long> len = std::move(e->hvp_len);
        e->hvp_len.clear();
        if ((int)len.size() != iters) FAIL(e, "mjb_policy_set_hvp_lengths: one length per CG iteration expected");
        for (long long l : len) if (l < 0 || l > n_idx) FAIL(e, "mjb_policy_set_hvp_lengths: length exceeds the index block stride");
        return cg_body(e, b, iters, damping, tol, idx_dev, n_idx, nullptr, &len);
    }
    e->hvp_len.clear();
    if (!e->graphs_on || iters < 1) return cg_body(e, b, iters, damping, tol, idx_dev, n_idx, nullptr);
    const long long n = idx_dev ? n_idx : e->n_roll;
    const int sms = e->num_sms - (e->fit_in_flight ? e->vf_sms : 0);
    const bool tc = e->tc_ok && e->tc_on;
    mjb_engine::CgGraph* hit = nullptr;
    for (auto& gph : e->cg_graphs)
        if (gph.n == n && gph.idx == idx_dev && gph.n_idx == n_idx && gph.iters == iters && gph.damping == damping &&
            gph.tol == tol && gph.sms == sms && gph.tc == tc && gph.p2p == e->p2p_on) { hit = &gph; break; }
    if (!hit) {
        if (e->cg_graphs.size() >= 8) {                       // shapes keep changing: drop the oldest
            auto& old = e->cg_graphs.front();
            if (old.exec) cudaGraphExecDestroy(old.exec);
            for (auto& ev : old.ev) if (ev) cudaEventDestroy(ev);
            e->cg_graphs.erase(e->cg_graphs.begin());
        }
        mjb_engine::CgGraph gph;
        gph.n = n; gph.idx = idx_dev; gph.n_idx = n_idx; gph.iters = iters; gph.damping = damping; gph.tol = tol;
        gph.sms = sms; gph.tc = tc; gph.p2p = e->p2p_on;
        gph.ev.assign((size_t)2 * iters, nullptr);
        for (auto& ev : gph.ev) CK(e, cudaEventCreate(&ev));
        // occupancy queries / attribute setters of the kernels must not run for the first time inside a capture
        if (!tc && e->occ[MODE_FVP] == 0) {
            e->occ[MODE_FVP] = e->linear ? 2 : occupancy_any(e->H, MODE_FVP, e->PL.YR);
            if (e->occ[MODE_FVP] <= 0) FAIL(e, "kernel does not fit on this device (occupancy 0)");
        }
        const long long launches0 = e->launches;
        cudaGraph_t graph = nullptr;
        bool ok = cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
        if (ok) {
            const int rc = cg_body(e, b, iters, damping, tol, idx_dev, n_idx, &gph.ev);
            const cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
            ok = rc == 0 && ce == cudaSuccess && graph != nullptr;
        }
        if (ok) ok = cudaGraphInstantiate(&gph.exec, graph, 0) == cudaSuccess;
        if (graph) cudaGraphDestroy(graph);
        e->launches = launches0;                              // capturing launched nothing
        if (!ok) {
            cudaGetLastError();
            for (auto& ev : gph.ev) if (ev) cudaEventDestroy(ev);
            e->graphs_on = false;                             // e.g. a collective that cannot be captured: stay eager
            return cg_body(e, b, iters, damping, tol, idx_dev, n_idx, nullptr);
        }
        e->cg_graphs.push_back(std::move(gph));
        hit = &e->cg_graphs.back();
    }
    CK(e, cudaGraphLaunch(hit->exec, e->stream));
    const bool tcp = tc;
    e->launches += 1 + (long long)iters * (tcp ? 4 : 5);      // kernels inside the graph (memset nodes not counted)
    e->last_cg_graph = hit;
    return 0;
}

int upload_idx(mjb_engine* e, const int32_t* idx, long long total) {
    if (ensure_idx(e, total)) return -1;
    return copy_in(e, e->idx_dev, idx, sizeof(int) * total);
}

}  // namespace

// =====================================================================================================
extern "C" {

int mjb_version(void) { return MJB_VERSION; }

const char* mjb_last_error(const mjb_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

void mjb_destroy(mjb_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    if (e->stream_vf) cudaStreamSynchronize(e->stream_vf);
    if (e->stream) cudaStreamSynchronize(e->stream);
    // captured CG graphs hold references on the communicator (NCCL keeps a comm with live graph-captured work alive and
    // ncclCommDestroy waits for them): the graphs go first
    for (auto& gph : e->cg_graphs) {
        if (gph.exec) cudaGraphExecDestroy(gph.exec);
        for (auto& ev : gph.ev) if (ev) cudaEventDestroy(ev);
    }
    e->cg_graphs.clear();
    cudaDeviceSynchronize();
    if (e->comm) g_nccl.CommDestroy(e->comm);
    for (int p = 0; p < (int)e->p2p_peer.size(); ++p)
        if (p != e->cfg.rank && e->p2p_peer[p]) cudaIpcCloseMemHandle(e->p2p_peer[p]);
    for (void* b : {(void*)e->ridge_ab, (void*)e->ridge_partial, (void*)e->ridge_G, (void*)e->ridge_coeff, (void*)e->ridge_err, (void*)e->ridge_T})
        if (b) cudaFree(b);
    if (e->p2p_buf) cudaFree(e->p2p_buf);
    if (e->p2p_peer_dev) cudaFree(e->p2p_peer_dev);
    if (e->p2p_seq) cudaFree(e->p2p_seq);
    void* bufs[] = {e->pnew.theta, e->pnew.prep, e->pnew.in_shift, e->pnew.in_scale, e->pnew.out_shift, e->pnew.out_scale,
                    e->pold.theta, e->pold.prep, e->pold.in_shift, e->pold.in_scale, e->pold.out_shift, e->pold.out_scale,
                    e->prep_tan, e->tc_prep_new, e->tc_prep_tan, e->tc_vscale, e->obs, e->act, e->rew, e->path_off, e->term, e->tstep, e->ret, e->adv, e->base,
                    e->adv_white, e->weights, e->path_ret, e->ll_old, e->mu_old, e->gpartial, e->eval_partial,
                    e->mom_scratch, e->dsc, e->g, e->x, e->r, e->p, e->Fp, e->tmpv, e->idx_dev, e->stage64, e->vf_w,
                    e->vf_m, e->vf_v, e->vf_wT, e->vf_prep, e->vf_feat, e->vf_ret32, e->vf_consts, e->vf_ks, e->perm_dev, e->fit_obs, e->fit_tstep, e->fit_ret,
                    e->sgd_m, e->sgd_v, e->sgd_wT, e->sgd_idx, e->sgd_out};
    for (void* b : bufs) if (b) cudaFree(b);
    if (e->pinned) cudaFreeHost(e->pinned);
    if (e->h_dsc) cudaFreeHost(e->h_dsc);
    for (auto& ev : e->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : e->user_ev) if (ev) cudaEventDestroy(ev);
    for (auto& pr : e->fvp_ev) for (auto& ev : pr) if (ev) cudaEventDestroy(ev);
    for (auto& ev : e->fit_ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : e->sgd_ev) if (ev) cudaEventDestroy(ev);
    if (e->stream_vf) { cudaStreamSynchronize(e->stream_vf); cudaStreamDestroy(e->stream_vf); }
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

int mjb_create(const mjb_config* cfg, mjb_engine** out) {
    if (!cfg || !out) { g_create_error = "null argument"; return -1; }
    *out = nullptr;
    mjb_engine* e = new mjb_engine();
    e->cfg = *cfg;
    for (auto& ev : e->ev) ev = nullptr;
    for (auto& ev : e->user_ev) ev = nullptr;
    for (auto& pr : e->fvp_ev) for (auto& ev : pr) ev = nullptr;
    auto fail = [&](const std::string& m) { g_create_error = m.empty() ? e->err : m; mjb_destroy(e); return -1; };
    if (cfg->obs_dim < 1 || cfg->act_dim < 1 || cfg->act_dim > 32) return fail("act_dim must be in [1,32], obs_dim >= 1");
    if (cfg->n_hidden != 0 && cfg->n_hidden != 2) return fail("only 0 (linear) or 2 hidden layers are supported");
    if (cfg->max_samples < 1 || cfg->max_paths < 1) return fail("max_samples/max_paths must be positive");
    if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size) return fail("bad world_size/rank");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return fail("no CUDA device (this engine has no CPU fallback)");
    if (cfg->device < 0 || cfg->device >= ndev) return fail("bad device ordinal");
    if (cudaSetDevice(cfg->device) != cudaSuccess) return fail("cudaSetDevice failed");
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, cfg->device);
    if (prop.major < 10) return fail("mjrl_b200 kernels are built for sm_100a (Blackwell) only");
    e->num_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) return fail("stream create failed");
    if (cudaStreamCreateWithFlags(&e->stream_vf, cudaStreamNonBlocking) != cudaSuccess) return fail("stream create failed");
    for (auto& ev : e->ev) if (cudaEventCreate(&ev) != cudaSuccess) return fail("event create failed");
    for (auto& ev : e->user_ev) if (cudaEventCreate(&ev) != cudaSuccess) return fail("event create failed");
    for (auto& pr : e->fvp_ev) for (auto& ev : pr) if (cudaEventCreate(&ev) != cudaSuccess) return fail("event create failed");
    for (auto& ev : e->fit_ev) if (cudaEventCreate(&ev) != cudaSuccess) return fail("event create failed");
    for (auto& ev : e->sgd_ev) if (cudaEventCreate(&ev) != cudaSuccess) return fail("event create failed");

    e->linear = cfg->n_hidden == 0;
    e->A = cfg->act_dim;
    if (e->linear) {
        e->LL = make_lin_layout(cfg->obs_dim, cfg->act_dim);
        e->d = e->LL.d; e->prep_total = e->LL.total; e->tLS = e->LL.tLS;
    } else {
        if (cfg->hidden[0] < 1 || cfg->hidden[1] < 1 || cfg->hidden[0] > 256 || cfg->hidden[1] > 256)
            return fail("hidden sizes must be in [1,256]");
        e->H = pad_hidden(std::max(cfg->hidden[0], cfg->hidden[1]));
        e->PL = make_prep_layout(e->H, cfg->obs_dim, cfg->act_dim, cfg->hidden[0], cfg->hidden[1], true);
        e->d = e->PL.d; e->prep_total = e->PL.total; e->tLS = e->PL.tLS;
    }
    const int vh0 = cfg->vf_hidden[0] > 0 ? cfg->vf_hidden[0] : 128, vh1 = cfg->vf_hidden[1] > 0 ? cfg->vf_hidden[1] : 128;
    if (vh0 > 256 || vh1 > 256 || vh0 % 4 || vh1 % 4) return fail("vf hidden sizes must be multiples of 4, <= 256");
    e->cfg.vf_hidden[0] = vh0; e->cfg.vf_hidden[1] = vh1;
    e->vfH = pad_hidden(std::max(vh0, vh1));
    e->VPL = make_prep_layout(e->vfH, cfg->obs_dim + 4, 1, vh0, vh1, false);
    e->vf_d = e->VPL.d;

    e->cap = cfg->max_samples;
    const size_t N = (size_t)e->cap, O = cfg->obs_dim, A = cfg->act_dim;
#define ALLOC(ptr, n) if (dalloc(e, &(ptr), (n))) return fail("")
    for (ParamSet* ps : {&e->pnew, &e->pold}) {
        ALLOC(ps->theta, e->d); ALLOC(ps->prep, e->prep_total);
        ALLOC(ps->in_shift, O); ALLOC(ps->in_scale, O); ALLOC(ps->out_shift, A); ALLOC(ps->out_scale, A);
        std::vector<float> ones(std::max(O, A), 1.0f);
        cudaMemcpyAsync(ps->in_scale, ones.data(), O * sizeof(float), cudaMemcpyHostToDevice, e->stream);
        cudaMemcpyAsync(ps->out_scale, ones.data(), A * sizeof(float), cudaMemcpyHostToDevice, e->stream);
        cudaStreamSynchronize(e->stream);
    }
    ALLOC(e->prep_tan, e->prep_total);
    e->tc_ok = e->linear ? lin_tc_supported(cfg->obs_dim, cfg->act_dim) : fvp_tc_supported(e->PL);
    if (const char* env = getenv("MJRL_B200_TC")) e->tc_on = atoi(env) != 0;
    if (const char* env = getenv("MJRL_B200_GRAPH")) e->graphs_on = atoi(env) != 0;
    if (e->tc_ok) {
        const size_t pb = e->linear ? lin_tc_prep_bytes() : fvp_tc_prep_bytes();
        ALLOC(e->tc_prep_new, pb); ALLOC(e->tc_prep_tan, pb); ALLOC(e->tc_vscale, 2);
    }
    ALLOC(e->obs, N * O); ALLOC(e->act, N * A); ALLOC(e->rew, N);
    ALLOC(e->path_off, (size_t)cfg->max_paths + 2); ALLOC(e->term, (size_t)cfg->max_paths + 1); ALLOC(e->tstep, N);
    ALLOC(e->ret, N); ALLOC(e->adv, N); ALLOC(e->base, N); ALLOC(e->adv_white, N); ALLOC(e->weights, N);
    ALLOC(e->path_ret, (size_t)cfg->max_paths + 1);
    ALLOC(e->ll_old, N); ALLOC(e->mu_old, N * A);
    e->max_grid = 2 * e->num_sms;
    e->gstride = round_up(e->d, 32);
    ALLOC(e->gpartial, (size_t)e->max_grid * e->gstride);
    ALLOC(e->eval_partial, (size_t)2 * e->max_grid);
    ALLOC(e->mom_scratch, 2 * 512);
    ALLOC(e->dsc, DS_TOTAL);
    if (cudaMallocHost(reinterpret_cast<void**>(&e->h_dsc), DS_TOTAL * sizeof(double)) != cudaSuccess) return fail("pinned alloc failed");
    memset(e->h_dsc, 0, DS_TOTAL * sizeof(double));
    ALLOC(e->g, e->d); ALLOC(e->x, e->d); ALLOC(e->r, e->d); ALLOC(e->p, e->d); ALLOC(e->Fp, e->d); ALLOC(e->tmpv, e->d);
    e->stage64_elems = N * std::max(O, A);
    ALLOC(e->stage64, e->stage64_elems);
    ALLOC(e->vf_w, e->vf_d); ALLOC(e->vf_m, e->vf_d); ALLOC(e->vf_v, e->vf_d);
    ALLOC(e->vf_wT, (size_t)(O + 4) * vh0 + (size_t)vh0 * vh1);
    ALLOC(e->vf_prep, e->VPL.total);
    ALLOC(e->sgd_m, e->d); ALLOC(e->sgd_v, e->d);
    if (!e->linear) ALLOC(e->sgd_wT, policy_sgd_scratch_floats(cfg->obs_dim, cfg->hidden[0], cfg->hidden[1], cfg->act_dim));
#undef ALLOC
    e->pinned_bytes = std::min<size_t>(N * std::max(O, A) * sizeof(double), (size_t)64 << 20);
    e->pinned_bytes = std::max<size_t>(e->pinned_bytes, (size_t)1 << 20);
    if (cudaMallocHost(&e->pinned, 2 * e->pinned_bytes) != cudaSuccess) return fail("pinned staging alloc failed");
    e->h_dsc[DS_SCALE + 1] = 1.0 / (double)cfg->world_size;
    if (cudaStreamSynchronize(e->stream) != cudaSuccess) return fail("init sync failed");
    *out = e;
    return 0;
}

int mjb_synchronize(mjb_engine* e) {
    CK(e, cudaStreamSynchronize(e->stream));
    if (e->fit_in_flight) CK(e, cudaStreamSynchronize(e->stream_vf));
    return 0;
}

int mjb_comm_unique_id(void* id128) {
    std::string err;
    if (!g_nccl.load(err)) { g_create_error = err; return -1; }
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return -1; }
    memcpy(id128, &id, sizeof(id));
    return 0;
}

int mjb_comm_init(mjb_engine* e, const void* id128) {
    if (e->cfg.world_size == 1) return 0;
    if (!g_nccl.load(e->err)) return -1;
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    CK(e, cudaSetDevice(e->cfg.device));
    NK(e, g_nccl.CommInitRank(&e->comm, e->cfg.world_size, id, e->cfg.rank));
    return 0;
}

// ---- all-reduce over NVLink peer memory: every rank exports its exchange buffer as a CUDA IPC handle, the host side
// all-gathers the 64-byte handles (torch.distributed) and every rank imports all of them.
int mjb_p2p_export(mjb_engine* e, void* handle64) {
    if (e->cfg.world_size == 1) FAIL(e, "mjb_p2p_export: single-rank engine");
    CK(e, cudaSetDevice(e->cfg.device));
    if (!e->p2p_buf) {
        const int ctas = (e->d + 127) / 128;
        e->p2p_slot = ((long long)e->d + 31) / 32 * 32;
        e->p2p_bytes = (size_t)2 * e->cfg.world_size * e->p2p_slot * sizeof(unsigned long long);
        CK(e, cudaMalloc(&e->p2p_buf, e->p2p_bytes));
        CK(e, cudaMemset(e->p2p_buf, 0, e->p2p_bytes));       // call numbers start at 1: a zeroed word is "not yet"
        CK(e, cudaMalloc(&e->p2p_seq, sizeof(int) * ctas));
        CK(e, cudaMemset(e->p2p_seq, 0, sizeof(int) * ctas));
        CK(e, cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t h;
    CK(e, cudaIpcGetMemHandle(&h, e->p2p_buf));
    static_assert(sizeof(h) == 64, "CUDA IPC handles are 64 bytes");
    memcpy(handle64, &h, 64);
    return 0;
}

int mjb_p2p_import(mjb_engine* e, const void* handles /* world x 64 bytes, rank order */) {
    if (!e->p2p_buf) FAIL(e, "mjb_p2p_import: call mjb_p2p_export first");
    CK(e, cudaSetDevice(e->cfg.device));
    const int W = e->cfg.world_size;
    e->p2p_peer.assign(W, nullptr);
    for (int p = 0; p < W; ++p) {
        if (p == e->cfg.rank) { e->p2p_peer[p] = e->p2p_buf; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const unsigned char*>(handles) + 64 * p, 64);
        const cudaError_t ce = cudaIpcOpenMemHandle(&e->p2p_peer[p], h, cudaIpcMemLazyEnablePeerAccess);
        if (ce != cudaSuccess) {
            e->p2p_peer[p] = nullptr;
            cudaGetLastError();
            FAIL(e, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(p) + "): " + cudaGetErrorString(ce));
        }
    }
    if (!e->p2p_peer_dev) CK(e, cudaMalloc(&e->p2p_peer_dev, sizeof(void*) * W));
    CK(e, cudaMemcpy(e->p2p_peer_dev, e->p2p_peer.data(), sizeof(void*) * W, cudaMemcpyHostToDevice));
    e->p2p_ready = true;
    return 0;
}

// on = 1 only takes effect after a successful import ON EVERY RANK (the caller agrees on that: a rank on NCCL and a rank
// on peer memory would wait for each other forever).  Returns the resulting state.
int mjb_p2p_enable(mjb_engine* e, int on) {
    e->p2p_on = on != 0 && e->p2p_ready && e->comm != nullptr;
    return e->p2p_on ? 1 : 0;
}

long long mjb_p2p_calls(mjb_engine* e) { return e->p2p_calls; }

// ------------------------------------------------------------------------ ridge baselines (Linear / Quadratic)
// Feature columns in the reference's order (linear_baseline.py:19-36, quadratic_baseline.py:20-43):
//   kind 0: [o (n) | 1 | al al^2 al^3 al^4]                      K = n + 5
//   kind 1: [o (n) | o_i o_j, i <= j (n (n + 1) / 2) | 1 | al al^2 al^3 al^4]
static int ridge_feature_count(int kind, int n) { return kind == 0 ? n + 5 : n + n * (n + 1) / 2 + 5; }
static int ridge_setup(mjb_engine* e, int kind) {
    const int n = e->cfg.obs_dim;
    if (kind != 0 && kind != 1) FAIL(e, "ridge baseline kind must be 0 (linear) or 1 (quadratic)");
    const int K = ridge_feature_count(kind, n);
    if (K + 1 > 4096) FAIL(e, "ridge baseline: more than 4095 features (quadratic features of a wide observation)");
    if (e->ridge_ab_kind == kind) return K;
    std::vector<short2> ab;
    const short ONE = (short)n, RET = (short)(n + 5);
    for (int c = 0; c < n; ++c) ab.push_back(make_short2((short)c, ONE));
    if (kind == 1)
        for (int i = 0; i < n; ++i)
            for (int j = i; j < n; ++j) ab.push_back(make_short2((short)i, (short)j));
    ab.push_back(make_short2(ONE, ONE));
    for (int k = 1; k <= 4; ++k) ab.push_back(make_short2((short)(n + k), ONE));
    ab.push_back(make_short2(RET, ONE));                           // the augmented returns column (Gram launches only)
    if (e->ridge_ab) cudaFree(e->ridge_ab);
    CK(e, cudaMalloc(&e->ridge_ab, sizeof(short2) * ab.size()));
    CK(e, cudaMemcpy(e->ridge_ab, ab.data(), sizeof(short2) * ab.size(), cudaMemcpyHostToDevice));
    if (e->ridge_coeff) cudaFree(e->ridge_coeff);
    CK(e, cudaMalloc(&e->ridge_coeff, sizeof(double) * (K + 1)));
    if (!e->ridge_err) CK(e, cudaMalloc(&e->ridge_err, sizeof(double) * 2048));
    e->ridge_ab_kind = kind; e->ridge_K = K;
    return K;
}

// T = scaled observations | 1 | time powers | returns | 0 of the resident batch (ridge.cu); rebuilt per call: the batch or
// its returns may have changed, and the pass is one write of n x (obs_dim + 7) doubles.
static int ridge_scaled(mjb_engine* e, const RidgeArgs& a) {
    const size_t need = (size_t)a.n * a.tile_cols;
    if (need > e->ridge_T_cap) {
        if (e->ridge_T) cudaFree(e->ridge_T);
        e->ridge_T = nullptr; e->ridge_T_cap = 0;
        CK(e, cudaMalloc(&e->ridge_T, sizeof(double) * need));
        e->ridge_T_cap = need;
    }
    RidgeArgs b = a;
    b.ret = e->ret;                                                // the returns column is always filled
    if (launch_ridge_scale(b, e->ridge_T, e->stream) != cudaSuccess) FAIL(e, "ridge scale launch failed");
    return 0;
}

int mjb_ridge_features(const mjb_engine* e, int kind) { return ridge_feature_count(kind, e->cfg.obs_dim); }

// Gram matrix of [F | y] over the resident rollout batch (summed over the ranks): out = (K + 1) x (K + 1) doubles, row-major;
// F^T F = out[:K, :K], F^T y = out[:K, K], y^T y = out[K, K].  Needs the returns (mjb_compute_returns / mjb_batch_set_returns).
int mjb_ridge_gram(mjb_engine* e, int kind, double* out) {
    const int K = ridge_setup(e, kind);
    if (K < 0) return -1;
    if (e->n_roll <= 0) FAIL(e, "mjb_ridge_gram: no rollout batch resident");
    const int KA = K + 1;
    RidgeArgs a;
    a.obs = e->obs; a.tstep = e->tstep; a.ret = e->ret; a.n = e->n_roll; a.obs_dim = e->cfg.obs_dim;
    a.K = KA; a.ab = e->ridge_ab; a.tile_cols = e->cfg.obs_dim + 7;
    a.nb = ridge_blocks(KA);
    const int npairs = a.nb * (a.nb + 1) / 2;
    a.splits = (int)std::max<long long>(1, std::min<long long>({256LL, (2LL * e->num_sms + npairs - 1) / npairs, (e->n_roll + 255) / 256}));
    if (KA <= 32) a.splits = (int)std::max<long long>(1, std::min<long long>(4LL * e->num_sms, (e->n_roll + 255) / 256));   // CTAs of 8 warps
    const size_t need = KA <= 32 ? (size_t)a.splits * 8 * 1024 : (size_t)a.splits * npairs * 4096;
    if (need > e->ridge_partial_cap) {
        if (e->ridge_partial) cudaFree(e->ridge_partial);
        CK(e, cudaMalloc(&e->ridge_partial, sizeof(double) * need));
        e->ridge_partial_cap = need;
    }
    if ((size_t)KA * KA > e->ridge_G_cap) {
        if (e->ridge_G) cudaFree(e->ridge_G);
        CK(e, cudaMalloc(&e->ridge_G, sizeof(double) * (size_t)KA * KA));
        e->ridge_G_cap = (size_t)KA * KA;
    }
    a.partial = e->ridge_partial;
    if (ridge_scaled(e, a)) return -1;
    const cudaError_t ce = launch_ridge_gram(a, e->ridge_T, e->ridge_G, e->stream);
    if (ce != cudaSuccess) FAIL(e, std::string("ridge gram launch: ") + cudaGetErrorString(ce));
    e->launches += 3;
    if (allreduce(e, e->ridge_G, (size_t)KA * KA, ncclDouble)) return -1;
    CK(e, cudaMemcpyAsync(out, e->ridge_G, sizeof(double) * (size_t)KA * KA, cudaMemcpyDeviceToHost, e->stream));
    e->d2h_bytes += (long long)(sizeof(double) * (size_t)KA * KA);
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

// Predictions F c of every resident rollout sample into the baseline buffer (what mjb_compute_advantages reads and
// mjb_batch_get(MJB_F_BASELINE) returns).  coeffs: K host doubles.  sq_err (nullable): sum over ALL ranks of (y - F c)^2.
int mjb_ridge_predict(mjb_engine* e, int kind, const double* coeffs, double* sq_err) {
    const int K = ridge_setup(e, kind);
    if (K < 0) return -1;
    if (e->n_roll <= 0) FAIL(e, "mjb_ridge_predict: no rollout batch resident");
    if (copy_in(e, e->ridge_coeff, coeffs, sizeof(double) * K)) return -1;
    RidgeArgs a;
    a.obs = e->obs; a.tstep = e->tstep; a.ret = sq_err ? e->ret : nullptr; a.n = e->n_roll; a.obs_dim = e->cfg.obs_dim;
    a.K = K; a.ab = e->ridge_ab; a.tile_cols = e->cfg.obs_dim + 7; a.partial = nullptr; a.splits = 0; a.nb = 0;
    const int grid = (int)std::max<long long>(1, std::min<long long>(2048, std::min<long long>(8LL * e->num_sms, (e->n_roll + 7) / 8)));
    if (ridge_scaled(e, a)) return -1;
    const cudaError_t ce = launch_ridge_predict(a, e->ridge_T, e->ridge_coeff, K, e->base, sq_err ? e->ridge_err : nullptr, grid, e->stream);
    if (ce != cudaSuccess) FAIL(e, std::string("ridge predict launch: ") + cudaGetErrorString(ce));
    e->launches += 2;
    if (sq_err) {
        std::vector<double> h(grid);
        CK(e, cudaMemcpyAsync(h.data(), e->ridge_err, sizeof(double) * grid, cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        double s = 0.0;
        for (int i = 0; i < grid; ++i) s += h[i];                  // fixed order
        e->h_dsc[DS_VF] = s;
        CK(e, cudaMemcpyAsync(e->dsc + DS_VF, e->h_dsc + DS_VF, sizeof(double), cudaMemcpyHostToDevice, e->stream));
        if (allreduce(e, e->dsc + DS_VF, 1, ncclDouble)) return -1;
        CK(e, cudaMemcpyAsync(e->h_dsc + DS_VF, e->dsc + DS_VF, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        *sq_err = e->h_dsc[DS_VF];
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------- batch
int mjb_vf_fit_end(mjb_engine* e, double* err_after);
static int finish_upload(mjb_engine* e, int which, int n_paths, const int32_t* len, const uint8_t* terminated, long long n) {
    if (which == MJB_BATCH_ROLLOUT) {
        e->h_path_off.assign((size_t)n_paths + 1, 0);
        for (int i = 0; i < n_paths; ++i) e->h_path_off[i + 1] = e->h_path_off[i] + len[i];
        CK(e, cudaMemcpyAsync(e->path_off, e->h_path_off.data(), sizeof(int) * (n_paths + 1), cudaMemcpyHostToDevice, e->stream));
        std::vector<unsigned char> t(n_paths, 0);
        if (terminated) memcpy(t.data(), terminated, n_paths);
        CK(e, cudaMemcpyAsync(e->term, t.data(), n_paths, cudaMemcpyHostToDevice, e->stream));
        launch_tstep(e->path_off, n_paths, e->tstep, e->stream);
        e->launches += 1;
        e->n_roll = n; e->n_paths = n_paths; e->n_demo = 0;
        e->have_adv = e->have_white = false;
        // global sample / path counts
        e->h_dsc[DS_CNT] = (double)n; e->h_dsc[DS_CNT + 1] = (double)n_paths;
        CK(e, cudaMemcpyAsync(e->dsc + DS_CNT, e->h_dsc + DS_CNT, 2 * sizeof(double), cudaMemcpyHostToDevice, e->stream));
        if (allreduce(e, e->dsc + DS_CNT, 2, ncclDouble)) return -1;
        CK(e, cudaMemcpyAsync(e->h_dsc + DS_CNT, e->dsc + DS_CNT, 2 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));     // also keeps the host vectors above alive long enough
        e->n_glob_roll = (long long)e->h_dsc[DS_CNT];
        e->n_glob_paths = (int)e->h_dsc[DS_CNT + 1];
        e->h_dsc[DS_SCALE] = 1.0 / (double)e->n_glob_roll;
        e->h_dsc[DS_SCALE + 1] = 1.0 / (double)e->cfg.world_size;
        CK(e, cudaMemcpyAsync(e->dsc + DS_SCALE, e->h_dsc + DS_SCALE, 2 * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    } else {
        e->n_demo = n;
    }
    e->old_cache_valid = false;
    e->uploads += 1;
    return 0;
}

int mjb_batch_upload(mjb_engine* e, int which, int32_t n_paths, const double* const* obs, const double* const* act,
                     const double* const* rew, const int32_t* len, const uint8_t* terminated) {
    if (which != MJB_BATCH_ROLLOUT && which != MJB_BATCH_DEMO) FAIL(e, "bad batch id");
    if (n_paths < 0 || (which == MJB_BATCH_ROLLOUT && n_paths > e->cfg.max_paths)) FAIL(e, "too many paths for max_paths");
    // The tensor-core fit works on its own fp32 feature / target copies, so the NEXT batch may be uploaded while it is
    // still running (sampler hand-off overlapped with the previous step's fit); only the FMA fallback kernel reads
    // the rollout rows in place and has to be joined first.  Demonstration rows live behind the rollout rows.
    if (which == MJB_BATCH_ROLLOUT && e->fit_in_flight && e->fit_reads_batch && mjb_vf_fit_end(e, nullptr)) return -1;
    long long n = 0;
    for (int i = 0; i < n_paths; ++i) { if (len[i] < 0) FAIL(e, "negative path length"); n += len[i]; }
    const long long row0 = which == MJB_BATCH_DEMO ? e->n_roll : 0;
    if (row0 + n > e->cap) FAIL(e, "batch exceeds max_samples");
    CK(e, cudaSetDevice(e->cfg.device));
    // Pack on the fly (samplers/core.py:85-92 path dicts -> batch_reinforce.py:180-182 concat order): each field streams
    // through a double-buffered pinned ring; a few host threads gather the per-path float64 arrays into the slot --
    // observations and actions are rounded to fp32 right there (the reference's `.float()`), so half the bytes cross
    // PCIe and no device-side cast pass is needed -- while the DMA of the previous slot is in flight.
    std::vector<size_t> pre((size_t)n_paths + 1, 0);
    for (int i = 0; i < n_paths; ++i) pre[i + 1] = pre[i] + (size_t)len[i];
    unsigned hw = std::thread::hardware_concurrency();
    int nthr = (int)std::min<unsigned>(8u, std::max<unsigned>(1u, hw));
    if (const char* env = getenv("MJRL_B200_UPLOAD_THREADS")) nthr = std::max(1, atoi(env));
    struct Field { const double* const* src; int width; int kind; };
    const Field fields[3] = {{rew, 1, 2}, {obs, e->cfg.obs_dim, 0}, {act, e->cfg.act_dim, 1}};
    cudaEvent_t done[2] = {e->ev[4], e->ev[5]};
    int slot = 0, used[2] = {0, 0};
    for (const Field& f : fields) {
        if (!f.src) continue;
        if (f.kind == 2 && which == MJB_BATCH_DEMO) continue;
        const bool to_f32 = f.kind != 2;
        const size_t esz = to_f32 ? sizeof(float) : sizeof(double);
        const size_t cap_el = e->pinned_bytes / esz;
        const size_t total_el = (size_t)n * f.width;
        char* dst_dev = f.kind == 2 ? reinterpret_cast<char*>(e->rew)
                      : f.kind == 0 ? reinterpret_cast<char*>(e->obs + (size_t)row0 * e->cfg.obs_dim)
                                    : reinterpret_cast<char*>(e->act + (size_t)row0 * e->cfg.act_dim);
        for (size_t el0 = 0; el0 < total_el; el0 += cap_el) {
            const size_t el1 = std::min(total_el, el0 + cap_el);
            if (used[slot]) CK(e, cudaEventSynchronize(done[slot]));
            char* pin = static_cast<char*>(e->pinned) + (size_t)slot * e->pinned_bytes;
            // elements [el0, el1) of the concatenated field, gathered by nthr threads (equal byte ranges)
            auto work = [&](int t, int T) {
                const size_t span = el1 - el0;
                size_t a0 = el0 + span * (size_t)t / (size_t)T, a1 = el0 + span * (size_t)(t + 1) / (size_t)T;
                // path containing element a0: last i with pre[i] * width <= a0
                size_t pi = (size_t)(std::upper_bound(pre.begin(), pre.end(), a0 / (size_t)f.width) - pre.begin()) - 1;
                while (a0 < a1) {
                    const size_t p_lo = pre[pi] * (size_t)f.width, p_hi = pre[pi + 1] * (size_t)f.width;
                    const size_t take = std::min(a1, p_hi) - a0;
                    const double* sp = f.src[pi] + (a0 - p_lo);
                    if (to_f32) {
                        float* dp = reinterpret_cast<float*>(pin) + (a0 - el0);
                        for (size_t k = 0; k < take; ++k) dp[k] = (float)sp[k];
                    } else {
                        memcpy(reinterpret_cast<double*>(pin) + (a0 - el0), sp, take * sizeof(double));
                    }
                    a0 += take;
                    if (a0 == p_hi) ++pi;
                }
            };
            const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)nthr, (el1 - el0) / 65536 + 1));
            if (T == 1) work(0, 1);
            else {
                std::vector<std::thread> pool;
                for (int t = 1; t < T; ++t) pool.emplace_back(work, t, T);
                work(0, T);
                for (auto& th : pool) th.join();
            }
            const size_t bytes = (el1 - el0) * esz;
            CK(e, cudaMemcpyAsync(dst_dev + el0 * esz, pin, bytes, cudaMemcpyHostToDevice, e->stream));
            e->h2d_bytes += (long long)bytes;
            CK(e, cudaEventRecord(done[slot], e->stream));
            used[slot] = 1;
            slot ^= 1;
        }
    }
    // the pinned slots must not be refilled by a later call before these copies have landed
    for (int sl = 0; sl < 2; ++sl) if (used[sl]) CK(e, cudaEventSynchronize(done[sl]));
    return finish_upload(e, which, n_paths, len, terminated, n);
}

int mjb_batch_upload_rollouts(mjb_engine* e, int32_t n_traj, int32_t horizon, const void* obs, const void* act, const void* rew,
                              int is_f64, const int32_t* len, const uint8_t* terminated) {
    if (n_traj < 0 || n_traj > e->cfg.max_paths) FAIL(e, "too many paths for max_paths");
    if (horizon < 1) FAIL(e, "bad horizon");
    if (e->fit_in_flight && e->fit_reads_batch && mjb_vf_fit_end(e, nullptr)) return -1;
    if (is_host_ptr(obs) || is_host_ptr(act) || is_host_ptr(rew))
        FAIL(e, "mjb_batch_upload_rollouts takes DEVICE arrays (host trajectories go through mjb_batch_upload)");
    long long n = 0;
    std::vector<int32_t> lens((size_t)n_traj, horizon);
    for (int i = 0; i < n_traj; ++i) {
        if (len) { if (len[i] < 0 || len[i] > horizon) FAIL(e, "path length outside [0, horizon]"); lens[i] = len[i]; }
        n += lens[i];
    }
    if (n > e->cap) FAIL(e, "batch exceeds max_samples");
    CK(e, cudaSetDevice(e->cfg.device));
    // path offsets first (the pack kernels read them), then three device-to-device packs: nothing crosses PCIe
    e->h_path_off.assign((size_t)n_traj + 1, 0);
    for (int i = 0; i < n_traj; ++i) e->h_path_off[i + 1] = e->h_path_off[i] + lens[i];
    CK(e, cudaMemcpyAsync(e->path_off, e->h_path_off.data(), sizeof(int) * (n_traj + 1), cudaMemcpyHostToDevice, e->stream));
    launch_pack_rollouts(obs, is_f64, horizon, e->cfg.obs_dim, e->path_off, n_traj, e->obs, 0, e->stream);
    launch_pack_rollouts(act, is_f64, horizon, e->cfg.act_dim, e->path_off, n_traj, e->act, 0, e->stream);
    launch_pack_rollouts(rew, is_f64, horizon, 1, e->path_off, n_traj, e->rew, 1, e->stream);
    e->launches += 3;
    CK(e, cudaGetLastError());
    return finish_upload(e, MJB_BATCH_ROLLOUT, n_traj, lens.data(), terminated, n);
}

int mjb_batch_upload_flat(mjb_engine* e, int which, int32_t n_paths, const double* obs, const double* act,
                          const double* rew, const int32_t* len, const uint8_t* terminated) {
    if (which != MJB_BATCH_ROLLOUT && which != MJB_BATCH_DEMO) FAIL(e, "bad batch id");
    if (n_paths < 0 || (which == MJB_BATCH_ROLLOUT && n_paths > e->cfg.max_paths)) FAIL(e, "too many paths for max_paths");
    if (which == MJB_BATCH_ROLLOUT && e->fit_in_flight && e->fit_reads_batch && mjb_vf_fit_end(e, nullptr)) return -1;
    long long n = 0;
    for (int i = 0; i < n_paths; ++i) n += len[i];
    const long long row0 = which == MJB_BATCH_DEMO ? e->n_roll : 0;
    if (row0 + n > e->cap) FAIL(e, "batch exceeds max_samples");
    CK(e, cudaSetDevice(e->cfg.device));
    if (copy_in(e, e->stage64, obs, sizeof(double) * n * e->cfg.obs_dim)) return -1;
    launch_f64_to_f32(e->stage64, e->obs + (size_t)row0 * e->cfg.obs_dim, n * e->cfg.obs_dim, e->stream);
    if (copy_in(e, e->stage64, act, sizeof(double) * n * e->cfg.act_dim)) return -1;
    launch_f64_to_f32(e->stage64, e->act + (size_t)row0 * e->cfg.act_dim, n * e->cfg.act_dim, e->stream);
    if (rew && which == MJB_BATCH_ROLLOUT && copy_in(e, e->rew, rew, sizeof(double) * n)) return -1;
    e->launches += 2;
    return finish_upload(e, which, n_paths, len, terminated, n);
}

int mjb_batch_set_advantages(mjb_engine* e, const double* adv_concat) {
    if (copy_in(e, e->adv, adv_concat, sizeof(double) * e->n_roll)) return -1;
    e->have_adv = true; e->have_white = false;
    return 0;
}

int mjb_batch_set_adv_white(mjb_engine* e, const float* adv_white) {
    if (copy_in(e, e->adv_white, adv_white, sizeof(float) * e->n_roll)) return -1;
    e->have_white = true;
    return 0;
}

int mjb_batch_set_baseline(mjb_engine* e, const float* base_concat) {
    if (copy_in(e, e->base, base_concat, sizeof(float) * e->n_roll)) return -1;
    return 0;
}

int mjb_batch_set_returns(mjb_engine* e, const double* ret_concat) {
    if (e->fit_in_flight && e->fit_reads_batch && mjb_vf_fit_end(e, nullptr)) return -1;   // fallback kernel: reads the returns in place
    if (copy_in(e, e->ret, ret_concat, sizeof(double) * e->n_roll)) return -1;
    return 0;
}

int64_t mjb_batch_size(const mjb_engine* e, int which) {
    return which == 2 ? e->n_glob_roll : (which == MJB_BATCH_DEMO ? e->n_demo : e->n_roll);
}

// ------------------------------------------------------------------------------- returns / advantages
int mjb_compute_returns(mjb_engine* e, double gamma) {
    if (e->fit_in_flight && e->fit_reads_batch && mjb_vf_fit_end(e, nullptr)) return -1;   // fallback kernel: reads the returns in place
    launch_returns(e->rew, e->path_off, e->n_paths, gamma, e->ret, e->stream);
    e->launches += 1;
    CK(e, cudaGetLastError());
    return 0;
}

int mjb_vf_fit_end(mjb_engine* e, double* err_after);

static int vf_predict_impl(mjb_engine* e);

int mjb_vf_predict(mjb_engine* e) {
    if (e->fit_in_flight && mjb_vf_fit_end(e, nullptr)) return -1;
    return vf_predict_impl(e);
}

// Predictions with the weights of the last COMPLETED fit, without joining a fit in flight: the kernel reads the prepared
// copy (vf_prep) that only mjb_vf_fit_end / mjb_vf_set_state refresh, never the live weights the fit is updating.
int mjb_vf_predict_prefit(mjb_engine* e) { return vf_predict_impl(e); }

static int vf_predict_impl(mjb_engine* e) {
    if (e->occ[MODE_VF] == 0) {
        e->occ[MODE_VF] = occupancy_any(e->vfH, MODE_VF, e->VPL.YR);
        if (e->occ[MODE_VF] <= 0) FAIL(e, "vf kernel does not fit");
    }
    const int MT = mlp_tile_rows_for(e->vfH);
    const long long tiles = (e->n_roll + MT - 1) / MT;
    const int sms = e->num_sms - (e->fit_in_flight ? e->vf_sms : 0);
    const int grid = (int)std::max<long long>(1, std::min<long long>(tiles, (long long)e->occ[MODE_VF] * sms));
    MlpArgs a;
    memset(&a, 0, sizeof(a));
    a.L = e->VPL; a.P = e->vf_prep; a.obs = e->obs; a.obs_dim = e->cfg.obs_dim; a.tstep = e->tstep; a.n = e->n_roll;
    a.vf_out = e->base;
    cudaError_t ce = launch_mlp_any(e->vfH, MODE_VF, a, grid, e->stream);
    if (ce != cudaSuccess) FAIL(e, std::string("vf predict launch: ") + cudaGetErrorString(ce));
    e->launches += 1;
    return 0;
}

int mjb_compute_advantages(mjb_engine* e, double gamma, double gae_lambda, int use_gae) {
    launch_advantages(e->rew, e->base, e->ret, e->path_off, e->term, e->n_paths, gamma, gamma * gae_lambda, use_gae,
                      e->adv, e->stream);
    e->launches += 1;
    e->have_adv = true; e->have_white = false;
    CK(e, cudaGetLastError());
    return 0;
}

static int d2any(mjb_engine* e, void* dst, const void* src, size_t bytes) {
    if (is_host_ptr(dst)) e->d2h_bytes += (long long)bytes;
    CK(e, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}
int mjb_get_returns(mjb_engine* e, double* out) { return d2any(e, out, e->ret, sizeof(double) * e->n_roll); }
int mjb_get_baseline(mjb_engine* e, float* out) { return d2any(e, out, e->base, sizeof(float) * e->n_roll); }
int mjb_get_advantages(mjb_engine* e, double* out) { return d2any(e, out, e->adv, sizeof(double) * e->n_roll); }
int mjb_get_adv_white(mjb_engine* e, float* out) { return d2any(e, out, e->adv_white, sizeof(float) * e->n_roll); }

int mjb_process_paths(mjb_engine* e, mjb_batch_stats* out) {
    if (!e->have_adv) FAIL(e, "mjb_process_paths: advantages not set");
    // Everything stays on the device and on the stream: mean, then population variance about the mean (two passes, like
    // numpy's std), whitening, per-path return statistics; the cross-rank reductions are NCCL calls on the same stream.
    // ONE host round trip at the end brings the seven scalars back.
    const double inv_n = 1.0 / (double)e->n_glob_roll, inv_p = 1.0 / (double)e->n_glob_paths;
    launch_moments(e->adv, e->n_roll, nullptr, e->mom_scratch, e->dsc + DS_MOM, e->stream);
    if (allreduce(e, e->dsc + DS_MOM, 2, ncclDouble)) return -1;
    launch_stats_finalize(e->dsc + DS_MOM, inv_n, e->dsc + DS_STATS, 0, e->stream);
    launch_moments(e->adv, e->n_roll, e->dsc + DS_STATS, e->mom_scratch, e->dsc + DS_MOM, e->stream);
    if (allreduce(e, e->dsc + DS_MOM, 2, ncclDouble)) return -1;
    launch_stats_finalize(e->dsc + DS_MOM, inv_n, e->dsc + DS_STATS, 1, e->stream);
    launch_whiten(e->adv, e->n_roll, e->dsc + DS_STATS, e->adv_white, e->stream);
    e->have_white = true;
    // path-return statistics (batch_reinforce.py:188-192)
    launch_path_sums(e->rew, e->path_off, e->n_paths, e->path_ret, e->stream);
    launch_path_stats(e->path_ret, e->n_paths, inv_p, e->dsc + DS_RET, 0, e->stream);
    if (e->comm) {
        if (allreduce(e, e->dsc + DS_RET, 1, ncclDouble, ncclSum)) return -1;
        if (allreduce(e, e->dsc + DS_RET + 1, 2, ncclDouble, ncclMax)) return -1;
    }
    launch_path_stats(e->path_ret, e->n_paths, inv_p, e->dsc + DS_RET, 1, e->stream);
    if (allreduce(e, e->dsc + DS_RET + 3, 1, ncclDouble)) return -1;
    e->launches += 11;
    CK(e, cudaGetLastError());
    if (out) {
        CK(e, cudaMemcpyAsync(e->h_dsc + DS_STATS, e->dsc + DS_STATS, 2 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaMemcpyAsync(e->h_dsc + DS_RET, e->dsc + DS_RET, 4 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        e->d2h_bytes += 6 * (long long)sizeof(double);
        CK(e, cudaStreamSynchronize(e->stream));
        const double* h = e->h_dsc + DS_RET;
        out->mean_return = h[0] * inv_p; out->std_return = std::sqrt(h[3] * inv_p);
        out->min_return = -h[1]; out->max_return = h[2];
        out->adv_mean = e->h_dsc[DS_STATS]; out->adv_std = e->h_dsc[DS_STATS + 1]; out->n_samples_global = e->n_glob_roll;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------ policy
int mjb_policy_dim(const mjb_engine* e) { return e->d; }

int mjb_policy_set_params(mjb_engine* e, const float* theta, int set_new, int set_old) {
    if (set_new && set_params(e, e->pnew, theta)) return -1;
    if (set_old && set_params(e, e->pold, theta)) return -1;
    if (set_new && set_old) e->old_equals_new = e->transforms_equal;
    else if (set_new || set_old) e->old_equals_new = false;
    if (set_old) e->old_cache_valid = false;
    return 0;
}

int mjb_policy_get_params(mjb_engine* e, float* theta_out, int which_old) {
    return d2any(e, theta_out, which_old ? e->pold.theta : e->pnew.theta, sizeof(float) * e->d);
}

int mjb_policy_set_transforms(mjb_engine* e, const float* in_shift, const float* in_scale, const float* out_shift,
                              const float* out_scale, int which_old) {
    ParamSet& ps = which_old ? e->pold : e->pnew;
    const size_t O = e->cfg.obs_dim, A = e->cfg.act_dim;
    if (in_shift && copy_in(e, ps.in_shift, in_shift, O * sizeof(float))) return -1;
    if (in_scale && copy_in(e, ps.in_scale, in_scale, O * sizeof(float))) return -1;
    if (out_shift && copy_in(e, ps.out_shift, out_shift, A * sizeof(float))) return -1;
    if (out_scale && copy_in(e, ps.out_scale, out_scale, A * sizeof(float))) return -1;
    CK(e, cudaStreamSynchronize(e->stream));
    if (in_shift || in_scale) {
        std::vector<float> hs(O), hc(O);
        CK(e, cudaMemcpy(hs.data(), ps.in_shift, O * sizeof(float), cudaMemcpyDeviceToHost));
        CK(e, cudaMemcpy(hc.data(), ps.in_scale, O * sizeof(float), cudaMemcpyDeviceToHost));
        ps.in_ident = true;
        for (size_t i = 0; i < O; ++i) ps.in_ident = ps.in_ident && hs[i] == 0.0f && hc[i] == 1.0f;
    }
    e->transforms_equal = false;       // conservative: the reference updates only policy.model (A10)
    e->old_equals_new = false;
    if (which_old) e->old_cache_valid = false;
    return 0;
}

int mjb_policy_eval(mjb_engine* e, double out[2]) { return eval_device(e, out); }

int mjb_policy_vpg(mjb_engine* e, int include_demo, double demo_lam, float* g_out) {
    if (vpg_device(e, include_demo, demo_lam, nullptr)) return -1;
    if (g_out) return d2any(e, g_out, e->g, sizeof(float) * e->d);
    return 0;
}

int mjb_policy_fvp(mjb_engine* e, const float* v, float damping, const int32_t* idx, int64_t n_idx, float* out) {
    if (copy_in(e, e->tmpv, v, sizeof(float) * e->d)) return -1;
    const int* idx_dev = nullptr;
    if (idx) {
        if (upload_idx(e, idx, n_idx)) return -1;
        if (set_subsample_scale(e, n_idx)) return -1;
        idx_dev = e->idx_dev;
    }
    if (fvp_device(e, e->tmpv, idx_dev, n_idx, e->Fp)) return -1;
    // + damping * v  (npg_cg.py:81)
    e->h_dsc[DS_ALPHA] = (double)damping;
    CK(e, cudaMemcpyAsync(e->dsc + DS_ALPHA, e->h_dsc + DS_ALPHA, sizeof(double), cudaMemcpyHostToDevice, e->stream));
    launch_axpy_clamp(e->Fp, e->tmpv, e->dsc + DS_ALPHA, 1.0, e->d, 0, 0.0f, e->Fp, e->stream);
    e->launches += 1;
    if (d2any(e, out, e->Fp, sizeof(float) * e->d)) return -1;
    const int slot = (int)((e->fvp_count - 1) % mjb_engine::kFvpRing);
    cudaEventElapsedTime(&e->last_fvp_ms, e->fvp_ev[slot][0], e->fvp_ev[slot][1]);
    return 0;
}

int mjb_policy_cg(mjb_engine* e, const float* b, int iters, float damping, float residual_tol, const int32_t* idx,
                  int64_t n_idx, float* x_out) {
    if (b && copy_in(e, e->g, b, sizeof(float) * e->d)) return -1;
    const int* idx_dev = nullptr;
    if (idx) {
        if (upload_idx(e, idx, (long long)iters * n_idx)) return -1;
        if (set_subsample_scale(e, e->hvp_len.empty() ? n_idx : e->hvp_len[0])) return -1;
        idx_dev = e->idx_dev;
    }
    if (cg_device(e, e->g, iters, damping, residual_tol, idx_dev, n_idx)) return -1;
    if (x_out) return d2any(e, x_out, e->x, sizeof(float) * e->d);
    return 0;
}

int mjb_policy_step(mjb_engine* e, int algo, double step_size_or_kl, double const_learn_rate, int cg_iters,
                    float damping, double demo_lam, const int32_t* hvp_idx, int64_t n_idx, mjb_step_stats* out) {
    if (algo < MJB_ALGO_NPG || algo > MJB_ALGO_DAPG) FAIL(e, "bad algo");
    mjb_step_stats st;
    memset(&st, 0, sizeof(st));
    const long long fvp0 = e->fvp_count;
    CK(e, cudaEventRecord(e->ev[0], e->stream));
    if (vpg_device(e, algo == MJB_ALGO_DAPG, demo_lam, &st.surr_before)) return -1;
    CK(e, cudaEventRecord(e->ev[1], e->stream));
    const int* idx_dev = nullptr;
    if (hvp_idx) {
        if (upload_idx(e, hvp_idx, (long long)cg_iters * n_idx)) return -1;
        if (set_subsample_scale(e, e->hvp_len.empty() ? n_idx : e->hvp_len[0])) return -1;
        idx_dev = e->idx_dev;
    }
    if (cg_device(e, e->g, cg_iters, damping, 1e-10f, idx_dev, n_idx)) return -1;
    launch_dot(e->g, e->x, e->d, e->dsc + DS_DOT, e->stream);
    e->launches += 1;
    CK(e, cudaEventRecord(e->ev[2], e->stream));
    CK(e, cudaMemcpyAsync(e->h_dsc + DS_CG, e->dsc + DS_CG, 8 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    st.cg_iters_run = (int)e->h_dsc[DS_CG + 2];
    const float gx = (float)e->h_dsc[DS_DOT];
    st.vpg_dot_npg = gx;
    // step size in the reference's fp32 scalar arithmetic (npg_cg.py:128-133, trpo.py:102-103, dapg.py:111-112)
    float alpha;
    double delta;
    if (algo == MJB_ALGO_NPG && const_learn_rate > 0.0) {
        alpha = (float)const_learn_rate;
        delta = (double)(alpha * alpha * gx);
    } else {
        delta = algo == MJB_ALGO_NPG ? step_size_or_kl : 2.0 * step_size_or_kl;
        alpha = sqrtf(fabsf((float)delta / (gx + 1e-20f)));
    }
    auto apply = [&](float al) -> int {
        e->h_dsc[DS_ALPHA] = (double)al;
        CK(e, cudaMemcpyAsync(e->dsc + DS_ALPHA, e->h_dsc + DS_ALPHA, sizeof(double), cudaMemcpyHostToDevice, e->stream));
        launch_axpy_clamp(e->pold.theta, e->x, e->dsc + DS_ALPHA, 1.0, e->d, e->A, e->cfg.min_log_std, e->pnew.theta, e->stream);
        e->launches += 1;
        if (set_params(e, e->pnew, nullptr)) return -1;
        e->old_equals_new = false;
        return 0;
    };
    double ev[2] = {0, 0};
    if (algo == MJB_ALGO_TRPO) {
        // trpo.py:108-120: shrink by 0.9 until KL < kl_dist (at most 100 probes, then alpha = 0)
        bool accepted = false;
        for (int k = 0; k < 100; ++k) {
            if (apply(alpha) || eval_device(e, ev)) return -1;
            if (ev[1] < step_size_or_kl) { accepted = true; break; }
            alpha = 0.9f * alpha;
            st.backtracks += 1;
            if (k == 99) alpha = 0.0f;
        }
        if (!accepted) { if (apply(alpha) || eval_device(e, ev)) return -1; }
    } else {
        if (apply(alpha) || eval_device(e, ev)) return -1;
    }
    CK(e, cudaEventRecord(e->ev[3], e->stream));
    st.alpha = alpha; st.delta = delta; st.surr_after = ev[0]; st.kl_dist = ev[1];
    // old <- new (set_param_values(new, set_new=True, set_old=True), npg_cg.py:142)
    CK(e, cudaMemcpyAsync(e->pold.theta, e->pnew.theta, sizeof(float) * e->d, cudaMemcpyDeviceToDevice, e->stream));
    CK(e, cudaMemcpyAsync(e->pold.prep, e->pnew.prep, sizeof(float) * e->prep_total, cudaMemcpyDeviceToDevice, e->stream));
    e->old_equals_new = e->transforms_equal;
    e->old_cache_valid = false;
    CK(e, cudaStreamSynchronize(e->stream));
    cudaEventElapsedTime(&st.time_vpg_ms, e->ev[0], e->ev[1]);
    cudaEventElapsedTime(&st.time_npg_ms, e->ev[1], e->ev[2]);
    cudaEventElapsedTime(&st.time_eval_ms, e->ev[2], e->ev[3]);
    if (e->last_cg_graph) {
        const auto& evs = e->last_cg_graph->ev;
        for (size_t k = 0; k + 1 < evs.size(); k += 2) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, evs[k], evs[k + 1]) != cudaSuccess) { cudaGetLastError(); continue; }
            st.fvp_kernel_ms_sum += ms;
            st.fvp_launches += 1;
            e->last_fvp_ms = ms;
        }
    }
    for (long long k = std::max(fvp0, e->fvp_count - mjb_engine::kFvpRing); k < e->fvp_count; ++k) {
        float ms = 0.f;
        const int slot = (int)(k % mjb_engine::kFvpRing);
        cudaEventElapsedTime(&ms, e->fvp_ev[slot][0], e->fvp_ev[slot][1]);
        st.fvp_kernel_ms_sum += ms;
        st.fvp_launches += 1;
        e->last_fvp_ms = ms;
    }
    if (out) *out = st;
    return 0;
}

// ------------------------------------------------------------------------ minibatch-Adam policy training
int mjb_policy_sgd(mjb_engine* e, int loss_kind, const int32_t* idx, int64_t steps, int batch, float lr, float clip_coef,
                   float* loss_out, float* clip_frac_out) {
    if (e->cfg.world_size > 1) FAIL(e, "mjb_policy_sgd: single-GPU only (the chain is not replicated across ranks)");
    if (e->linear) FAIL(e, "mjb_policy_sgd: the minibatch-Adam kernel covers the Gaussian MLP policy, not LinearPolicy");
    if (loss_kind != SGD_PPO && loss_kind != SGD_BC_MLE && loss_kind != SGD_BC_MSE) FAIL(e, "mjb_policy_sgd: bad loss kind");
    if (batch < 1 || batch > 64) FAIL(e, "mjb_policy_sgd: minibatch size must be in [1, 64]");
    if (steps < 0 || steps > 0x7fffffffLL) FAIL(e, "mjb_policy_sgd: bad step count");
    if (policy_sgd_smem_bytes(e->cfg.obs_dim, e->cfg.hidden[0], e->cfg.hidden[1], e->A) > policy_sgd_max_smem())
        FAIL(e, "mjb_policy_sgd: obs_dim too large for the kernel's shared-memory activations at this width");
    if (e->n_roll <= 0) FAIL(e, "mjb_policy_sgd: no batch resident");
    if (loss_kind == SGD_PPO && !e->have_white) FAIL(e, "mjb_policy_sgd: PPO needs mjb_process_paths first");
    if (steps == 0) return 0;
    if (loss_kind == SGD_PPO && ensure_old_cache(e, e->n_roll)) return -1;    // LL under the old policy and transforms
    const long long total = steps * (long long)batch;
    if (total > e->sgd_idx_cap) {
        if (e->sgd_idx) cudaFree(e->sgd_idx);
        e->sgd_idx = nullptr; e->sgd_idx_cap = 0;
        CK(e, cudaMalloc(&e->sgd_idx, sizeof(int) * total));
        e->sgd_idx_cap = total;
    }
    if (copy_in(e, e->sgd_idx, idx, sizeof(int) * total)) return -1;
    if ((loss_out || clip_frac_out) && steps > e->sgd_out_cap) {
        if (e->sgd_out) cudaFree(e->sgd_out);
        e->sgd_out = nullptr; e->sgd_out_cap = 0;
        CK(e, cudaMalloc(&e->sgd_out, sizeof(float) * 2 * steps));
        e->sgd_out_cap = steps;
    }
    PolicySgdArgs a;
    a.K0 = e->cfg.obs_dim; a.h1 = e->cfg.hidden[0]; a.h2 = e->cfg.hidden[1]; a.A = e->A; a.loss_kind = loss_kind;
    a.obs = e->obs; a.act = e->act; a.adv = e->adv_white; a.ll_old = e->ll_old;
    a.in_shift = e->pnew.in_shift; a.in_scale = e->pnew.in_scale; a.out_shift = e->pnew.out_shift; a.out_scale = e->pnew.out_scale;
    a.idx = e->sgd_idx; a.steps = steps; a.batch = batch;
    a.lr = lr; a.beta1 = 0.9f; a.beta2 = 0.999f; a.eps = 1e-8f;
    a.clip_lo = (float)(1.0 - (double)clip_coef); a.clip_hi = (float)(1.0 + (double)clip_coef);
    a.step0 = e->sgd_step;
    a.theta = e->pnew.theta; a.m = e->sgd_m; a.v = e->sgd_v; a.wT = e->sgd_wT;
    a.loss_out = loss_out ? e->sgd_out : nullptr;
    a.clip_out = clip_frac_out ? e->sgd_out + steps : nullptr;     // (all zero for the BC losses)
    CK(e, cudaEventRecord(e->sgd_ev[0], e->stream));
    const cudaError_t ce = launch_policy_sgd(a, e->stream);
    if (ce != cudaSuccess) FAIL(e, std::string("policy_sgd launch: ") + cudaGetErrorString(ce));
    CK(e, cudaEventRecord(e->sgd_ev[1], e->stream));
    e->launches += 1;
    e->sgd_timed = true;
    e->sgd_step += steps;
    // theta_new changed in place: refresh what is keyed on it (no log_std clamp here -- the reference evaluates
    // surr_after / kl_dist before set_param_values clamps, ppo_clip.py:99-102)
    launch_prep_mlp(e->pnew.theta, e->PL, e->pnew.prep, e->stream);
    e->launches += 1;
    if (e->tc_ok) { launch_tc_prep(e->pnew.theta, e->PL, nullptr, e->tc_prep_new, e->stream); e->launches += 1; }
    e->old_equals_new = false;
    CK(e, cudaGetLastError());
    if (loss_out) CK(e, cudaMemcpyAsync(loss_out, e->sgd_out, sizeof(float) * steps, cudaMemcpyDefault, e->stream));
    if (clip_frac_out) CK(e, cudaMemcpyAsync(clip_frac_out, a.clip_out, sizeof(float) * steps, cudaMemcpyDefault, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

int mjb_policy_adam_set(mjb_engine* e, const float* m, const float* v, int64_t step) {
    if (m && copy_in(e, e->sgd_m, m, sizeof(float) * e->d)) return -1;
    if (v && copy_in(e, e->sgd_v, v, sizeof(float) * e->d)) return -1;
    if (step >= 0) e->sgd_step = step;
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

int mjb_policy_adam_get(mjb_engine* e, float* m, float* v, int64_t* step) {
    if (m && d2any(e, m, e->sgd_m, sizeof(float) * e->d)) return -1;
    if (v && d2any(e, v, e->sgd_v, sizeof(float) * e->d)) return -1;
    if (step) *step = e->sgd_step;
    return 0;
}

int mjb_policy_bc_loss(mjb_engine* e, int loss_kind, double* out) {
    if (loss_kind != SGD_BC_MLE && loss_kind != SGD_BC_MSE) FAIL(e, "mjb_policy_bc_loss: loss kind must be MLE or MSE");
    if (e->cfg.world_size > 1) FAIL(e, "mjb_policy_bc_loss: single-GPU only");
    if (e->n_roll <= 0) FAIL(e, "mjb_policy_bc_loss: no batch resident");
    // the EVAL tile kernel writes per-row LL / mean of theta_new into the old-policy cache buffers: the cache is void after
    const int grid = run_policy(e, MODE_EVAL, e->pnew, nullptr, e->n_roll, nullptr, nullptr, OLD_WRITE);
    if (grid < 0) return -1;
    e->old_cache_valid = false;
    if (launch_bc_loss_sum(e->ll_old, e->mu_old, e->act, e->n_roll, e->A, loss_kind, e->mom_scratch, e->dsc + DS_BCLOSS,
                           e->stream) != cudaSuccess) FAIL(e, "bc loss launch failed");
    e->launches += 2;
    CK(e, cudaMemcpyAsync(e->h_dsc + DS_BCLOSS, e->dsc + DS_BCLOSS, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    const double sum = e->h_dsc[DS_BCLOSS];
    // torch.mean in fp32: round the mean to fp32 like the reference's scalar
    *out = loss_kind == SGD_BC_MLE ? (double)(float)(-sum / (double)e->n_roll)
                                   : (double)(float)(sum / ((double)e->n_roll * (double)e->A));
    return 0;
}

int mjb_policy_sgd_timing(mjb_engine* e, float* last_ms) {
    *last_ms = 0.f;
    if (!e->sgd_timed) return 0;
    CK(e, cudaEventSynchronize(e->sgd_ev[1]));
    CK(e, cudaEventElapsedTime(last_ms, e->sgd_ev[0], e->sgd_ev[1]));
    return 0;
}

int mjb_policy_set_hvp_lengths(mjb_engine* e, const int64_t* n_each, int iters) {
    e->hvp_len.clear();
    if (n_each) for (int i = 0; i < iters; ++i) e->hvp_len.push_back((long long)n_each[i]);
    return 0;
}

int mjb_policy_last_vectors(mjb_engine* e, float* vpg_out, float* npg_out) {
    if (vpg_out && d2any(e, vpg_out, e->g, sizeof(float) * e->d)) return -1;
    if (npg_out && d2any(e, npg_out, e->x, sizeof(float) * e->d)) return -1;
    return 0;
}

// ------------------------------------------------------------------------------------------ baseline
int mjb_vf_dim(const mjb_engine* e) { return e->vf_d; }

int mjb_vf_set_state(mjb_engine* e, const float* w, const float* m, const float* v, int64_t step) {
    if (e->fit_in_flight && mjb_vf_fit_end(e, nullptr)) return -1;
    if (w && copy_in(e, e->vf_w, w, sizeof(float) * e->vf_d)) return -1;
    if (m && copy_in(e, e->vf_m, m, sizeof(float) * e->vf_d)) return -1;
    if (v && copy_in(e, e->vf_v, v, sizeof(float) * e->vf_d)) return -1;
    if (step >= 0) e->vf_step = step;
    launch_prep_mlp(e->vf_w, e->VPL, e->vf_prep, e->stream);
    e->launches += 1;
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

int mjb_vf_get_state(mjb_engine* e, float* w, float* m, float* v, int64_t* step) {
    if (e->fit_in_flight && mjb_vf_fit_end(e, nullptr)) return -1;
    if (w && d2any(e, w, e->vf_w, sizeof(float) * e->vf_d)) return -1;
    if (m && d2any(e, m, e->vf_m, sizeof(float) * e->vf_d)) return -1;
    if (v && d2any(e, v, e->vf_v, sizeof(float) * e->vf_d)) return -1;
    if (step) *step = e->vf_step;
    return 0;
}

static int vf_error(mjb_engine* e, double* err) {
    if (mjb_vf_predict(e)) return -1;
    launch_vf_error(e->ret, e->base, e->n_roll, e->mom_scratch, e->dsc + DS_VF, e->stream);
    e->launches += 2;
    if (allreduce(e, e->dsc + DS_VF, 2, ncclDouble)) return -1;
    CK(e, cudaMemcpyAsync(e->h_dsc + DS_VF, e->dsc + DS_VF, 2 * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(e, cudaStreamSynchronize(e->stream));
    *err = e->h_dsc[DS_VF] / (e->h_dsc[DS_VF + 1] + 1e-8);
    return 0;
}

// Launch the whole fit (all epochs).  Communication, permutation upload and feature building run on the main
// stream; the sequential Adam kernels run on `fs` (== main stream for the synchronous call, the side stream for
// mjb_vf_fit_begin) behind an event, so the policy update can proceed concurrently on the remaining SMs.
static int vf_fit_launch(mjb_engine* e, const int32_t* perms, int epochs, int batch_size, float lr, float reg_coef,
                         cudaStream_t fs) {
    const long long N = e->n_glob_roll;
    const int steps = (int)(N / batch_size) - 1;            // optimize_model.py:24
    if (steps < 1) FAIL(e, "MLPBaseline.fit needs at least 2*batch_size samples (the reference crashes: optimize_model.py:24,35)");
    const float* fobs = e->obs; const int* ftstep = e->tstep; const double* fret = e->ret;
    if (e->comm) {
        // replicated sequential fit: gather every rank's (obs, tstep, returns) in rank order
        if (N > e->fit_cap) {
            if (e->fit_obs) { cudaFree(e->fit_obs); cudaFree(e->fit_tstep); cudaFree(e->fit_ret); }
            e->fit_cap = N;
            CK(e, cudaMalloc(&e->fit_obs, sizeof(float) * N * e->cfg.obs_dim));
            CK(e, cudaMalloc(&e->fit_tstep, sizeof(int) * N));
            CK(e, cudaMalloc(&e->fit_ret, sizeof(double) * N));
        }
        std::vector<double> cnt(e->cfg.world_size, 0.0);
        cnt[e->cfg.rank] = (double)e->n_roll;
        double* dcnt = e->mom_scratch;                       // reuse (world_size <= 512)
        CK(e, cudaMemcpyAsync(dcnt, cnt.data(), sizeof(double) * cnt.size(), cudaMemcpyHostToDevice, e->stream));
        if (allreduce(e, dcnt, cnt.size(), ncclDouble)) return -1;
        CK(e, cudaMemcpyAsync(cnt.data(), dcnt, sizeof(double) * cnt.size(), cudaMemcpyDeviceToHost, e->stream));
        CK(e, cudaStreamSynchronize(e->stream));
        NK(e, g_nccl.GroupStart());
        long long off = 0;
        for (int r = 0; r < e->cfg.world_size; ++r) {
            const long long c = (long long)cnt[r];
            NK(e, g_nccl.Broadcast(e->obs, e->fit_obs + off * e->cfg.obs_dim, c * e->cfg.obs_dim, ncclFloat, r, e->comm, e->stream));
            NK(e, g_nccl.Broadcast(e->tstep, e->fit_tstep + off, c, ncclInt32, r, e->comm, e->stream));
            NK(e, g_nccl.Broadcast(e->ret, e->fit_ret + off, c, ncclDouble, r, e->comm, e->stream));
            off += c;
        }
        NK(e, g_nccl.GroupEnd());
        fobs = e->fit_obs; ftstep = e->fit_tstep; fret = e->fit_ret;
    }
    if ((long long)epochs * N > e->perm_cap) {
        if (e->perm_dev) cudaFree(e->perm_dev);
        e->perm_cap = (long long)epochs * N;
        CK(e, cudaMalloc(&e->perm_dev, sizeof(int) * e->perm_cap));
    }
    // all epochs' permutations go up front (the caller's host buffer is free again when this function returns)
    if (copy_in(e, e->perm_dev, perms, sizeof(int) * (size_t)epochs * N)) return -1;
    if (e->comm) NK(e, g_nccl.Broadcast(e->perm_dev, e->perm_dev, (size_t)epochs * N, ncclInt32, 0, e->comm, e->stream));
    VfFitArgs a;
    a.K = e->cfg.obs_dim + 4; a.H1 = e->cfg.vf_hidden[0]; a.H2 = e->cfg.vf_hidden[1]; a.obs_dim = e->cfg.obs_dim;
    a.obs = fobs; a.tstep = ftstep; a.returns = fret; a.n = N;
    a.steps = steps; a.batch = batch_size; a.lr = lr; a.reg = reg_coef; a.beta1 = 0.9f; a.beta2 = 0.999f; a.eps = 1e-8f;
    a.w = e->vf_w; a.m = e->vf_m; a.v = e->vf_v; a.wT = e->vf_wT; a.loss_out = nullptr;
    // the tensor-core kernel where the shape allows; every other shape runs the single-CTA fp32-FMA kernel
    const bool use_tc = e->vf_tc_on && vf_tc_supported(a.K, a.H1, a.H2, a.batch);
    e->vf_sms = use_tc ? vf_tc_sms(a.K) : 1;
    e->fit_reads_batch = !use_tc && !e->comm;        // (the replicated multi-GPU fit works on gathered copies)
    if (use_tc) {
        if (N > e->vf_feat_cap) {
            if (e->vf_feat) { cudaFree(e->vf_feat); cudaFree(e->vf_ret32); }
            e->vf_feat_cap = N;
            CK(e, cudaMalloc(&e->vf_feat, sizeof(float) * (size_t)N * vf_tc_feat_pitch(a.K)));
            CK(e, cudaMalloc(&e->vf_ret32, sizeof(float) * (size_t)N));
        }
        if (vf_build_features(a, e->vf_feat, e->vf_ret32, e->stream) != cudaSuccess) FAIL(e, "vf feature kernel launch failed");
        e->launches += 1;
        if (e->vf_sms > 1 && !e->vf_ks) CK(e, cudaMalloc(&e->vf_ks, vf_tc_scratch_bytes()));
        if (steps > e->vf_consts_cap) {
            if (e->vf_consts) cudaFree(e->vf_consts);
            e->vf_consts_cap = steps + 1024;
            CK(e, cudaMalloc(&e->vf_consts, sizeof(float4) * (size_t)e->vf_consts_cap));
        }
    }
    CK(e, cudaStreamSynchronize(e->stream));                 // host permutation buffer consumed; inputs of the fit complete
    CK(e, cudaEventRecord(e->fit_ev[0], fs));
    for (int ep = 0; ep < epochs; ++ep) {
        a.perm = e->perm_dev + (size_t)ep * N;
        a.step0 = e->vf_step;
        cudaError_t ce;
        if (use_tc) { ce = launch_vf_fit_tc(a, e->vf_feat, e->vf_ret32, e->vf_consts, e->vf_ks, fs); e->launches += 2; }
        else { ce = launch_vf_fit(a, fs); e->launches += 1; }
        if (ce != cudaSuccess) FAIL(e, std::string("vf fit launch (batch<=64, multiple of 4; sizes must fit 220 KB smem): ") + cudaGetErrorString(ce));
        e->vf_step += steps;
    }
    CK(e, cudaEventRecord(e->fit_ev[1], fs));
    e->fit_timed = true;
    return 0;
}

int mjb_vf_fit_end(mjb_engine* e, double* err_after) {
    if (e->fit_in_flight) {
        CK(e, cudaStreamSynchronize(e->stream_vf));
        e->fit_in_flight = false;
    }
    launch_prep_mlp(e->vf_w, e->VPL, e->vf_prep, e->stream);
    e->launches += 1;
    if (err_after && vf_error(e, err_after)) return -1;
    CK(e, cudaStreamSynchronize(e->stream));
    return 0;
}

int mjb_vf_fit_begin(mjb_engine* e, const int32_t* perms, int epochs, int batch_size, float lr, float reg_coef, double* err_before) {
    if (e->fit_in_flight && mjb_vf_fit_end(e, nullptr)) return -1;
    if (err_before && vf_error(e, err_before)) return -1;
    if (vf_fit_launch(e, perms, epochs, batch_size, lr, reg_coef, e->stream_vf)) return -1;
    e->fit_in_flight = true;
    return 0;
}

int mjb_vf_fit(mjb_engine* e, const int32_t* perms, int epochs, int batch_size, float lr, float reg_coef, double err_out[2]) {
    if (e->fit_in_flight && mjb_vf_fit_end(e, nullptr)) return -1;
    if (err_out && vf_error(e, &err_out[0])) return -1;
    if (vf_fit_launch(e, perms, epochs, batch_size, lr, reg_coef, e->stream)) return -1;
    return mjb_vf_fit_end(e, err_out ? &err_out[1] : nullptr);
}

int mjb_event_record(mjb_engine* e, int slot) {
    if (slot < 0 || slot >= 8) FAIL(e, "event slot out of range");
    CK(e, cudaEventRecord(e->user_ev[slot], e->stream));
    return 0;
}
int mjb_event_elapsed_ms(mjb_engine* e, int slot_a, int slot_b, float* ms) {
    if (slot_a < 0 || slot_a >= 8 || slot_b < 0 || slot_b >= 8) FAIL(e, "event slot out of range");
    CK(e, cudaEventSynchronize(e->user_ev[slot_b]));
    CK(e, cudaEventElapsedTime(ms, e->user_ev[slot_a], e->user_ev[slot_b]));
    return 0;
}

// Developer aid: per-phase clock64 cycle counters of the tensor-core fit kernel.
int mjb_dev_vf_profile(mjb_engine* e, long long* out16, int enable) {
    // enable: 1 = arm the counters, 0 = read the head CTA's 16 counters and disarm, 2 = read K-split helper 0's 16 counters
    static long long* dev = nullptr;
    if (!dev) { CK(e, cudaMalloc(&dev, 32 * sizeof(long long))); }
    if (enable == 1) { CK(e, cudaMemset(dev, 0, 32 * sizeof(long long))); vf_tc_set_prof(dev); return 0; }
    CK(e, cudaStreamSynchronize(e->stream));
    CK(e, cudaMemcpy(out16, dev + (enable == 2 ? 16 : 0), 16 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (enable == 2) return 0;
    vf_tc_set_prof(nullptr);
    return 0;
}

// Developer aid: per-phase cycle counters of the tensor-core linear-policy FVP kernel (summed over CTAs).
int mjb_dev_lin_profile(mjb_engine* e, long long* out8 /* 16 values */, int enable) {
    static unsigned long long* dev = nullptr;
    if (!dev) { CK(e, cudaMalloc(&dev, 16 * sizeof(long long))); }
    if (enable) { CK(e, cudaMemset(dev, 0, 16 * sizeof(long long))); lin_tc_set_prof(dev); return 0; }
    CK(e, cudaStreamSynchronize(e->stream));
    CK(e, cudaMemcpy(out8, dev, 16 * sizeof(long long), cudaMemcpyDeviceToHost));
    lin_tc_set_prof(nullptr);
    return 0;
}

int mjb_policy_set_tensor_cores(mjb_engine* e, int on) {
    e->tc_on = on != 0;
    return (e->tc_ok || !on) ? 0 : 1;       // 1: requested but this shape runs on the fp32 FMA kernels
}

int mjb_vf_set_tensor_cores(mjb_engine* e, int on) {
    e->vf_tc_on = on != 0;
    return 0;
}
int64_t mjb_kernel_launches(const mjb_engine* e) { return e->launches; }
int mjb_transfer_stats(const mjb_engine* e, mjb_transfer_stats_t* out) {
    out->h2d_bytes = e->h2d_bytes; out->d2h_bytes = e->d2h_bytes; out->uploads = e->uploads;
    return 0;
}
int mjb_fvp_timing(mjb_engine* e, float* last_ms) { *last_ms = e->last_fvp_ms; return 0; }
int mjb_vf_fit_timing(mjb_engine* e, float* last_ms) {
    *last_ms = 0.f;
    if (!e->fit_timed) return 0;
    if (e->fit_in_flight && mjb_vf_fit_end(e, nullptr)) return -1;
    CK(e, cudaEventSynchronize(e->fit_ev[1]));
    CK(e, cudaEventElapsedTime(last_ms, e->fit_ev[0], e->fit_ev[1]));
    return 0;
}

}  // extern "C"
