// Minibatch-Adam training of the Gaussian-MLP policy: PPO-clip (algos/ppo_clip.py:88-97) and behaviour cloning
// (algos/behavior_cloning.py:120-127, MLE or MSE loss).  Both loops are long chains of dependent Adam steps on small
// minibatches (10 epochs x N/64 steps for PPO's defaults), the same shape of work as the baseline fit, so this kernel
// follows vf_fit.cu: ONE persistent CTA runs the whole chain.  Per step it gathers the B rows named by the host-drawn
// index block, applies the policy's input transform, runs forward / loss / backward with feature-major activations in
// shared memory, and Adam-updates every parameter from the gradient it just accumulated in registers.  Weights live in
// global memory (L1/L2-resident) in the flat reference layout [W1, b1, W2, b2, W3, b3, log_std], plus transposed copies
// of W1 and W2 so every inner loop reads them coalesced.  Every sum runs in a fixed order (no atomics): a repeated call
// is bit-identical.
#include "adam.cuh"
#include "kernels.h"

namespace mjb {

constexpr int SB = 64;             // max minibatch rows
constexpr int SL = SB + 4;         // row pitch of feature-major activations
constexpr int ST = 1024;           // threads

// out4[n][4 samples q] = sum_k inT[k][4q..] * WT[k][n]
__device__ __forceinline__ float4 sgd_dense(const float* __restrict__ inT, const float* WT, int NOUT, int R, int n, int q) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
    for (int k = 0; k < R; ++k) {
        const float w = WT[k * NOUT + n];
        const float4 x = *reinterpret_cast<const float4*>(inT + k * SL + 4 * q);
        acc.x = fmaf(x.x, w, acc.x); acc.y = fmaf(x.y, w, acc.y); acc.z = fmaf(x.z, w, acc.z); acc.w = fmaf(x.w, w, acc.w);
    }
    return acc;
}

// acc[i][j] += sum_b A[a0 + i][b] * B[b0 + 32 j][b] over all SB columns (columns past the batch are zero): the 4 x 4
// block of W2's gradient a thread owns.  One float4 column group per iteration keeps it inside 64 registers.
__device__ __forceinline__ void sgd_wgrad(float (&acc)[4][4], const float* __restrict__ A, int a0,
                                          const float* __restrict__ B, int b0) {
#pragma unroll 1
    for (int m = 0; m < SB; m += 4) {
        float4 x[4], y[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) x[i] = *reinterpret_cast<const float4*>(A + (a0 + i) * SL + m);
#pragma unroll
        for (int j = 0; j < 4; ++j) y[j] = *reinterpret_cast<const float4*>(B + (b0 + 32 * j) * SL + m);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float t = acc[i][j];
                t = fmaf(x[i].x, y[j].x, t); t = fmaf(x[i].y, y[j].y, t);
                t = fmaf(x[i].z, y[j].z, t); t = fmaf(x[i].w, y[j].w, t);
                acc[i][j] = t;
            }
    }
}

__device__ __forceinline__ float4 tanh4(float4 z, float b) {
    return make_float4(tanhf(z.x + b), tanhf(z.y + b), tanhf(z.z + b), tanhf(z.w + b));
}

template <int KIND>
__global__ void __launch_bounds__(ST, 1) policy_sgd_kernel(const PolicySgdArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int K = a.K0, H1 = a.h1, H2 = a.h2, A = a.A, B = a.batch;
    const int H1p = round_up(H1, 128), H2p = round_up(H2, 128);   // rows padded so 128-wide wgrad blocks stay in bounds
    const int QB = (B + 3) / 4;                                    // float4 sample groups that hold real rows
    float* xT = sm;                          // [K][SL]   transformed inputs
    float* h1T = xT + K * SL;                // [H1p][SL] tanh(layer 1)  (becomes delta1)
    float* h2T = h1T + H1p * SL;             // [H2p][SL] tanh(layer 2)  (becomes delta2)
    float* dyT = h2T + H2p * SL;             // [A][SL]   mean, then d loss / d (pre-transform output)
    float* gsT = dyT + A * SL;               // [A][SL]   per-sample d loss / d log_std
    float* sl = gsT + A * SL;                // [SB]      per-sample loss
    float* sc = sl + SB;                     // [SB]      1 where the clipped branch zeroed the sample's gradient
    __shared__ AdamC s_c;
    __shared__ float s_ls_sum;
    const int tid = threadIdx.x;
    const int oW1 = 0, ob1 = H1 * K, oW2 = ob1 + H1, ob2 = oW2 + H2 * H1, oW3 = ob2 + H2, ob3 = oW3 + A * H2, oLS = ob3 + A;
    float* w = a.theta; float* mo = a.m; float* vo = a.v;
    float* W1T = a.wT;                       // [K][H1]
    float* W2T = a.wT + K * H1;              // [H1][H2]
    float* W3N = W2T + H1 * H2;              // [A*H2 + A] updated W3, b3 of the current step
    for (int i = tid; i < H1 * K; i += ST) { const int n = i / K, k = i % K; W1T[k * H1 + n] = w[oW1 + i]; }
    for (int i = tid; i < H2 * H1; i += ST) { const int n = i / H1, k = i % H1; W2T[k * H2 + n] = w[oW2 + i]; }
    for (int i = tid; i < (K + H1p + H2p + 2 * A) * SL + 2 * SB; i += ST) sm[i] = 0.0f;
    __syncthreads();

    for (int s = 0; s < (int)a.steps; ++s) {
        if (tid == 0) {
            const double t = (double)(a.step0 + s + 1);
            const double bc1 = 1.0 - pow((double)a.beta1, t), bc2 = 1.0 - pow((double)a.beta2, t);
            s_c.one_m_b1 = (float)(1.0 - (double)a.beta1);
            s_c.b2 = a.beta2;
            s_c.one_m_b2 = (float)(1.0 - (double)a.beta2);
            s_c.bc2_sqrt = (float)sqrt(bc2);
            s_c.eps = a.eps;
            s_c.neg_step = (float)(-((double)a.lr / bc1));
            s_c.reg = 0.0f;
            float t2 = 0.0f;
            for (int j = 0; j < A; ++j) t2 += w[oLS + j];
            s_ls_sum = t2;
        }
        // ---- gather + input transform (fc_network.py:44, same arithmetic as the EVAL tile kernel) ----
        const int* pidx = a.idx + (size_t)s * B;
        for (int f = tid; f < B * K; f += ST) {
            const int b = f / K, k = f - b * K;
            const long long r = pidx[b];
            xT[k * SL + b] = (a.obs[r * K + k] - a.in_shift[k]) / (a.in_scale[k] + 1e-8f);
        }
        __syncthreads();
        // ---- forward (tanh hidden layers, gaussian_mlp.py:104-111) ----
        for (int o = tid; o < H1 * QB; o += ST) {
            const int n = o % H1, q = o / H1;
            *reinterpret_cast<float4*>(h1T + n * SL + 4 * q) = tanh4(sgd_dense(xT, W1T, H1, K, n, q), w[ob1 + n]);
        }
        __syncthreads();
        for (int o = tid; o < H2 * QB; o += ST) {
            const int n = o % H2, q = o / H2;
            *reinterpret_cast<float4*>(h2T + n * SL + 4 * q) = tanh4(sgd_dense(h1T, W2T, H2, H1, n, q), w[ob2 + n]);
        }
        __syncthreads();
        {   // mu[a][4q..] = (h2 . W3[a] + b3[a]) * out_scale + out_shift: 8 lanes split the reduction, xor-shuffle sum
            const int total = 8 * QB * A;
#pragma unroll 1
            for (int u = 0; u < 4; ++u) {
                const int o = tid + u * ST;
                const int seg = o & 7, q = (o >> 3) % QB, aa = (o >> 3) / QB;
                float4 y = make_float4(0.f, 0.f, 0.f, 0.f);
                if (o < total) {
                    const float* w3 = w + oW3 + aa * H2;
                    for (int n = seg; n < H2; n += 8) {
                        const float ww = w3[n];
                        const float4 h = *reinterpret_cast<const float4*>(h2T + n * SL + 4 * q);
                        y.x = fmaf(h.x, ww, y.x); y.y = fmaf(h.y, ww, y.y); y.z = fmaf(h.z, ww, y.z); y.w = fmaf(h.w, ww, y.w);
                    }
                }
#pragma unroll
                for (int x = 4; x > 0; x >>= 1) {
                    y.x += __shfl_xor_sync(0xffffffffu, y.x, x); y.y += __shfl_xor_sync(0xffffffffu, y.y, x);
                    y.z += __shfl_xor_sync(0xffffffffu, y.z, x); y.w += __shfl_xor_sync(0xffffffffu, y.w, x);
                }
                if (o < total && seg == 0) {
                    const float b3 = w[ob3 + aa], os = a.out_scale[aa], oh = a.out_shift[aa];
                    float4 mu;
                    mu.x = (y.x + b3) * os + oh; mu.y = (y.y + b3) * os + oh; mu.z = (y.z + b3) * os + oh; mu.w = (y.w + b3) * os + oh;
                    *reinterpret_cast<float4*>(dyT + aa * SL + 4 * q) = mu;
                }
            }
        }
        __syncthreads();
        // ---- per-sample loss and cotangent d loss / d y (y = output layer before the output transform) ----
        if (tid < SB) {
            const int b = tid;
            if (b < B) {
                const long long r = pidx[b];
                if (KIND == SGD_BC_MSE) {
                    // mean((mu - a)^2) over B x A elements (torch.nn.MSELoss); log_std is not in the graph
                    const float norm = 2.0f / (float)(B * A);
                    float l = 0.0f;
                    for (int j = 0; j < A; ++j) {
                        const float diff = dyT[j * SL + b] - a.act[r * A + j];
                        l = fmaf(diff, diff, l);
                        dyT[j * SL + b] = norm * diff * a.out_scale[j];
                    }
                    sl[b] = l;
                } else {
                    float z2 = 0.0f;
                    for (int j = 0; j < A; ++j) {
                        const float z = (a.act[r * A + j] - dyT[j * SL + b]) / expf(w[oLS + j]);
                        z2 += z * z;
                        dyT[j * SL + b] = z;
                    }
                    const float ll = -0.5f * z2 - s_ls_sum - 0.5f * (float)A * 1.8378770664093453f;
                    float c;                                   // d loss / d LL_b
                    if (KIND == SGD_PPO) {
                        // loss = -mean(min(LR A, clip(LR, 1-e, 1+e) A)); clamp passes the gradient on [lo, hi]
                        // (bounds inclusive), min sends it to the smaller term (a tie splits 1/2 + 1/2 = all of it)
                        const float lr = expf(ll - a.ll_old[r]), adv = a.adv[r];
                        const float lc = fminf(fmaxf(lr, a.clip_lo), a.clip_hi);
                        const float s1 = lr * adv, s2 = lc * adv;
                        const bool live = (lr >= a.clip_lo && lr <= a.clip_hi) || s1 < s2;
                        c = live ? -(lr * adv) / (float)B : 0.0f;
                        sl[b] = -fminf(s1, s2);
                        sc[b] = live ? 0.0f : 1.0f;
                    } else {
                        c = -1.0f / (float)B;                  // loss = -mean(LL)
                        sl[b] = -ll;
                    }
                    for (int j = 0; j < A; ++j) {
                        const float z = dyT[j * SL + b];
                        dyT[j * SL + b] = c * (z / expf(w[oLS + j])) * a.out_scale[j];   // dLL/dmu = z / sigma
                        gsT[j * SL + b] = c * (z * z - 1.0f);                             // dLL/dlog_std = z^2 - 1
                    }
                }
            } else {
                for (int j = 0; j < A; ++j) { dyT[j * SL + b] = 0.0f; gsT[j * SL + b] = 0.0f; }
            }
        }
        __syncthreads();
        const AdamC c = s_c;
        if (tid == 0 && (a.loss_out || a.clip_out)) {
            float l = 0.0f, nc = 0.0f;
            for (int b = 0; b < B; ++b) { l += sl[b]; nc += sc[b]; }
            if (a.loss_out) a.loss_out[s] = l / (float)(KIND == SGD_BC_MSE ? B * A : B);
            if (a.clip_out) a.clip_out[s] = nc / (float)B;
        }
        // ---- output layer: gradients + Adam, new values parked in W3N until delta2 has read the old ones ----
        for (int o = tid; o < A * H2 + A; o += ST) {
            float g = 0.0f;
            int p;
            if (o < A * H2) {
                const int aa = o / H2, n = o - aa * H2;
                for (int b = 0; b < SB; b += 4) {
                    const float4 d = *reinterpret_cast<const float4*>(dyT + aa * SL + b);
                    const float4 h = *reinterpret_cast<const float4*>(h2T + n * SL + b);
                    g = fmaf(d.x, h.x, g); g = fmaf(d.y, h.y, g); g = fmaf(d.z, h.z, g); g = fmaf(d.w, h.w, g);
                }
                p = oW3 + o;
            } else {
                for (int b = 0; b < B; ++b) g += dyT[(o - A * H2) * SL + b];
                p = ob3 + (o - A * H2);
            }
            W3N[o] = adam_step(g, w[p], mo + p, vo + p, c);
        }
        if (KIND != SGD_BC_MSE && tid < A) {               // MSE: log_std has no gradient, torch's Adam skips it
            float g = 0.0f;
            for (int b = 0; b < B; ++b) g += gsT[tid * SL + b];
            w[oLS + tid] = adam_step(g, w[oLS + tid], mo + oLS + tid, vo + oLS + tid, c);
        }
        __syncthreads();                                   // h2 reads done: delta2 overwrites it
        // ---- delta2 = (dy W3) * (1 - h2^2), in place (reads the pre-update W3) ----
        for (int o = tid; o < H2 * QB; o += ST) {
            const int n = o % H2, q = o / H2;
            float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int aa = 0; aa < A; ++aa) {
                const float ww = w[oW3 + aa * H2 + n];
                const float4 y = *reinterpret_cast<const float4*>(dyT + aa * SL + 4 * q);
                d.x = fmaf(y.x, ww, d.x); d.y = fmaf(y.y, ww, d.y); d.z = fmaf(y.z, ww, d.z); d.w = fmaf(y.w, ww, d.w);
            }
            float4 h = *reinterpret_cast<const float4*>(h2T + n * SL + 4 * q);
            h.x = (1.0f - h.x * h.x) * d.x; h.y = (1.0f - h.y * h.y) * d.y;
            h.z = (1.0f - h.z * h.z) * d.z; h.w = (1.0f - h.w * h.w) * d.w;
            *reinterpret_cast<float4*>(h2T + n * SL + 4 * q) = h;
        }
        __syncthreads();                                   // delta2 complete, every read of W3 done
        for (int o = tid; o < A * H2 + A; o += ST) w[o < A * H2 ? oW3 + o : ob3 + (o - A * H2)] = W3N[o];
        // ---- W2 / b2 gradients + Adam: the new W2 goes to W2T only, delta1 below still reads the old W2 ----
        for (int nb = 0; nb < H2; nb += 128)
            for (int kb = 0; kb < H1; kb += 128) {
                float g[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) g[i][j] = 0.0f;
                const int n0 = nb + (tid / 32) * 4, k0 = kb + (tid % 32);
                sgd_wgrad(g, h2T, n0, h1T, k0);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int n = n0 + i, k = k0 + 32 * j;
                        if (n < H2 && k < H1) {
                            const int p = oW2 + n * H1 + k;
                            W2T[k * H2 + n] = adam_step(g[i][j], w[p], mo + p, vo + p, c);
                        }
                    }
            }
        if (tid < H2) {
            float g = 0.0f;
            for (int b = 0; b < B; ++b) g += h2T[tid * SL + b];
            w[ob2 + tid] = adam_step(g, w[ob2 + tid], mo + ob2 + tid, vo + ob2 + tid, c);
        }
        __syncthreads();                                   // wgrad reads of h1 complete
        // ---- delta1 = (delta2 W2_old) * (1 - h1^2), in place ----
        for (int o = tid; o < H1 * QB; o += ST) {
            const int k = o % H1, q = o / H1;
            float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int n = 0; n < H2; ++n) {
                const float ww = w[oW2 + n * H1 + k];
                const float4 e = *reinterpret_cast<const float4*>(h2T + n * SL + 4 * q);
                d.x = fmaf(e.x, ww, d.x); d.y = fmaf(e.y, ww, d.y); d.z = fmaf(e.z, ww, d.z); d.w = fmaf(e.w, ww, d.w);
            }
            const float4 h = *reinterpret_cast<const float4*>(h1T + k * SL + 4 * q);
            d.x *= 1.0f - h.x * h.x; d.y *= 1.0f - h.y * h.y; d.z *= 1.0f - h.z * h.z; d.w *= 1.0f - h.w * h.w;
            *reinterpret_cast<float4*>(h1T + k * SL + 4 * q) = d;
        }
        __syncthreads();                                   // every read of the old W2 done
        for (int o = tid; o < H2 * H1; o += ST) { const int n = o / H1, k = o - n * H1; w[oW2 + o] = W2T[k * H2 + n]; }
        // ---- W1 / b1 gradients + Adam ----
        for (int o = tid; o < H1 * K; o += ST) {
            const int n = o / K, k = o - n * K;
            float g = 0.0f;
            for (int b = 0; b < SB; b += 4) {
                const float4 d = *reinterpret_cast<const float4*>(h1T + n * SL + b);
                const float4 x = *reinterpret_cast<const float4*>(xT + k * SL + b);
                g = fmaf(d.x, x.x, g); g = fmaf(d.y, x.y, g); g = fmaf(d.z, x.z, g); g = fmaf(d.w, x.w, g);
            }
            const int p = oW1 + o;
            const float wn = adam_step(g, w[p], mo + p, vo + p, c);
            w[p] = wn;
            W1T[k * H1 + n] = wn;
        }
        if (tid < H1) {
            float g = 0.0f;
            for (int b = 0; b < B; ++b) g += h1T[tid * SL + b];
            w[ob1 + tid] = adam_step(g, w[ob1 + tid], mo + ob1 + tid, vo + ob1 + tid, c);
        }
        __syncthreads();
    }
}

size_t policy_sgd_smem_bytes(int K0, int h1, int h2, int A) {
    return ((size_t)(K0 + round_up(h1, 128) + round_up(h2, 128) + 2 * A) * SL + 2 * SB) * sizeof(float);
}

size_t policy_sgd_scratch_floats(int K0, int h1, int h2, int A) { return (size_t)K0 * h1 + (size_t)h1 * h2 + (size_t)A * (h2 + 1); }

cudaError_t launch_policy_sgd(const PolicySgdArgs& a, cudaStream_t s) {
    if (a.batch < 1 || a.batch > SB || a.h1 < 1 || a.h1 > 256 || a.h2 < 1 || a.h2 > 256 || a.A < 1 || a.A > 32)
        return cudaErrorInvalidValue;
    const size_t smem = policy_sgd_smem_bytes(a.K0, a.h1, a.h2, a.A);
    if (smem > policy_sgd_max_smem()) return cudaErrorInvalidValue;
    auto run = [&](auto kern) -> cudaError_t {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        kern<<<1, ST, smem, s>>>(a);
        return cudaGetLastError();
    };
    switch (a.loss_kind) {
        case SGD_PPO: return run(policy_sgd_kernel<SGD_PPO>);
        case SGD_BC_MLE: return run(policy_sgd_kernel<SGD_BC_MLE>);
        case SGD_BC_MSE: return run(policy_sgd_kernel<SGD_BC_MSE>);
    }
    return cudaErrorInvalidValue;
}

// ---- full-batch BC loss (behavior_cloning.py:83-105 with idx = all rows): a fixed-grid, fixed-order reduction of the
// per-row log-likelihoods / means that the EVAL tile kernel wrote
constexpr int kLossGrid = 128;

__global__ void __launch_bounds__(256) bc_loss_partial(const float* __restrict__ ll, const float* __restrict__ mu,
                                                       const float* __restrict__ act, long long n, int A, int kind,
                                                       double* partial) {
    __shared__ double red[32];
    double t = 0.0;
    if (kind == SGD_BC_MLE) {
        for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += 256LL * gridDim.x) t += (double)ll[i];
    } else {
        for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n * A; i += 256LL * gridDim.x) {
            const float d = mu[i] - act[i];
            t += (double)(d * d);
        }
    }
    t = block_sum(t, red);
    if (threadIdx.x == 0) partial[blockIdx.x] = t;
}

__global__ void bc_loss_final(const double* partial, int grid, double* out) {
    __shared__ double red[32];
    double t = 0.0;
    for (int i = threadIdx.x; i < grid; i += blockDim.x) t += partial[i];
    t = block_sum(t, red);
    if (threadIdx.x == 0) *out = t;
}

cudaError_t launch_bc_loss_sum(const float* ll, const float* mu, const float* act, long long n, int A, int kind,
                               double* scratch, double* out, cudaStream_t s) {
    bc_loss_partial<<<kLossGrid, 256, 0, s>>>(ll, mu, act, n, A, kind, scratch);
    bc_loss_final<<<1, 128, 0, s>>>(scratch, kLossGrid, out);
    return cudaGetLastError();
}

}  // namespace mjb
