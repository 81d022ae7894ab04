// MLPBaseline.fit (baselines/mlp_baseline.py:61-95 + utils/optimize_model.py:7-36): epochs x (N/bs - 1)
// *sequential* minibatch-Adam steps on mean((V(phi) - R)^2), L2 weight decay folded into the gradient
// (torch.optim.Adam(weight_decay=reg_coef)), Adam state persisting across calls.
//
// The chain is strictly sequential (step k+1 reads the weights step k wrote), so it cannot be sharded
// over samples without changing the reference's semantics; it is latency-bound, not a throughput
// roofline (SURVEY 8d).  This kernel runs the whole epoch as ONE persistent CTA: per step it gathers the
// 64 rows named by the host-drawn permutation, builds the features on the fly, runs forward / backward
// with feature-major activations in shared memory, and each thread Adam-updates the parameters whose
// gradient it just accumulated in registers.  Weights live in global memory (L1/L2-resident, 78 KB) in
// both natural and transposed form so every inner loop reads them coalesced.
#include "adam.cuh"
#include "kernels.h"

namespace mjb {

constexpr int VB = 64;             // max minibatch rows
constexpr int VL = VB + 4;         // row pitch of feature-major activations
constexpr int VT = 1024;           // threads

// out4[n][4 samples q] = sum_k inT[k][4q..] * WT[k][n]   for unit o = n + NOUT*q
__device__ __forceinline__ float4 dense_unit(const float* __restrict__ inT, const float* WT, int NOUT, int R, int n, int q) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int k = 0; k < R; ++k) {
        const float w = WT[k * NOUT + n];
        const float4 x = *reinterpret_cast<const float4*>(inT + k * VL + 4 * q);
        acc.x = fmaf(x.x, w, acc.x); acc.y = fmaf(x.y, w, acc.y); acc.z = fmaf(x.z, w, acc.z); acc.w = fmaf(x.w, w, acc.w);
    }
    return acc;
}

__global__ void __launch_bounds__(VT, 1) vf_fit_kernel(const VfFitArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int K = a.K, H1 = a.H1, H2 = a.H2, B = a.batch;
    const int H1p = round_up(H1, 128), H2p = round_up(H2, 128);   // rows padded so 128-wide wgrad blocks stay in bounds
    float* xT = sm;                          // [K][VL]
    float* h1T = xT + K * VL;                // [H1p][VL]  (becomes delta1)
    float* h2T = h1T + H1p * VL;             // [H2p][VL]  (becomes delta2)
    float* yv = h2T + H2p * VL;              // [VB] prediction
    float* tv = yv + VB;                     // [VB] target
    float* dy = tv + VB;                     // [VB]
    __shared__ AdamC s_c;
    const int tid = threadIdx.x;
    const int oW1 = 0, ob1 = H1 * K, oW2 = ob1 + H1, ob2 = oW2 + H2 * H1, oW3 = ob2 + H2, ob3 = oW3 + H2;
    float* w = a.w; float* mo = a.m; float* vo = a.v;
    float* W1T = a.wT;                       // [K][H1]
    float* W2T = a.wT + K * H1;              // [H1][H2]
    // build the transposed copies once
    for (int i = tid; i < H1 * K; i += VT) { const int n = i / K, k = i % K; W1T[k * H1 + n] = w[oW1 + i]; }
    for (int i = tid; i < H2 * H1; i += VT) { const int n = i / H1, k = i % H1; W2T[k * H2 + n] = w[oW2 + i]; }
    for (int i = tid; i < (K + H1p + H2p) * VL + 3 * VB; i += VT) sm[i] = 0.0f;
    __syncthreads();

    for (int s = 0; s < a.steps; ++s) {
        if (tid == 0) {
            const double t = (double)(a.step0 + s + 1);
            const double bc1 = 1.0 - pow((double)a.beta1, t), bc2 = 1.0 - pow((double)a.beta2, t);
            s_c.one_m_b1 = (float)(1.0 - (double)a.beta1);
            s_c.b2 = a.beta2;
            s_c.one_m_b2 = (float)(1.0 - (double)a.beta2);
            s_c.bc2_sqrt = (float)sqrt(bc2);
            s_c.eps = a.eps;
            s_c.neg_step = (float)(-((double)a.lr / bc1));
            s_c.reg = a.reg;
        }
        // ---- gather the minibatch: features (mlp_baseline.py:36-58) and targets ----
        const int* pidx = a.perm + (size_t)s * B;
        for (int f = tid; f < B * K; f += VT) {
            const int b = f / K, k = f - b * K;
            const long long r = pidx[b];
            float val;
            if (k < a.obs_dim) {
                double x = (double)a.obs[r * a.obs_dim + k];
                x = fmin(fmax(x, -10.0), 10.0) / 10.0;
                val = (float)x;
            } else {
                const double tau = (double)a.tstep[r] / 1000.0;
                double p = tau;
                for (int q = a.obs_dim; q < k; ++q) p *= tau;
                val = (float)p;
            }
            xT[k * VL + b] = val;
        }
        if (tid < B) tv[tid] = (float)a.returns[pidx[tid]];
        __syncthreads();
        // ---- forward ----
        for (int o = tid; o < H1 * 16; o += VT) {
            const int n = o % H1, q = o / H1;
            float4 z = dense_unit(xT, W1T, H1, K, n, q);
            const float bb = w[ob1 + n];
            z.x = fmaxf(z.x + bb, 0.f); z.y = fmaxf(z.y + bb, 0.f); z.z = fmaxf(z.z + bb, 0.f); z.w = fmaxf(z.w + bb, 0.f);
            *reinterpret_cast<float4*>(h1T + n * VL + 4 * q) = z;
        }
        __syncthreads();
        for (int o = tid; o < H2 * 16; o += VT) {
            const int n = o % H2, q = o / H2;
            float4 z = dense_unit(h1T, W2T, H2, H1, n, q);
            const float bb = w[ob2 + n];
            z.x = fmaxf(z.x + bb, 0.f); z.y = fmaxf(z.y + bb, 0.f); z.z = fmaxf(z.z + bb, 0.f); z.w = fmaxf(z.w + bb, 0.f);
            *reinterpret_cast<float4*>(h2T + n * VL + 4 * q) = z;
        }
        __syncthreads();
        {   // y[b] = sum_n h2[n][b] W3[n] + b3 : 16 lanes per sample pair-reduce via shuffles
            const int b = tid / 16, l = tid % 16;
            float t = 0.0f;
            if (b < B) for (int n = l; n < H2; n += 16) t = fmaf(h2T[n * VL + b], w[oW3 + n], t);
            t += __shfl_xor_sync(0xffffffffu, t, 8); t += __shfl_xor_sync(0xffffffffu, t, 4);
            t += __shfl_xor_sync(0xffffffffu, t, 2); t += __shfl_xor_sync(0xffffffffu, t, 1);
            if (b < B && l == 0) {
                const float y = t + w[ob3];
                yv[b] = y;
                dy[b] = 2.0f * (y - tv[b]) / (float)B;   // d mean((y-t)^2) / dy
            }
        }
        __syncthreads();
        const AdamC c = s_c;
        if (a.loss_out && tid == 0) {
            float l = 0.0f;
            for (int b = 0; b < B; ++b) l += (yv[b] - tv[b]) * (yv[b] - tv[b]);
            a.loss_out[s] = l / (float)B;
        }
        // ---- last layer grads + delta2 (in place over h2) ----
        // each thread owns n (W3[n]) for n < H2; thread H2 owns b3
        float gw3 = 0.0f;
        if (tid < H2) {
            for (int b = 0; b < B; ++b) gw3 = fmaf(dy[b], h2T[tid * VL + b], gw3);
        } else if (tid == H2) {
            for (int b = 0; b < B; ++b) gw3 += dy[b];
        }
        __syncthreads();
        for (int o = tid; o < H2 * 16; o += VT) {
            const int n = o % H2, q = o / H2;
            const float w3 = w[oW3 + n];
            float4 h = *reinterpret_cast<const float4*>(h2T + n * VL + 4 * q);
            const float4 d = *reinterpret_cast<const float4*>(dy + 4 * q);
            h.x = h.x > 0.f ? d.x * w3 : 0.f; h.y = h.y > 0.f ? d.y * w3 : 0.f;
            h.z = h.z > 0.f ? d.z * w3 : 0.f; h.w = h.w > 0.f ? d.w * w3 : 0.f;
            *reinterpret_cast<float4*>(h2T + n * VL + 4 * q) = h;
        }
        __syncthreads();
        if (tid < H2) w[oW3 + tid] = adam_step(gw3, w[oW3 + tid], mo + oW3 + tid, vo + oW3 + tid, c);
        else if (tid == H2) w[ob3] = adam_step(gw3, w[ob3], mo + ob3, vo + ob3, c);
        // ---- delta h1 = delta2 W2 (needs the *pre-update* W2): keep in registers until W2 grads are done ----
        float4 dh[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int o = tid + u * VT;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            if (o < H1 * 16) {
                const int k = o % H1, q = o / H1;
#pragma unroll 4
                for (int n = 0; n < H2; ++n) {
                    const float ww = w[oW2 + n * H1 + k];
                    const float4 d = *reinterpret_cast<const float4*>(h2T + n * VL + 4 * q);
                    acc.x = fmaf(d.x, ww, acc.x); acc.y = fmaf(d.y, ww, acc.y); acc.z = fmaf(d.z, ww, acc.z); acc.w = fmaf(d.w, ww, acc.w);
                }
            }
            dh[u] = acc;
        }
        __syncthreads();                                   // all reads of W2 done before anyone updates it
        // ---- W2 / b2 grads + Adam ----
        for (int nb = 0; nb < H2; nb += 128)
            for (int kb = 0; kb < H1; kb += 128) {
                float g[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) g[i][j] = 0.0f;
                const int n0 = nb + (tid / 32) * 4, k0 = kb + (tid % 32);
                wgrad_acc<VB, 4, 4>(g, h2T, n0, 1, h1T, k0, 32);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int n = n0 + i, k = k0 + 32 * j;
                        if (n < H2 && k < H1) {
                            const int p = oW2 + n * H1 + k;
                            const float wn = adam_step(g[i][j], w[p], mo + p, vo + p, c);
                            w[p] = wn;
                            W2T[k * H2 + n] = wn;
                        }
                    }
            }
        if (tid < H2) {
            float g = 0.0f;
            for (int b = 0; b < B; ++b) g += h2T[tid * VL + b];
            w[ob2 + tid] = adam_step(g, w[ob2 + tid], mo + ob2 + tid, vo + ob2 + tid, c);
        }
        __syncthreads();                                   // wgrad reads of h1 complete
        // ---- delta1 = dh * relu'(h1) in place ----
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int o = tid + u * VT;
            if (o < H1 * 16) {
                const int k = o % H1, q = o / H1;
                const float4 h = *reinterpret_cast<const float4*>(h1T + k * VL + 4 * q);
                float4 d = dh[u];
                d.x = h.x > 0.f ? d.x : 0.f; d.y = h.y > 0.f ? d.y : 0.f; d.z = h.z > 0.f ? d.z : 0.f; d.w = h.w > 0.f ? d.w : 0.f;
                *reinterpret_cast<float4*>(h1T + k * VL + 4 * q) = d;
            }
        }
        __syncthreads();
        // ---- W1 / b1 grads + Adam ----
        for (int o = tid; o < H1 * K; o += VT) {
            const int n = o / K, k = o - n * K;
            float g = 0.0f;
            for (int b = 0; b < VB; b += 4) {
                const float4 d = *reinterpret_cast<const float4*>(h1T + n * VL + b);
                const float4 x = *reinterpret_cast<const float4*>(xT + k * VL + b);
                g = fmaf(d.x, x.x, g); g = fmaf(d.y, x.y, g); g = fmaf(d.z, x.z, g); g = fmaf(d.w, x.w, g);
            }
            const int p = oW1 + o;
            const float wn = adam_step(g, w[p], mo + p, vo + p, c);
            w[p] = wn;
            W1T[k * H1 + n] = wn;
        }
        if (tid < H1) {
            float g = 0.0f;
            for (int b = 0; b < B; ++b) g += h1T[tid * VL + b];
            w[ob1 + tid] = adam_step(g, w[ob1 + tid], mo + ob1 + tid, vo + ob1 + tid, c);
        }
        __syncthreads();
    }
}

cudaError_t launch_vf_fit(const VfFitArgs& a, cudaStream_t s) {
    if (a.batch > VB || a.batch < 1 || (a.batch % 4) != 0) return cudaErrorInvalidValue;
    if (a.H1 > 256 || a.H2 > 256 || a.H1 % 4 || a.H2 % 4) return cudaErrorInvalidValue;
    const size_t smem = ((size_t)(a.K + round_up(a.H1, 128) + round_up(a.H2, 128)) * VL + 3 * VB) * sizeof(float);
    if (smem > 220 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(vf_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    vf_fit_kernel<<<1, VT, smem, s>>>(a);
    return cudaGetLastError();
}

}  // namespace mjb
