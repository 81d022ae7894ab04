// MLPBaseline.fit on ONE SM with tcgen05 tensor cores (baselines/mlp_baseline.py:61-95, utils/optimize_model.py:7-36).
//
// The minibatch-Adam chain is sequential, so the step time is latency.  Splitting the hidden units over a thread-block
// cluster costs three distributed-shared-memory hand-offs per step (measured slower in round 1); this kernel keeps the
// whole (obs+4) -> 128 -> 128 -> 1 network, its gradients and its optimizer state on one SM and runs the five GEMMs of a
// step as tcgen05.mma with the HIDDEN UNITS on the M axis (M = 128 is the full-rate shape; the 64-row minibatch is N):
//
//   z1^T  [u][n] = W1 [u][k]  x   [n][k]        A = W1  (K-major)   B = X    (K-major)
//   z2^T  [o][n] = W2 [o][i]  h1^T[i][n]        A = W2  (K-major)   B = h1^T (MN-major)
//   dh1^T [i][n] = W2 [o][i]  dz2^T[o][n]       A = W2  (MN-major)  B = dz2^T(MN-major)   -- the same W2 buffer
//   gW2   [o][i] = dz2^T[o][n] h1^T[i][n]       A = dz2^T (K-major) B = h1^T (K-major)    -- the same h1^T buffer
//   gW1   [u][k] = dz1^T[u][n] x   [n][k]       A = dz1^T (K-major) B = X    (MN-major)   -- the same X buffer
//
// All operands are two-term fp16 splits (hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM), written by the epilogue
// threads in the no-swizzle core-tiled layout of tc_common.cuh: thread (unit u, column quarter) owns a TMEM lane, so
// it writes whole 16-byte core-matrix rows and nothing is ever transposed.
// The B operand's two terms are N-concatenated ([B hi | B lo] are adjacent column groups), so a product costs two
// MMAs per k-step; small operands carry power-of-two scales (SW, SA, SG below) that keep their fp16 low terms normal.
// State: W2's fp32 master copy lives in registers (32 per thread), its Adam moments in TMEM (2 x 128 columns), W1's
// state and the small vectors in shared memory.  512 threads; one elected lane of a converged warp 0 issues the MMAs;
// gW2 is issued before dh1 so that half of W2's Adam update runs under the dh1 GEMM.
// Semantics (minibatch order, 1/B scaling, L2-in-gradient weight decay, bias correction, state persistence) are the
// reference's; sums run in a fixed order (deterministic).
#include <cuda_fp16.h>

#include "kernels.h"
#include "tc_common.cuh"

namespace mjb {

using namespace tc;

namespace {

constexpr int H = 128, NB = 64, KP = 32, NT = 512;
// Power-of-two operand scales (exact to apply and to undo): they keep the fp16 LOW terms out of the subnormal range,
// where a two-term split would lose its 22 significant bits (weights ~0.1 -> lo ~5e-5; gradients ~1e-4 -> lo ~5e-8).
constexpr float SW = 64.0f;                // weights W1, W2
constexpr float SA = 16.0f;                // activations: features x, hidden h1
constexpr float SG = 1024.0f;              // back-propagated deltas dz2, dz1
constexpr int LB128 = 16 * 128;            // column-group stride of buffers with 128 rows
constexpr int LB64 = 16 * 64;              // ... with 64 rows (X)
constexpr int W2_BYTES = H * H * 2, W1_BYTES = H * KP * 2, X_BYTES = NB * KP * 2, HT_BYTES = H * NB * 2;

// shared memory map (bytes)
constexpr int S_W2H = 0, S_W2L = S_W2H + W2_BYTES, S_W1H = S_W2L + W2_BYTES, S_W1L = S_W1H + W1_BYTES;
constexpr int S_XH = S_W1L + W1_BYTES, S_XL = S_XH + X_BYTES, S_HH = S_XL + X_BYTES, S_HL = S_HH + HT_BYTES;
constexpr int S_DH = S_HL + HT_BYTES, S_DL = S_DH + HT_BYTES;
constexpr int S_F32 = S_DL + HT_BYTES;
// fp32 area (floats)
constexpr int F_W1W = 0, F_W1M = F_W1W + KP * H, F_W1V = F_W1M + KP * H;       // W1 state, [k][u]
constexpr int F_VEC = F_W1V + KP * H;                                          // b1,b2,w3: (w,m,v)[128] each -> 9 x 128
constexpr int F_B3 = F_VEC + 9 * H;                                            // b3 w,m,v (+pad)
constexpr int F_YP = F_B3 + 4;                                                 // ypart[4][64]
constexpr int F_GW3 = F_YP + 4 * NB, F_GB2 = F_GW3 + 4 * H, F_GB1 = F_GB2 + 4 * H, F_GB3 = F_GB1 + 4 * H;
constexpr int F_T = F_GB3 + 4;                                                 // targets t[2][64] (double-buffered with X)
constexpr int F_END = F_T + 2 * NB;
constexpr int S_X2 = S_F32 + F_END * 4;                                        // second minibatch buffer [X hi | X lo]
constexpr int S_BAR = S_X2 + 2 * X_BYTES;
constexpr int S_TOTAL = S_BAR + 32;

// TMEM columns.  D holds [X*hi | X*lo] halves of the N-concatenated products; gW1 reuses its columns (D is dead by then)
constexpr uint32_t T_D = 0, T_G1 = 0, T_G2 = 128, T_M = 256, T_V = 384, T_COLS = 512;

struct TcFitArgs {
    int K, KF, steps;                        // KF: row pitch of feat (K rounded up to 8, zero-filled)
    const float* feat; const float* ret32; const int* perm;
    float reg, beta1, beta2, eps;
    float* w; float* m; float* v;
    const float4* consts;                    // per-step {1/sqrt(1-b2^t), -lr/(1-b1^t), sqrt(1-b2^t), -eps*sqrt(1-b2^t)}
    long long* prof;
    // ---- K-split layer 1 (input features beyond KP): helper CTAs of the same cluster, hand-offs through L2 ----
    int nh;                                  // helper CTAs (0 = everything on the head CTA)
    float* zpart;                            // [2][nh][128 units][64 samples] fp32: layer-1 partial sums (scaled SW*SA)
    unsigned char* dzop;                     // [2][dz1 hi 16 KB | dz1 lo 16 KB]: the head's dz1^T operand, core-tiled
    int* flags;                              // [0] head: dz1 of step s published = s+1 ; [1+h] helper h: partial of step s = s+1
};

// ---- hand-off flags in global memory (release / acquire at gpu scope) ----
__device__ __forceinline__ void flag_release(int* f, int v) {   // (st.release carries the one gpu-scope fence; cumulative over
    asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(f), "r"(v) : "memory");   //  the CTA barrier before it)
}
// spins until *f >= target; a partner that never arrives is a bug, so the wait is bounded (~2 s) and then traps
__device__ __forceinline__ void flag_wait_ge(const int* f, int target) {
    const long long t0 = clock64();
    int v;
    for (;;) {
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(f) : "memory");
        if (v >= target) return;
        if (clock64() - t0 > 4000000000ll) __trap();
    }
}

struct AdamP { float one_m_b1, b2, one_m_b2, rbc2_sqrt, eps, neg_step, reg; };

// torch.optim.Adam update.  One SM updates all 20 k parameters every step, so the square root and the division use
// the MUFU approximations (<= 2 ulp each, the same order as the two-term fp16 rounding of the GEMM operands).  The update
// is MUFU-bound (16 results / clock / SM: ~1000 cycles per half of W2); a one-MUFU variant (rsqrt + series for the eps
// term, exact fallback under a branch) was measured SLOWER -- 2400 cycles per half -- because the branch keeps ptxas
// from interleaving the eight independent parameter pairs of a chunk.
__device__ __forceinline__ float adam_apply(float g, float w, float& m, float& v, const AdamP& c) {
    g = fmaf(c.reg, w, g);
    m = fmaf(c.one_m_b1, g - m, m);
    v = fmaf(c.one_m_b2 * g, g, v * c.b2);
    float sq, rc;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(v));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(fmaf(sq, c.rbc2_sqrt, c.eps)));
    return fmaf(c.neg_step, m * rc, w);
}

// ---- packed fp32x2 arithmetic (sm_100 FFMA2 / FMUL2 / FADD2): two IEEE-rounded lanes per instruction, bit-identical to
//      the scalar forms; halves the issue slots of the element-wise Adam update ----
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk2(f32x2 r, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(r)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { f32x2 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

struct AdamP2 { f32x2 one_m_b1, b2, one_m_b2, rbc2_sqrt, eps, neg_step, reg, gscale; };

// two parameters at once; same operation sequence as adam_apply (so the results are bit-identical)
__device__ __forceinline__ void adam_apply2(float g0, float g1, float& w0, float& w1, float& m0, float& m1, float& v0, float& v1,
                                            const AdamP2& c) {
    const f32x2 w = pk2(w0, w1);
    f32x2 m = pk2(m0, m1), v = pk2(v0, v1);
    f32x2 g = mul2(pk2(g0, g1), c.gscale);
    g = fma2(c.reg, w, g);
    m = fma2(c.one_m_b1, sub2(g, m), m);
    v = fma2(mul2(c.one_m_b2, g), g, mul2(v, c.b2));
    upk2(v, v0, v1);
    float s0, s1, r0, r1;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s0) : "f"(v0));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s1) : "f"(v1));
    float d0, d1;
    upk2(fma2(pk2(s0, s1), c.rbc2_sqrt, c.eps), d0, d1);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(d0));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(d1));
    upk2(fma2(c.neg_step, mul2(m, pk2(r0, r1)), w), w0, w1);
    upk2(m, m0, m1);
}

// 8 consecutive fp32 values -> fp16 hi / lo, one 16-byte core-matrix row each
__device__ __forceinline__ void split8_store(const float (&x)[8], unsigned char* hi, unsigned char* lo) {
    __half2 h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        h[j] = __floats2half2_rn(x[2 * j], x[2 * j + 1]);
        const float2 b = __half22float2(h[j]);
        l[j] = __floats2half2_rn(x[2 * j] - b.x, x[2 * j + 1] - b.y);
    }
    *reinterpret_cast<uint4*>(hi) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint4*>(lo) = *reinterpret_cast<const uint4*>(l);
}

// D (+)= A B^T over KS 16-element reduction steps with two-term operands (hi*hi + lo*hi + hi*lo).  Descriptors are built
// once and advanced by one add per step (tc_common.cuh: desc_adv); the loop is fully unrolled.
template <int KS>
__device__ __forceinline__ void gemm3(uint32_t d, uint32_t ah, uint32_t al, uint32_t a_step, uint32_t a_lbo, uint32_t a_sbo,
                                      uint32_t bh, uint32_t bl, uint32_t b_step, uint32_t b_lbo, uint32_t b_sbo, uint32_t idesc) {
    uint64_t dah = make_desc(ah, a_lbo, a_sbo), dal = make_desc(al, a_lbo, a_sbo);
    uint64_t dbh = make_desc(bh, b_lbo, b_sbo), dbl = make_desc(bl, b_lbo, b_sbo);
    // NOT unrolled: only one thread runs this and the tensor queue paces it, while every unrolled MMA costs ~10
    // instructions of a loop body that has to stay inside the 32 KB instruction cache (see the note at the kernel)
#pragma unroll 1
    for (int j = 0; j < KS; ++j) {
        mma_f16(d, dah, dbh, idesc, j > 0);
        mma_f16(d, dal, dbh, idesc, true);
        mma_f16(d, dah, dbl, idesc, true);
        dah = desc_adv(dah, a_step); dal = desc_adv(dal, a_step);
        dbh = desc_adv(dbh, b_step); dbl = desc_adv(dbl, b_step);
    }
}

// Same product with the B terms N-concatenated: the buffer pair [B hi | B lo] is contiguous along N, so
//   D[:, 0:n] (+)= A_hi B_hi + A_lo B_hi   and   D[:, n:2n] (+)= A_hi B_lo     -- two MMAs per step instead of three;
// the epilogue adds the two column halves.
template <int KS>
__device__ __forceinline__ void gemm2c(uint32_t d, uint32_t ah, uint32_t al, uint32_t a_step, uint32_t a_lbo, uint32_t a_sbo,
                                       uint32_t bh, uint32_t b_step, uint32_t b_lbo, uint32_t b_sbo,
                                       uint32_t idesc_2n, uint32_t idesc_n) {
    uint64_t dah = make_desc(ah, a_lbo, a_sbo), dal = make_desc(al, a_lbo, a_sbo);
    uint64_t dbh = make_desc(bh, b_lbo, b_sbo);
#pragma unroll 1
    for (int j = 0; j < KS; ++j) {
        mma_f16(d, dah, dbh, idesc_2n, j > 0);
        mma_f16(d, dal, dbh, idesc_n, true);
        dah = desc_adv(dah, a_step); dal = desc_adv(dal, a_step);
        dbh = desc_adv(dbh, b_step);
    }
}

// ---- helper CTA of the K-split (cluster rank 1 + h): owns the 64 input features [KP + 64 h, KP + 64 h + 64) of layer 1 -- their
// weights (fp16 hi/lo operand + fp32 master), Adam moments, and its own copy of the minibatch columns.  Per step it sends
// the head the partial pre-activations z1_h = W1_h x_h^T (32 KB fp32 through L2) and, once the head has published dz1
// (its 32 KB fp16 hi/lo operand, fetched with one TMA bulk copy), computes gW1_h = dz1 x_h and updates its slice.
// The slice's fp32 master weights and Adam moments live in registers (16 parameters x 3 per thread).  Partial sums travel in a
// thread-major layout (float4 index (4 cq + j) * 128 + u) so that both sides move 512 contiguous bytes per warp instruction.
// Shared-memory map of a helper (bytes): W1 operand 2 x 16 KB | X 2 parities x (8 + 8) KB | dz1 16 + 16 KB.
constexpr int KH = 64;                                   // features per helper
constexpr int HS_W1H = 0, HS_W1L = HS_W1H + H * KH * 2, HS_X = HS_W1L + H * KH * 2, HS_XB = NB * KH * 2;
constexpr int HS_DZ = HS_X + 4 * HS_XB, HS_BAR = HS_DZ + 2 * HT_BYTES, HS_TOTAL = HS_BAR + 32;
constexpr uint32_t HT_Z = 0, HT_G = 64, HT_COLS = 256;

template <bool PROF>
__device__ __forceinline__ void ks_helper(const TcFitArgs& a, unsigned char* smem, uint32_t* s_tmem, long long* s_prof, int h) {
    long long t_last = PROF ? clock64() : 0;
#define KS_PROF(i) do { if (PROF && threadIdx.x == 0) { const long long _t = clock64(); s_prof[i] += _t - t_last; t_last = _t; } } while (0)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + HS_BAR);      // [0] MMA done, [1] dz1 landed
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, cq = warp >> 2, u = 32 * q + lane;
    const int K = a.K, k0 = KP + KH * h;                              // first feature of this helper
    if (warp == 0) tmem_alloc(s_tmem, HT_COLS);
    if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); }
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = *s_tmem, sbase = smem_u32(smem);
    const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
    const uint32_t rowoff = (uint32_t)((u >> 3) * 128 + (u & 7) * 16);
    // ---- state slice: W1[u][k0 + 16 cq .. + 15] (natural layout W1[u * K + k]); columns beyond K are zero and stay zero ----
    float sw[16], sm[16], sv[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const int k = k0 + 16 * cq + j;
        const bool in = k < K;
        sw[j] = in ? a.w[u * K + k] : 0.0f;
        sm[j] = in ? a.m[u * K + k] : 0.0f;
        sv[j] = in ? a.v[u * K + k] : 0.0f;
    }
    auto store_w1 = [&]() {
#pragma unroll
        for (int g8 = 0; g8 < 2; ++g8) {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = SW * sw[8 * g8 + j];
            const uint32_t o = rowoff + (uint32_t)(2 * cq + g8) * LB128;
            split8_store(x, smem + HS_W1H + o, smem + HS_W1L + o);
        }
    };
    store_w1();
    // ---- minibatch gather: thread -> (row gn, 8 features gk .. gk+7 of this helper's 64) ----
    const int gn = tid >> 3, gk = 8 * (tid & 7);
    const uint32_t xoff = core_offset(gn, gk, NB);
    float xr[8];
    auto load_rows = [&](int idx) {
        if (k0 + gk < a.KF) {                                        // (row pitch KF is a multiple of 8: whole groups, 32-byte aligned)
            const float4* p = reinterpret_cast<const float4*>(a.feat + (size_t)idx * a.KF + k0 + gk);
            const float4 t0 = __ldg(p), t1 = __ldg(p + 1);
            xr[0] = t0.x; xr[1] = t0.y; xr[2] = t0.z; xr[3] = t0.w; xr[4] = t1.x; xr[5] = t1.y; xr[6] = t1.z; xr[7] = t1.w;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) xr[j] = 0.0f;
        }
    };
    auto stage_x = [&](int par) {
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = SA * xr[j];
        unsigned char* xb = smem + HS_X + par * 2 * HS_XB;
        split8_store(x, xb + xoff, xb + HS_XB + xoff);
    };
    int i1 = 0, i2 = 0;
    float4 cst_next = a.consts[0];
    load_rows(a.perm[gn]);
    stage_x(0);
    if (a.steps > 1) i1 = a.perm[NB + gn];
    if (a.steps > 2) i2 = a.perm[2 * NB + gn];
    const uint32_t ID_Z = make_idesc_f16(128, NB, false, false);
    const uint32_t ID_Gc = make_idesc_f16(128, 2 * KH, false, true), ID_G = make_idesc_f16(128, KH, false, true);
    uint32_t p0 = 0, p1 = 0;
    AdamP2 ap;
    ap.one_m_b1 = pk2(1.0f - a.beta1, 1.0f - a.beta1); ap.b2 = pk2(a.beta2, a.beta2);
    ap.one_m_b2 = pk2(1.0f - a.beta2, 1.0f - a.beta2); ap.eps = pk2(a.eps, a.eps); ap.reg = pk2(a.reg, a.reg);
    ap.gscale = pk2(1.0f / (SG * SA), 1.0f / (SG * SA));
    ap.rbc2_sqrt = ap.neg_step = pk2(0.0f, 0.0f);
    for (int s = 0; s < a.steps; ++s) {
        fence_proxy_async(); tcgen05_fence_before(); __syncthreads();       // X(s) staged, slice operand current
        KS_PROF(0);
        const uint32_t xb = sbase + HS_X + (uint32_t)(s & 1) * 2 * HS_XB;
        if (tid == 0) {                                              // z1_h^T = W1_h x_h^T
            tcgen05_fence_after();
            gemm3<KH / 16>(tmem + HT_Z, sbase + HS_W1H, sbase + HS_W1L, 2 * LB128, LB128, 128,
                           xb, xb + HS_XB, 2 * LB64, LB64, 128, ID_Z);
            mma_commit(&bars[0]);
            KS_PROF(11);
        }
        if (s + 1 < a.steps) load_rows(i1);
        i1 = i2;
        if (s + 3 < a.steps) i2 = a.perm[(size_t)(s + 3) * NB + gn];
        const float4 cst = cst_next;
        if (s + 1 < a.steps) cst_next = a.consts[s + 1];
        ap.rbc2_sqrt = pk2(cst.x, cst.x); ap.neg_step = pk2(cst.y, cst.y);
        KS_PROF(1);
        mbar_wait(&bars[0], p0); p0 ^= 1; tcgen05_fence_after();
        KS_PROF(2);
        {                                                            // partial pre-activations -> L2 (fp32, still scaled SW*SA)
            uint32_t z[16];
            tmem_ld16(tlane + HT_Z + 16 * cq, z);
            tmem_ld_wait();
            float4* dst = reinterpret_cast<float4*>(a.zpart + ((size_t)(s & 1) * a.nh + h) * (H * NB)) + (4 * cq) * H + u;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                dst[j * H] = make_float4(__uint_as_float(z[4 * j]), __uint_as_float(z[4 * j + 1]), __uint_as_float(z[4 * j + 2]), __uint_as_float(z[4 * j + 3]));
        }
        tcgen05_fence_before();
        __syncthreads();
        KS_PROF(3);
        if (tid == 0) flag_release(a.flags + 1 + h, s + 1);
        KS_PROF(4);
        if (s + 1 < a.steps) stage_x((s + 1) & 1);
        KS_PROF(5);                   // next minibatch while the head works on this one
        if (tid == 0) {                                              // the head's dz1 operand of this step: one TMA bulk copy
            flag_wait_ge(a.flags, s + 1);
            KS_PROF(6);
            asm volatile("fence.proxy.async.global;\n" ::: "memory");
            mbar_expect_tx(&bars[1], 2 * HT_BYTES);
            bulk_g2s(smem + HS_DZ, a.dzop + (size_t)(s & 1) * 2 * HT_BYTES, 2 * HT_BYTES, &bars[1]);
        }
        mbar_wait(&bars[1], p1); p1 ^= 1;
        fence_proxy_async(); tcgen05_fence_before(); __syncthreads();
        KS_PROF(7);
        if (tid == 0) {                                              // gW1_h = dz1 x_h  ([hi | lo] columns of x concatenated along N)
            tcgen05_fence_after();
            gemm2c<NB / 16>(tmem + HT_G, sbase + HS_DZ, sbase + HS_DZ + HT_BYTES, 2 * LB128, LB128, 128,
                            xb, 2 * 128, 128, LB64, ID_Gc, ID_G);
            mma_commit(&bars[0]);
        }
        KS_PROF(8);
        mbar_wait(&bars[0], p0); p0 ^= 1; tcgen05_fence_after();
        KS_PROF(9);
        {                                                            // Adam on W1[u][k0 + 16 cq ..]
            uint32_t g[16], gl[16];
            tmem_ld16(tlane + HT_G + 16 * cq, g);
            tmem_ld16(tlane + HT_G + KH + 16 * cq, gl);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; j += 2)
                adam_apply2(__uint_as_float(g[j]) + __uint_as_float(gl[j]), __uint_as_float(g[j + 1]) + __uint_as_float(gl[j + 1]),
                            sw[j], sw[j + 1], sm[j], sm[j + 1], sv[j], sv[j + 1], ap);
            store_w1();
        }
        KS_PROF(10);
    }
    __syncthreads();
    if (PROF && a.prof && h == 0 && tid < 16) a.prof[16 + tid] += s_prof[tid];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const int k = k0 + 16 * cq + j;
        if (k < K) { a.w[u * K + k] = sw[j]; a.m[u * K + k] = sm[j]; a.v[u * K + k] = sv[j]; }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, HT_COLS);
}

// one lane of a converged warp: the MMA issuer.  Warp 0 enters the issue block whole and elect.sync picks the lane, so
// the issue loop runs converged instead of in a divergent tid == 0 branch (52 instead of 62 cycles per N = 64 MMA in
// tools/mma_rate_probe.cu)
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(p));
    return p != 0;
}

// PROF = true instantiates the per-phase clock64 counters (tools/vf_fit_profile.py); the production instance carries none
// of that code.  Code size matters here: a single resident CTA runs a ~2.7 k-instruction step body 15 624 times, and a
// body that does not fit the 32 KB instruction cache is re-fetched from L2 every step (the fetch stalls showed up as
// ~1.3 k unexplained cycles per step that moved with whatever code ran "cold").
// KS = true is the cluster form for more than KP input features: CTA 0 is this head, CTAs 1 .. nh run ks_helper.
template <bool PROF, bool KS>
__global__ void __launch_bounds__(NT, 1) vf_fit_tc_kernel(const TcFitArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    float* sf = reinterpret_cast<float*>(smem + S_F32);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S_BAR);
    __shared__ uint32_t s_tmem;
    __shared__ long long s_prof[16];
    if (KS && blockIdx.x > 0) {                                      // helper CTAs of the K-split (cluster ranks 1 ..)
        if (threadIdx.x < 16) s_prof[threadIdx.x] = 0;
        ks_helper<PROF>(a, smem, &s_tmem, s_prof, (int)blockIdx.x - 1);
        return;
    }
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, cq = warp >> 2, u = 32 * q + lane;       // TMEM lane = hidden unit u; column quarter cq
    const int K = a.K;
    // natural (nn.Sequential) offsets
    const int oW1 = 0, ob1 = H * K, oW2 = ob1 + H, ob2 = oW2 + H * H, oW3 = ob2 + H, ob3 = oW3 + H;

    if (warp == 0) tmem_alloc(&s_tmem, T_COLS);
    if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); }
    if (tid < 16) s_prof[tid] = 0;
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem = s_tmem, sbase = smem_u32(smem);
    const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
    const uint32_t rowoff = (uint32_t)((u >> 3) * 128 + (u & 7) * 16);      // core-tiled row offset of unit u (rows = 128)

    // ---- load the state ----
    float w2[32];                                                    // W2[u][32cq .. 32cq+31], fp32 master
    {
        uint32_t mv[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) w2[j] = a.w[oW2 + u * H + 32 * cq + j];
#pragma unroll
        for (int j = 0; j < 32; ++j) mv[j] = __float_as_uint(a.m[oW2 + u * H + 32 * cq + j]);
        tmem_st32(tlane + T_M + 32 * cq, mv);
#pragma unroll
        for (int j = 0; j < 32; ++j) mv[j] = __float_as_uint(a.v[oW2 + u * H + 32 * cq + j]);
        tmem_st32(tlane + T_V + 32 * cq, mv);
        tmem_st_wait();
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = SW * w2[8 * c8 + j];
            const uint32_t o = rowoff + (uint32_t)(4 * cq + c8) * LB128;
            split8_store(x, smem + S_W2H + o, smem + S_W2L + o);
        }
    }
    {                                                                // W1[u][8cq .. 8cq+7] (zero beyond K)
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = 8 * cq + j;
            const bool in = k < K;
            const float wv = in ? a.w[oW1 + u * K + k] : 0.0f;
            x[j] = SW * wv;
            sf[F_W1W + k * H + u] = wv;
            sf[F_W1M + k * H + u] = in ? a.m[oW1 + u * K + k] : 0.0f;
            sf[F_W1V + k * H + u] = in ? a.v[oW1 + u * K + k] : 0.0f;
        }
        const uint32_t o = rowoff + (uint32_t)cq * LB128;
        split8_store(x, smem + S_W1H + o, smem + S_W1L + o);
    }
    if (cq == 0) {                                                   // vectors: b1, b2, w3 (w, m, v)
        const int offs[3] = {ob1, ob2, oW3};
#pragma unroll
        for (int p = 0; p < 3; ++p) {
            sf[F_VEC + (3 * p + 0) * H + u] = a.w[offs[p] + u];
            sf[F_VEC + (3 * p + 1) * H + u] = a.m[offs[p] + u];
            sf[F_VEC + (3 * p + 2) * H + u] = a.v[offs[p] + u];
        }
    }
    if (tid == 0) { sf[F_B3] = a.w[ob3]; sf[F_B3 + 1] = a.m[ob3]; sf[F_B3 + 2] = a.v[ob3]; }

    // ---- minibatch gather pipeline: thread -> (row n, 4 features) ----
    const int gn = tid >> 3, gk = 4 * (tid & 7);
    const uint32_t xoff = core_offset(gn, gk, NB);
    float xr[4] = {0.f, 0.f, 0.f, 0.f};
    float tt = 0.0f;
    auto load_rows = [&](int idx) {
        // feature rows are padded to a multiple of 8 columns (zeros): one aligned 16-byte load per thread
        const float4 t4 = gk < a.KF ? __ldg(reinterpret_cast<const float4*>(a.feat + (size_t)idx * a.KF + gk)) : make_float4(0.f, 0.f, 0.f, 0.f);
        xr[0] = t4.x; xr[1] = t4.y; xr[2] = t4.z; xr[3] = t4.w;
        if (gk == 0) tt = a.ret32[idx];
    };
    // The minibatch operand is double-buffered (step parity): the rows of step s+1 are staged while the gW2 GEMM of step
    // s runs and nobody else has work, instead of on the critical path after the last GEMM of the step.
    auto stage_x = [&](int par) {
        const int xo = par ? S_X2 : S_XH;
        const float s0 = SA * xr[0], s1 = SA * xr[1], s2 = SA * xr[2], s3 = SA * xr[3];
        const __half2 h01 = __floats2half2_rn(s0, s1), h23 = __floats2half2_rn(s2, s3);
        const float2 b01 = __half22float2(h01), b23 = __half22float2(h23);
        const __half2 l01 = __floats2half2_rn(s0 - b01.x, s1 - b01.y), l23 = __floats2half2_rn(s2 - b23.x, s3 - b23.y);
        uint2 hv, lv;
        hv.x = *reinterpret_cast<const uint32_t*>(&h01); hv.y = *reinterpret_cast<const uint32_t*>(&h23);
        lv.x = *reinterpret_cast<const uint32_t*>(&l01); lv.y = *reinterpret_cast<const uint32_t*>(&l23);
        *reinterpret_cast<uint2*>(smem + xo + xoff) = hv;
        *reinterpret_cast<uint2*>(smem + xo + X_BYTES + xoff) = lv;
        if (gk == 0) sf[F_T + par * NB + gn] = tt;
    };
    int i1 = 0, i2 = 0;
    float4 cst_next = a.consts[0];                                   // Adam constants: prefetched one step ahead
    load_rows(a.perm[gn]);
    stage_x(0);
    if (a.steps > 1) i1 = a.perm[NB + gn];
    if (a.steps > 2) i2 = a.perm[2 * NB + gn];

    const uint32_t ID_L1 = make_idesc_f16(128, NB, false, false);
    const uint32_t ID_L2 = make_idesc_f16(128, NB, false, true), ID_L2c = make_idesc_f16(128, 2 * NB, false, true);
    const uint32_t ID_DH = make_idesc_f16(128, NB, true, true), ID_DHc = make_idesc_f16(128, 2 * NB, true, true);
    const uint32_t ID_G2 = make_idesc_f16(128, H, false, false);
    const uint32_t ID_G1 = make_idesc_f16(128, KP, false, true), ID_G1c = make_idesc_f16(128, 2 * KP, false, true);
    uint32_t p0 = 0, p1 = 0;
    auto wait0 = [&]() { mbar_wait(&bars[0], p0); p0 ^= 1; tcgen05_fence_after(); };
    auto wait1 = [&]() { mbar_wait(&bars[1], p1); p1 ^= 1; tcgen05_fence_after(); };
    auto sync_ops = [&]() { fence_proxy_async(); tcgen05_fence_before(); __syncthreads(); };

    long long t_last = clock64();
#define TC_PROF(i) do { if (PROF && tid == 0) { const long long _t = clock64(); s_prof[i] += _t - t_last; t_last = _t; } } while (0)

    AdamP ap;
    ap.one_m_b1 = 1.0f - a.beta1; ap.b2 = a.beta2; ap.one_m_b2 = 1.0f - a.beta2; ap.eps = a.eps; ap.reg = a.reg;
    AdamP2 ap2;
    ap2.one_m_b1 = pk2(ap.one_m_b1, ap.one_m_b1); ap2.b2 = pk2(ap.b2, ap.b2); ap2.one_m_b2 = pk2(ap.one_m_b2, ap.one_m_b2);
    ap2.eps = pk2(ap.eps, ap.eps); ap2.reg = pk2(ap.reg, ap.reg); ap2.gscale = pk2(1.0f / (SG * SA), 1.0f / (SG * SA));
    ap2.rbc2_sqrt = ap2.neg_step = 0;
    ap.rbc2_sqrt = ap.neg_step = 0.0f;

    for (int s = 0; s < a.steps; ++s) {
        sync_ops();                                                  // X(s), weights(s) staged
        TC_PROF(13);                                                 // (barrier skew at the top of the step)
        if (warp == 0) {                                             // layer 1: z1^T = W1 x^T
            tcgen05_fence_after();
            if (elect_one()) {
                const uint32_t xb = sbase + ((s & 1) ? S_X2 : S_XH);
                gemm3<KP / 16>(tmem + T_D, sbase + S_W1H, sbase + S_W1L, 2 * LB128, LB128, 128,
                               xb, xb + X_BYTES, 2 * LB64, LB64, 128, ID_L1);
                mma_commit(&bars[0]);
            }
            __syncwarp();
        }
        TC_PROF(14);                                                 // (issue of the six layer-1 MMAs)
        const float4 cst = cst_next;
        ap.rbc2_sqrt = cst.x; ap.neg_step = cst.y;
        ap2.rbc2_sqrt = pk2(cst.x, cst.x); ap2.neg_step = pk2(cst.y, cst.y);
        TC_PROF(0);
        wait0();
        TC_PROF(1);
        uint32_t mask1 = 0;
        {                                                            // h1 = relu(z1 + b1) -> h1^T operand rows
            uint32_t z[16];
            tmem_ld16(tlane + T_D + 16 * cq, z);
            tmem_ld_wait();
            if (KS) {                                                // + the helpers' partial sums over the features beyond KP
                if (tid == 0) for (int hh = 0; hh < a.nh; ++hh) flag_wait_ge(a.flags + 1 + hh, s + 1);
                __syncthreads();
                TC_PROF(15);                                         // (waiting for the helpers' partial sums)
                // thread-major layout (see ks_helper); helper hh + 1's 64 bytes are in flight while hh's are added
                const float4* src = reinterpret_cast<const float4*>(a.zpart + (size_t)(s & 1) * a.nh * (H * NB)) + (4 * cq) * H + u;
                float4 t[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) t[j] = __ldcg(src + j * H);
                for (int hh = 0; hh < a.nh; ++hh) {                  // fixed order: deterministic
                    float4 nx[4];
                    if (hh + 1 < a.nh) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) nx[j] = __ldcg(src + (size_t)(hh + 1) * (H * NB / 4) + j * H);
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        z[4 * j] = __float_as_uint(__uint_as_float(z[4 * j]) + t[j].x);
                        z[4 * j + 1] = __float_as_uint(__uint_as_float(z[4 * j + 1]) + t[j].y);
                        z[4 * j + 2] = __float_as_uint(__uint_as_float(z[4 * j + 2]) + t[j].z);
                        z[4 * j + 3] = __float_as_uint(__uint_as_float(z[4 * j + 3]) + t[j].w);
                        t[j] = nx[j];
                    }
                }
            }
            const float b = sf[F_VEC + 0 * H + u];
            float x[8];
#pragma unroll
            for (int g = 0; g < 2; ++g) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float zz = fmaf(__uint_as_float(z[8 * g + j]), 1.0f / (SW * SA), b);
                    const bool on = zz > 0.0f;
                    mask1 |= (on ? 1u : 0u) << (8 * g + j);
                    x[j] = on ? SA * zz : 0.0f;
                }
                const uint32_t o = rowoff + (uint32_t)(2 * cq + g) * LB128;
                split8_store(x, smem + S_HH + o, smem + S_HL + o);
            }
        }
        sync_ops();
        TC_PROF(2);
        if (warp == 0) {                                             // layer 2: z2^T = W2 h1
            tcgen05_fence_after();
            if (elect_one()) {
                gemm2c<H / 16>(tmem + T_D, sbase + S_W2H, sbase + S_W2L, 2 * LB128, LB128, 128,
                               sbase + S_HH, 2 * 128, 128, LB128, ID_L2c, ID_L2);
                mma_commit(&bars[0]);
            }
            __syncwarp();
        }
        TC_PROF(3);
        // gathers for the coming steps, issued while the layer-2 GEMM runs and nobody has work: rows of step s+1 (consumed
        // by stage_x in the gW2 shadow below), the permutation entry of step s+3, the Adam constants of step s+1
        if (s + 1 < a.steps) load_rows(i1);
        i1 = i2;
        if (s + 3 < a.steps) i2 = a.perm[(size_t)(s + 3) * NB + gn];
        if (s + 1 < a.steps) cst_next = a.consts[s + 1];
        wait0();
        TC_PROF(4);
        float h2[16];
        uint32_t mask2 = 0;
        const float w3u = sf[F_VEC + 6 * H + u];
        {                                                            // h2 = relu(z2 + b2); partial outputs
            uint32_t z[16], zl[16];
            tmem_ld16(tlane + T_D + 16 * cq, z);
            tmem_ld16(tlane + T_D + NB + 16 * cq, zl);
            tmem_ld_wait();
            const float b = sf[F_VEC + 3 * H + u];
            float p[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float zz = fmaf(__uint_as_float(z[j]) + __uint_as_float(zl[j]), 1.0f / (SW * SA), b);
                const bool on = zz > 0.0f;
                mask2 |= (on ? 1u : 0u) << j;
                h2[j] = on ? zz : 0.0f;
                p[j] = w3u * h2[j];
            }
            // transpose-reduce over the 32 units of this warp: lane ends with the sum for n = 16cq + (lane >> 1)
#pragma unroll
            for (int st = 0; st < 4; ++st) {
                const int half = 8 >> st;                            // values kept after this stage
                const bool up = (lane >> (4 - st)) & 1;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (i < half) {
                        const float send = up ? p[i] : p[i + half];
                        const float keep = up ? p[i + half] : p[i];
                        p[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16 >> st);
                    }
                }
            }
            p[0] += __shfl_xor_sync(0xffffffffu, p[0], 1);
            if ((lane & 1) == 0) sf[F_YP + q * NB + 16 * cq + (lane >> 1)] = p[0];
        }
        // the 16 outputs of this column quarter need the partials of its four warps only: named barrier 1 + cq
        asm volatile("bar.sync %0, 128;\n" ::"r"(1 + cq) : "memory");
        TC_PROF(5);
        {                                                            // dy, small gradients, dz2^T operand rows
            const float b3 = sf[F_B3];
            float gw3 = 0.0f, gb2 = 0.0f, gb3 = 0.0f;
            float x[8];
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                const int n0 = 16 * cq + 8 * g;
                float y[8], tg[8];
#pragma unroll
                for (int h4 = 0; h4 < 2; ++h4) {                     // fixed-order sum of the four quadrant partials
                    const float4 p0 = *reinterpret_cast<const float4*>(sf + F_YP + n0 + 4 * h4);
                    const float4 p1 = *reinterpret_cast<const float4*>(sf + F_YP + NB + n0 + 4 * h4);
                    const float4 p2 = *reinterpret_cast<const float4*>(sf + F_YP + 2 * NB + n0 + 4 * h4);
                    const float4 p3 = *reinterpret_cast<const float4*>(sf + F_YP + 3 * NB + n0 + 4 * h4);
                    const float4 t4 = *reinterpret_cast<const float4*>(sf + F_T + (s & 1) * NB + n0 + 4 * h4);
                    y[4 * h4 + 0] = (((p0.x + p1.x) + p2.x) + p3.x) + b3; y[4 * h4 + 1] = (((p0.y + p1.y) + p2.y) + p3.y) + b3;
                    y[4 * h4 + 2] = (((p0.z + p1.z) + p2.z) + p3.z) + b3; y[4 * h4 + 3] = (((p0.w + p1.w) + p2.w) + p3.w) + b3;
                    tg[4 * h4 + 0] = t4.x; tg[4 * h4 + 1] = t4.y; tg[4 * h4 + 2] = t4.z; tg[4 * h4 + 3] = t4.w;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float dy = (2.0f / (float)NB) * (y[j] - tg[j]);
                    gw3 = fmaf(h2[8 * g + j], dy, gw3);
                    gb3 += dy;
                    const float dz = ((mask2 >> (8 * g + j)) & 1u) ? dy * w3u : 0.0f;
                    gb2 += dz;
                    x[j] = SG * dz;
                }
                const uint32_t o = rowoff + (uint32_t)(2 * cq + g) * LB128;
                split8_store(x, smem + S_DH + o, smem + S_DL + o);
            }
            sf[F_GW3 + cq * H + u] = gw3;
            sf[F_GB2 + cq * H + u] = gb2;
            if (u == 0) sf[F_GB3 + cq] = gb3;
        }
        sync_ops();
        TC_PROF(6);
        if (warp == 0) {                                             // gW2 = dz2 h1^T -> bar 1, then dh1^T = W2^T dz2 -> bar 0
            tcgen05_fence_after();
            if (elect_one()) {
                gemm3<NB / 16>(tmem + T_G2, sbase + S_DH, sbase + S_DL, 2 * LB128, LB128, 128,
                               sbase + S_HH, sbase + S_HL, 2 * LB128, LB128, 128, ID_G2);
                mma_commit(&bars[1]);
                gemm2c<H / 16>(tmem + T_D, sbase + S_W2H, sbase + S_W2L, 2 * 128, 128, LB128,
                               sbase + S_DH, 2 * 128, 128, LB128, ID_DHc, ID_DH);
                mma_commit(&bars[0]);
            }
            __syncwarp();
        }
        TC_PROF(7);
        // ---- nothing depends on these until the next step: they run while the gW2 GEMM has the tensor pipe to itself ----
        if (cq >= 2) {                                               // b2 (cq 2) and w3 (cq 3): gradients are complete after E2b
            const int p = cq - 1;
            const int gsrc = p == 1 ? F_GB2 : F_GW3;
            const float g = ((sf[gsrc + u] + sf[gsrc + H + u]) + sf[gsrc + 2 * H + u]) + sf[gsrc + 3 * H + u];
            float mj = sf[F_VEC + (3 * p + 1) * H + u], vj = sf[F_VEC + (3 * p + 2) * H + u];
            sf[F_VEC + (3 * p + 0) * H + u] = adam_apply(g, sf[F_VEC + (3 * p + 0) * H + u], mj, vj, ap);
            sf[F_VEC + (3 * p + 1) * H + u] = mj; sf[F_VEC + (3 * p + 2) * H + u] = vj;
        }
        if (tid == NT - 1) {
            const float g = ((sf[F_GB3] + sf[F_GB3 + 1]) + sf[F_GB3 + 2]) + sf[F_GB3 + 3];
            float mj = sf[F_B3 + 1], vj = sf[F_B3 + 2];
            sf[F_B3] = adam_apply(g, sf[F_B3], mj, vj, ap);
            sf[F_B3 + 1] = mj; sf[F_B3 + 2] = vj;
        }
        if (s + 1 < a.steps) stage_x((s + 1) & 1);                   // minibatch of step s+1 (rows loaded at the top of this step)
        wait1();                                                     // gW2 done: its Adam half runs under the dh1 GEMM
        auto adam_w2 = [&](int c16) {                                // W2[u][32cq + 16 c16 ..]: moments in TMEM
            uint32_t g[16], mm[16], vv[16];
            tmem_ld16(tlane + T_G2 + 32 * cq + 16 * c16, g);
            tmem_ld16(tlane + T_M + 32 * cq + 16 * c16, mm);
            tmem_ld16(tlane + T_V + 32 * cq + 16 * c16, vv);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
                float m0 = __uint_as_float(mm[j]), m1 = __uint_as_float(mm[j + 1]);
                float v0 = __uint_as_float(vv[j]), v1 = __uint_as_float(vv[j + 1]);
                adam_apply2(__uint_as_float(g[j]), __uint_as_float(g[j + 1]), w2[16 * c16 + j], w2[16 * c16 + j + 1], m0, m1, v0, v1, ap2);
                mm[j] = __float_as_uint(m0); mm[j + 1] = __float_as_uint(m1);
                vv[j] = __float_as_uint(v0); vv[j + 1] = __float_as_uint(v1);
            }
            tmem_st16(tlane + T_M + 32 * cq + 16 * c16, mm);
            tmem_st16(tlane + T_V + 32 * cq + 16 * c16, vv);
        };
        auto store_w2 = [&](int c16) {                               // new operand rows (W2 must not be read by an MMA now)
#pragma unroll
            for (int g8 = 0; g8 < 2; ++g8) {
                float x[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) x[j] = SW * w2[16 * c16 + 8 * g8 + j];
                const uint32_t o = rowoff + (uint32_t)(4 * cq + 2 * c16 + g8) * LB128;
                split8_store(x, smem + S_W2H + o, smem + S_W2L + o);
            }
        };
        adam_w2(0);
        TC_PROF(8);
        wait0();                                                     // dh1 done: D ready, W2 and dz buffers free
        {                                                            // dz1 = relu'(z1) dh1 -> dz1^T operand rows
            uint32_t z[16], zl[16];
            tmem_ld16(tlane + T_D + 16 * cq, z);
            tmem_ld16(tlane + T_D + NB + 16 * cq, zl);
            tmem_ld_wait();
            float x0[8], x1[8];
            float gb1 = 0.0f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                // TMEM holds SW*SG*dh1; the operand keeps the SG scale
                x0[j] = ((mask1 >> j) & 1u) ? (__uint_as_float(z[j]) + __uint_as_float(zl[j])) * (1.0f / SW) : 0.0f;
                x1[j] = ((mask1 >> (8 + j)) & 1u) ? (__uint_as_float(z[8 + j]) + __uint_as_float(zl[8 + j])) * (1.0f / SW) : 0.0f;
                gb1 += x0[j];
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) gb1 += x1[j];
            sf[F_GB1 + cq * H + u] = gb1 * (1.0f / SG);
            const uint32_t o = rowoff + (uint32_t)(2 * cq) * LB128;
            split8_store(x0, smem + S_DH + o, smem + S_DL + o);
            split8_store(x1, smem + S_DH + o + LB128, smem + S_DL + o + LB128);
            if (KS) {                                                // the same operand rows for the helpers, through L2
                unsigned char* gd = a.dzop + (size_t)(s & 1) * 2 * HT_BYTES;
                split8_store(x0, gd + o, gd + HT_BYTES + o);
                split8_store(x1, gd + o + LB128, gd + HT_BYTES + o + LB128);
                asm volatile("fence.proxy.async.global;\n" ::: "memory");     // read next by a helper's TMA (async proxy)
            }
        }
        sync_ops();
        TC_PROF(9);
        if (KS && tid == 0) flag_release(a.flags, s + 1);            // every thread's dz1 rows are written (barrier above)
        if (warp == 0) {                                             // gW1 = dz1 x -> bar 0, under the second Adam half of W2
            tcgen05_fence_after();
            if (elect_one()) {
                gemm2c<NB / 16>(tmem + T_G1, sbase + S_DH, sbase + S_DL, 2 * LB128, LB128, 128,
                                sbase + ((s & 1) ? S_X2 : S_XH), 2 * 128, 128, LB64, ID_G1c, ID_G1);
                mma_commit(&bars[0]);
            }
            __syncwarp();
        }
        store_w2(0);
        adam_w2(1);
        store_w2(1);
        if (cq == 1) {                                               // b1 (its gradient is complete after E3); fixed-order sum
            const float g = ((sf[F_GB1 + u] + sf[F_GB1 + H + u]) + sf[F_GB1 + 2 * H + u]) + sf[F_GB1 + 3 * H + u];
            float mj = sf[F_VEC + 1 * H + u], vj = sf[F_VEC + 2 * H + u];
            sf[F_VEC + u] = adam_apply(g, sf[F_VEC + u], mj, vj, ap);
            sf[F_VEC + 1 * H + u] = mj; sf[F_VEC + 2 * H + u] = vj;
        }
        TC_PROF(10);
        wait0();                                                     // gW1 done (X and dz buffers free)
        TC_PROF(11);
        {                                                            // W1[u][8cq ..]: state in shared memory ([k][u])
            uint32_t g[8], gl[8];
            tmem_ld8(tlane + T_G1 + 8 * cq, g);
            tmem_ld8(tlane + T_G1 + KP + 8 * cq, gl);
            tmem_ld_wait();
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = 8 * cq + j;
                float mj = sf[F_W1M + k * H + u], vj = sf[F_W1V + k * H + u];
                const float wn = adam_apply((__uint_as_float(g[j]) + __uint_as_float(gl[j])) * (1.0f / (SG * SA)),
                                            sf[F_W1W + k * H + u], mj, vj, ap);
                sf[F_W1W + k * H + u] = wn; sf[F_W1M + k * H + u] = mj; sf[F_W1V + k * H + u] = vj;
                x[j] = SW * wn;
            }
            const uint32_t o = rowoff + (uint32_t)cq * LB128;
            split8_store(x, smem + S_W1H + o, smem + S_W1L + o);
        }
        tmem_st_wait();
        TC_PROF(12);
    }
    __syncthreads();
    if (PROF && a.prof && tid < 16) a.prof[tid] += s_prof[tid];

    // ---- write the state back (natural layout) ----
    {
        uint32_t mv[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) a.w[oW2 + u * H + 32 * cq + j] = w2[j];
        tmem_ld32(tlane + T_M + 32 * cq, mv);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) a.m[oW2 + u * H + 32 * cq + j] = __uint_as_float(mv[j]);
        tmem_ld32(tlane + T_V + 32 * cq, mv);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) a.v[oW2 + u * H + 32 * cq + j] = __uint_as_float(mv[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = 8 * cq + j;
        if (k < K) {
            a.w[oW1 + u * K + k] = sf[F_W1W + k * H + u];
            a.m[oW1 + u * K + k] = sf[F_W1M + k * H + u];
            a.v[oW1 + u * K + k] = sf[F_W1V + k * H + u];
        }
    }
    if (cq == 0) {
        const int offs[3] = {ob1, ob2, oW3};
#pragma unroll
        for (int p = 0; p < 3; ++p) {
            a.w[offs[p] + u] = sf[F_VEC + (3 * p + 0) * H + u];
            a.m[offs[p] + u] = sf[F_VEC + (3 * p + 1) * H + u];
            a.v[offs[p] + u] = sf[F_VEC + (3 * p + 2) * H + u];
        }
    }
    if (tid == 0) { a.w[ob3] = sf[F_B3]; a.m[ob3] = sf[F_B3 + 1]; a.v[ob3] = sf[F_B3 + 2]; }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, T_COLS);
}

__global__ void tc_adam_consts_kernel(float4* out, int steps, long long step0, float lr, float beta1, float beta2, float eps) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= steps) return;
    const double t = (double)(step0 + s + 1);
    const double bc1 = 1.0 - pow((double)beta1, t), bc2 = 1.0 - pow((double)beta2, t);
    out[s] = make_float4((float)(1.0 / sqrt(bc2)), (float)(-((double)lr / bc1)), (float)sqrt(bc2), (float)(-(double)eps * sqrt(bc2)));
}

long long* g_tc_prof = nullptr;

// fp32 feature matrix of the whole batch, in the reference's dtypes (mlp_baseline.py:36-58): fp64 feature map, then
// .astype(float32); built once per fit, all epochs gather minibatch rows from it.
__global__ void vf_features_kernel(const float* __restrict__ obs, const int* __restrict__ tstep,
                                   const double* __restrict__ returns, long long n, int obs_dim, int K, int KF,
                                   float* __restrict__ feat, float* __restrict__ ret32) {
    // rows of KF = round_up(K, 8) columns, the pad zero-filled: the fit kernels gather them with aligned 16-byte loads
    const long long total = n * KF;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / KF;
        const int k = (int)(i - r * KF);
        float val;
        if (k >= K) {
            val = 0.0f;
        } else if (k < obs_dim) {
            double x = (double)obs[r * obs_dim + k];
            x = fmin(fmax(x, -10.0), 10.0) / 10.0;
            val = (float)x;
        } else {
            const double tau = (double)tstep[r] / 1000.0;
            double p = tau;
            for (int q = obs_dim; q < k; ++q) p *= tau;
            val = (float)p;
        }
        feat[i] = val;
        if (k == 0) ret32[r] = (float)returns[r];
    }
}

}  // namespace

int vf_tc_feat_pitch(int K) { return (K + 7) & ~7; }

cudaError_t vf_build_features(const VfFitArgs& v, float* feat, float* ret32, cudaStream_t s) {
    vf_features_kernel<<<148 * 8, 256, 0, s>>>(v.obs, v.tstep, v.returns, v.n, v.obs_dim, v.K, vf_tc_feat_pitch(v.K), feat, ret32);
    return cudaGetLastError();
}

void vf_tc_set_prof(long long* dev16) { g_tc_prof = dev16; }

constexpr int KS_MAX_HELPERS = 7;                                   // portable cluster size 8 = head + 7 helpers
static int ks_helpers(int K) { return K <= KP ? 0 : (K - KP + KH - 1) / KH; }
bool vf_tc_supported(int K, int H1, int H2, int batch) {
    return batch == NB && H1 == H && H2 == H && K >= 1 && ks_helpers(K) <= KS_MAX_HELPERS;
}
int vf_tc_sms(int K) { return 1 + ks_helpers(K); }
// scratch of the K-split hand-offs: flags (256 B) | dz1 operand 2 x 32 KB | partial sums 2 x 7 x 32 KB
size_t vf_tc_scratch_bytes() { return 256 + 2 * 2 * (size_t)HT_BYTES + 2 * (size_t)KS_MAX_HELPERS * H * NB * 4; }

cudaError_t launch_vf_fit_tc(const VfFitArgs& v, const float* feat, const float* ret32, float4* consts, void* scratch, cudaStream_t s) {
    tc_adam_consts_kernel<<<(v.steps + 255) / 256, 256, 0, s>>>(consts, v.steps, v.step0, v.lr, v.beta1, v.beta2, v.eps);
    TcFitArgs a;
    a.K = v.K; a.KF = vf_tc_feat_pitch(v.K); a.steps = v.steps; a.feat = feat; a.ret32 = ret32; a.perm = v.perm;
    a.reg = v.reg; a.beta1 = v.beta1; a.beta2 = v.beta2; a.eps = v.eps;
    a.w = v.w; a.m = v.m; a.v = v.v; a.consts = consts; a.prof = g_tc_prof;
    a.nh = ks_helpers(v.K);
    a.flags = nullptr; a.dzop = nullptr; a.zpart = nullptr;
    if (a.nh == 0) {
        auto kern = a.prof ? vf_fit_tc_kernel<true, false> : vf_fit_tc_kernel<false, false>;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S_TOTAL);
        if (e != cudaSuccess) return e;
        kern<<<1, NT, S_TOTAL, s>>>(a);
        return cudaGetLastError();
    }
    // K-split: one cluster of 1 + nh CTAs (co-scheduled, so the flag waits between them cannot deadlock)
    unsigned char* sc = static_cast<unsigned char*>(scratch);
    a.flags = reinterpret_cast<int*>(sc);
    a.dzop = sc + 256;
    a.zpart = reinterpret_cast<float*>(sc + 256 + 2 * 2 * (size_t)HT_BYTES);
    cudaError_t e = cudaMemsetAsync(a.flags, 0, 256, s);
    if (e != cudaSuccess) return e;
    auto kern = a.prof ? vf_fit_tc_kernel<true, true> : vf_fit_tc_kernel<false, true>;
    constexpr int SMEM = S_TOTAL > HS_TOTAL ? S_TOTAL : HS_TOTAL;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1 + a.nh); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = SMEM; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 1 + a.nh; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, a);
}

}  // namespace mjb
