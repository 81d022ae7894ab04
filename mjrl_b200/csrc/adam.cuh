// torch.optim.Adam's per-element update (single-tensor path, no amsgrad), shared by the sequential minibatch kernels
// (vf_fit.cu: value net, policy_sgd.cu: policy).  The per-step constants are computed in double from the step
// count, as torch does with its Python-float bias corrections.
#pragma once
#include "common.cuh"

namespace mjb {

struct AdamC { float one_m_b1, b2, one_m_b2, bc2_sqrt, eps, neg_step, reg; };

__device__ __forceinline__ float adam_step(float g, float w, float* m, float* v, const AdamC& c) {
    g = fmaf(c.reg, w, g);                               // grad.add(param, alpha=weight_decay)
    const float mn = *m + c.one_m_b1 * (g - *m);         // exp_avg.lerp_(grad, 1-beta1)
    const float vn = fmaf(c.one_m_b2 * g, g, *v * c.b2); // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1-beta2)
    *m = mn; *v = vn;
    const float denom = sqrtf(vn) / c.bc2_sqrt + c.eps;
    return fmaf(c.neg_step, mn / denom, w);              // param.addcdiv_(exp_avg, denom, value=-step_size)
}

}  // namespace mjb
