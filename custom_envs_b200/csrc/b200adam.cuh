// The Adam baseline of libb200env (b2e_step_adam, include/b200env.h): Keras 2.2 Adam.get_updates with
// amsgrad = False in place of the agent's learning rates.  Included by b200env.cu and b200tiny.cu, whose
// Adam kernels take these arguments next to Dev and StepArgs.
#pragma once
#include "b200env_shared.cuh"

namespace {

struct AdamArgs {
    const float *lr;                 // [E]
    float *m, *v;                    // [E, P], natural order, owned by the caller
    float b1, b2, eps;
};

// alpha_t = lr sqrt(1 - b2^t) / (1 - b1^t) of env e at its step t, evaluated in fp64 and rounded once
__device__ __forceinline__ float adam_alpha(const AdamArgs &o, int e, int t) {
    const double b1t = pow((double)o.b1, (double)t), b2t = pow((double)o.b2, (double)t);
    return (float)((double)o.lr[e] * sqrt(1.0 - b2t) / (1.0 - b1t));
}

// g: the gradient of the MEAN minibatch loss; m, v: the moments of step t - 1, in and out (zero at t = 1
// whatever they hold).  Returns the per-parameter rate alpha_t / (sqrt(v_t) + eps) that multiplies m_t.
__device__ __forceinline__ float adam_moments(const AdamArgs &o, float alpha, bool first, float g, float &m, float &v) {
    const float mp = first ? 0.f : m, vp = first ? 0.f : v;
    m = fmaf(o.b1, mp, __fmul_rn(1.f - o.b1, g));
    v = fmaf(o.b2, vp, __fmul_rn(1.f - o.b2, __fmul_rn(g, g)));
    return alpha / (sqrtf(v) + o.eps);
}

// g = g0 / cnt: the batch-SUM gradient over the minibatch's valid rows (cnt = 0: the func problem, g = g0)
__device__ __forceinline__ float adam_mean_grad(float g0, float cnt) { return cnt > 0.f ? g0 / cnt : g0; }

// The Adam argument of a kernel that serves both steps: a pack of none (b2e_step) or one AdamArgs (b2e_step_adam)
__device__ __forceinline__ const AdamArgs &adam_of(const AdamArgs &o) { return o; }

}  // namespace
