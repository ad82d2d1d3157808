// Shared device-side declarations of libb200env: the per-handle device view (Dev), the launch
// arguments, the per-env scalar state and the small helpers every kernel file uses.  Included by
// b200env.cu (fused / streaming kernels, C ABI) and b200tc.cu (tcgen05 eval kernel).
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "b200env.h"

namespace {

constexpr int RAW_DEPTH = 5;      // reference envs/multioptlrs.py:42
constexpr int MAXI = 4;           // forward work items per warp
constexpr int NSTAT = 8;

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_EVAL = 2, MODE_EVAL_STEP = 3, MODE_EVAL_FIRST = 4 };
enum { PASS_U = 0, PASS_G = 1, PASS_R = 2, PASS_E = 3, PASS_S = 4 };
enum { ST_ABSW = 0, ST_LR = 1, ST_LR2 = 2, ST_G = 3, ST_ABSADJG = 4, ST_GDIFF = 5, ST_STATE = 6 };

struct EnvScalars {
    double raw_gsum[RAW_DEPTH];
    float raw_loss[RAW_DEPTH];
    float adj_loss[B2E_MAX_HISTORY];
    float loss_prev;
    int raw_pos, head, nvalid, step, cursor, ord_sel, episode;
};

struct Dev {
    int env_kind, kind, hidden;
    int D, Dp, Ds, N1, N1p, C, Cp;
    int P, Pp, P1, tailP, N, B, E, H, OD;
    int max_batches, act_ver, rew_ver, obs_ver;
    int KT, ntiles;
    int nsc, ncc, nks, fitems;
    int N1g, KR, gcc;
    int row_lex, index_mode, auto_reset;
    int env_base;                    // global index of env 0 of this handle (b2e_config.env_base): the Glorot initialiser's env
    unsigned long long seed;
    float lim1, lim2;
    const float *X;
    const int *labels;
    const float *targets;
    float *w, *gprev, *gnext, *ringw, *ringg;
    double *part;
    EnvScalars *sc;
    int *ord;
    const int *perm;
    long long perm_stride;
    const int *row_of_param;
    const int *param_of_row;
    int off_red2;
    int off_T, off_T2, off_H, off_dP, off_tw, off_tg, off_Z, off_red, off_stage, off_rows, off_idx,
        off_y, off_lb, off_misc;
    int stage_stride, xslack;
    int split, nseg;
    int obs_units;                   // 32-row units per warp item of the observation kernel (32; fewer for small batches: more waves)
    int fast, cg;                    // register-tiled GEMM path (N1 % 8 == 0, B <= 32, 256 threads)
    int ev_X0, ev_X1, ev_W0, ev_W1, ev_XS;   // eval kernel: streamed X / W tile buffers
    int nsegU;
    double *part_u;
    // ring-only steps (b2e_step with obs_out = NULL): partial sums of ring_adjg_kernel [E][nsegU][4] and the
    // per-slot sums of |adjusted weights| / |adjusted gradients| [E][H][2] that states_mean / states_sum
    // are rebuilt from without re-reading the rings
    double *part_r, *slot_abs;
    // observation layout (utils/utils_env.py:22-44): first column of each key's block or -1
    int col_w, col_l, col_g;
    float *w2, *g2;                  // x_{t-2} planes of the raw History, observation version 2
    // generic dense stack (any number of hidden layers / batch size): see gen_eval_kernel
    int generic, nlayers;            // nlayers = Dense layers = hidden layers + 1
    int dims[B2E_MAX_LAYERS + 1];    // widths n_0 = D, n_1.., n_nlayers = C
    int woff[B2E_MAX_LAYERS], boff[B2E_MAX_LAYERS];   // parameter offsets of kernel / bias of layer l
    int aoff[B2E_MAX_LAYERS + 1];    // workspace offset of the activations of layer l (0 = inputs)
    int doff0, doff1;                // two delta buffers [B, max width]
    float *ws;                       // per-CTA workspace
    long long ws_stride;
};

struct StepArgs {
    const float *actions;
    const int *ext_idx;
    const int *ext_cnt;
    float *obs;
    float *reward;
    unsigned char *done;
    double *info;
    const unsigned char *mask;
    const float *init_params;
    float *grad_out;
    float *loss_out;
    int mode;
    int e_begin, e_count;
    // optional work list (reset pipeline of the tcgen05 eval kernel): the envs to visit, ascending, and
    // how many, both in device memory; null = the range e_begin .. e_begin + e_count
    const int *env_list;
    const int *env_count;
};

struct Stats {
    float f[NSTAT];
    double lr, lr2;
};

// ------------------------------------------------------------------ small helpers
__device__ __forceinline__ float nan_to_num_f(float x) {
    if (x != x) return 0.0f;
    if (isinf(x)) return copysignf(FLT_MAX, x);
    return x;
}
__device__ __forceinline__ double nan_to_num_d(double x) {
    if (x != x) return 0.0;
    if (isinf(x)) return copysign(DBL_MAX, x);
    return x;
}
__device__ __forceinline__ float clip_m1(float x) {          // multioptlrs.py:99
    return fminf(fmaxf(nan_to_num_f(x), -100.0f), 100.0f) - 1.0f;
}
__device__ __forceinline__ float action_to_lr(float a, int ver) {   // utils_env.py:102-123
    switch (ver) {
        case 0: return exp10f(a - 4.0f);
        case 1: return a * 1e-3f;
        case 2: return exp2f(a);
        default: return fmaxf((a + 1e3f) * 1e-6f, 0.0f);
    }
}
__device__ __forceinline__ float action_to_delta(float a, int ver) {  // multioptimize.py:95-102
    if (ver == 1) return a * 1e-3f;
    const float mag = exp10f(fabsf(a) - 3.0f);
    return a > 0.f ? mag : (a < 0.f ? -mag : 0.f);
}
// adjusted weight / gradient / loss per observation version (utils/utils_env.py:126-164);
// x0 newest, x1, x2 the two entries before it in the raw History
__device__ __forceinline__ float adjust_w(int ver, float w0, float w1, float w2) {
    switch (ver) {
        case 2: return fabsf(w1 - w2) / (fabsf(w0 - w1) + 1e-8f);
        case 3: return nan_to_num_f(w0 / fabsf(w1));
        default: return w0 / (fabsf(w1) + 1e-3f);
    }
}
__device__ __forceinline__ float adjust_g(int ver, float g0, float g1, float g2) {
    switch (ver) {
        case 1: return g0 * 1e2f;
        case 2: return (g0 - g1) / (fabsf(g1 - g2) + 1e-3f);
        case 3: return nan_to_num_f(g0 / fabsf(g1));
        default: return g0 / (fabsf(g1) + 1e-3f);
    }
}
__device__ __forceinline__ double adjust_l(int ver, double l0, double l1, double l2) {
    switch (ver) {
        case 2: return (l0 - l1) / (fabs(l1 - l2) + 1e-3);
        case 3: return nan_to_num_d(l0 / fabs(l1));
        default: return l0 / (fabs(l1) + 1e-3);
    }
}
__device__ __forceinline__ float glorot(unsigned long long seed, int e, int episode, int p,
                                        float limit) {
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(p + 1);
    z ^= ((unsigned long long)(unsigned)e << 32) | (unsigned)episode;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    float u = (float)((unsigned)(z >> 40)) * (1.0f / 16777216.0f);
    return (2.0f * u - 1.0f) * limit;
}
__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct Totals {
    double v[NSTAT];
};

__device__ __forceinline__ void zero_stats(Stats &st) {
#pragma unroll
    for (int i = 0; i < NSTAT; ++i) st.f[i] = 0.f;
    st.lr = st.lr2 = 0.0;
}

// deterministic block reduction of the per-thread statistics; result valid in thread 0
__device__ void block_reduce(const Stats &st, Totals &tot, double *red) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
#pragma unroll
    for (int i = 0; i < NSTAT; ++i) {
        double v = (i == ST_LR) ? st.lr : (i == ST_LR2) ? st.lr2 : (double)st.f[i];
        v = warp_sum(v);
        if (lane == 0) red[warp * NSTAT + i] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 0; i < NSTAT; ++i) {
            double v = 0.0;
            for (int w = 0; w < nw; ++w) v += red[w * NSTAT + i];
            tot.v[i] = v;
        }
    }
    __syncthreads();
}

// deterministic block sum of one value (fixed order); result in every thread
__device__ double block_sum(double v, double *red) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += red[w];
    return t;
}

// ------------------------------------------------------------- minibatch stream
__device__ __forceinline__ const int *order_ptr(const Dev &d, int e, int sel) {
    return d.ord + ((size_t)sel * d.E + e) * d.N;
}

// InMemoryDataSet.on_epoch_end with the env's fixed permutation: new[i] = old[perm[i]]
__device__ void shuffle_order(const Dev &d, int e, EnvScalars *sc) {
    const int sel = sc->ord_sel;
    const int *src = order_ptr(d, e, sel);
    int *dst = d.ord + ((size_t)(sel ^ 1) * d.E + e) * d.N;
    const int *pm = d.perm + (size_t)e * d.perm_stride;
    for (int i = threadIdx.x; i < d.N; i += blockDim.x) dst[i] = src[pm[i]];
    __syncthreads();
    if (threadIdx.x == 0) sc->ord_sel = sel ^ 1;
    __syncthreads();
}

__device__ void current_batch(const Dev &d, const StepArgs &a, int e, const EnvScalars *sc,
                              const int *&idx, int &cnt) {
    if (d.kind == B2E_PROBLEM_FUNC) { idx = nullptr; cnt = 0; return; }
    if (d.index_mode == B2E_INDEX_EXTERNAL) {
        idx = a.ext_idx + (size_t)e * d.B;
        cnt = a.ext_cnt[e];
    } else {
        const int lo = sc->cursor * d.B;
        idx = order_ptr(d, e, sc->ord_sel) + lo;
        cnt = min(d.B, d.N - lo);
    }
}

// Scalar bookkeeping of one env-step once g_t and L_t are known (one thread): raw and
// adjusted loss histories, reward, done, the scalar info entries, minibatch cursor.
// misc[4] = 1 when the epoch wrapped (the CTA reshuffles), misc[1] = done.
__device__ void step_scalars(const Dev &d, const StepArgs &a, EnvScalars *sc, int e, float loss,
                             double gsum, float *misc) {
    const bool lrs = d.env_kind == B2E_ENV_MULTIOPTLRS;
    const int head_new = (sc->head + 1) % d.H;
    const int nvalid_new = min(sc->nvalid + 1, d.H);
    const double l1 = (double)sc->raw_loss[sc->raw_pos];
    const double l2 = (double)sc->raw_loss[(sc->raw_pos + RAW_DEPTH - 1) % RAW_DEPTH];
    const double adjl = lrs ? nan_to_num_d((double)loss / fabs((double)sc->loss_prev))
                            : adjust_l(d.obs_ver, (double)loss, l1, l2);
    double reward;
    switch (d.rew_ver) {                                       // utils_env.py:71-99
        case 0: reward = -adjl; break;
        case 1: reward = (double)(1.0f / loss); break;
        case 2: reward = -adjl * 100.0; break;
        case 3: reward = (double)(1.0f / loss) * 100.0; break;
        case 4: reward = (double)logf(1.0f / loss); break;
        case 5: reward = -(adjl - 1.0) * (adjl - 1.0); break;
        default: reward = -(adjl - 1.0); break;
    }
    const int step = sc->step + 1;                             // baseenvironment.py:37
    bool done = step >= d.max_batches;
    if (lrs) {
        reward = fmin(fmax(reward, -100.0), 100.0);            // multioptlrs.py:103
        if (!done && loss > 1e4f) {                            // multioptlrs.py:105-107
            done = true;
            reward -= (double)(d.max_batches - step);
        }
    }
    const int rp = (sc->raw_pos + 1) % RAW_DEPTH;
    sc->raw_pos = rp;
    sc->raw_loss[rp] = loss;
    sc->raw_gsum[rp] = gsum;
    sc->loss_prev = loss;
    sc->adj_loss[head_new] = (float)adjl;
    sc->head = head_new;
    sc->nvalid = nvalid_new;
    sc->step = step;
    double gs = 0.0, ls = 0.0;
    for (int i = 0; i < RAW_DEPTH; ++i) { gs += sc->raw_gsum[i]; ls += (double)sc->raw_loss[i]; }
    double *info = a.info + (size_t)e * B2E_INFO_STRIDE;
    info[0] = done ? (double)loss : nan("");                   // multioptlrs.py:108-110
    info[1] = (double)loss;
    info[8] = gs / (RAW_DEPTH * (double)d.P);
    info[9] = gs;
    info[10] = ls / RAW_DEPTH;
    info[11] = adjl;
    info[14] = reward;                                         // baseenvironment.py:40
    info[15] = (double)step;
    a.reward[e] = (float)reward;
    a.done[e] = done ? 1 : 0;
    misc[1] = done ? 1.f : 0.f;
    misc[4] = 0.f;
    // MultiOptLRs moves to the next minibatch (multioptlrs.py:128); MultiOptimize never does
    if (lrs && d.kind != B2E_PROBLEM_FUNC && d.index_mode == B2E_INDEX_INTERNAL) {
        const int cur = sc->cursor + 1;                        // optimize_nn.py:102-112
        misc[4] = (cur * d.B >= d.N) ? 1.f : 0.f;
        sc->cursor = (cur * d.B >= d.N) ? 0 : cur;
    }
}

}  // namespace
