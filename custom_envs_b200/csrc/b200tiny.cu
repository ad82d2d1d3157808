// Warp-per-env step of libb200env for tiny problems (BASELINE config 2: softmax regression on
// iris-shaped data, 4 -> 3, P = 15 agents, minibatch 32, 1024 lock-step envs).
//
// One env-step = MultiOptLRs.base_step (reference envs/multioptlrs.py:80-129): gradient at w_{t-1},
// per-parameter learning-rate update, loss / gradient at w_t on the same minibatch, adjusted
// histories, observation rows, reward, done flag, the 14 info statistics, minibatch cursor, and
// base_reset (multioptlrs.py:66-78) for envs that finished.  The block-per-env fused kernel
// (optenv_kernel, b200env.cu) spends 32 us per batched step on this shape: eight block barriers per
// phase around 15 parameters of work, 3.5 rounds of CTAs.  Here a WARP owns an env:
//   lane = minibatch sample for the forward / softmax cross-entropy (features in registers, the
//          weights broadcast from the warp's shared-memory slice),
//   lane = parameter (up to 3 per lane) for the gradient sums, update, ratios, rings, observation row,
// every exchange is a __syncwarp or a shuffle, the statistics are warp reductions in fp64, and the
// 1024 envs are one wave of 256 four-warp CTAs.  Arithmetic per element is that of the fused kernel
// (same formulas, sums over the samples in index order), so both are held to the same oracle.
#include <cuda_runtime.h>
#include <stdint.h>

#include "b200env_shared.cuh"
#include "b200tiny.h"

namespace {
namespace tiny {

constexpr int DMAX = 8, CMAX = 8, PL = 3, WARPS = 4, PMAX = 32 * PL, OBS_MAX = 1536;

struct WarpSmem {
    float w[PMAX];                // the env's parameters (kernel [D][C] row major, then bias [C])
    float xs[32 * DMAX];          // minibatch features [sample][feature]
    float zs[32 * CMAX];          // d loss / d logits [sample][class]
    float obs[OBS_MAX];           // observation rows of the env in VecEnv row order
};

struct Batch {
    float x[DMAX];
    float yt[CMAX];
    int y, cnt;
};

__device__ __forceinline__ float ratio_nn(float num, float den) { return nan_to_num_f(num / fabsf(den)); }
__device__ __forceinline__ float clip_only_m1(float x) { return fminf(fmaxf(x, -100.0f), 100.0f) - 1.0f; }

// DD / CC > 0: feature and output counts known at compile time (iris: 4, 3), which keeps the unrolled code -- every
// warp runs it exactly once, so the kernel is bound by instruction fetch -- as short as the problem
template <int DD, int CC>
__device__ __forceinline__ void load_batch(const Dev &d, const StepArgs &a, int e, const EnvScalars *sc, int lane, Batch &b) {
    constexpr int DB = DD ? DD : DMAX, CB = CC ? CC : CMAX;
    const int D = DD ? DD : d.D, C = CC ? CC : d.C;
    const int *idx;
    current_batch(d, a, e, sc, idx, b.cnt);
    const bool live = lane < b.cnt;
    const size_t row = live ? (size_t)idx[lane] : 0;
#pragma unroll
    for (int k = 0; k < DMAX; ++k) b.x[k] = 0.f;
#pragma unroll
    for (int k = 0; k < DB; ++k) b.x[k] = (live && k < D) ? d.X[row * d.Dp + k] : 0.f;
    b.y = 0;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) b.yt[c] = 0.f;
    if (d.kind == B2E_PROBLEM_SOFTMAX) {
        b.y = live ? d.labels[row] : 0;
    } else {
#pragma unroll
        for (int c = 0; c < CB; ++c) if (live && c < C) b.yt[c] = d.targets[row * C + c];
    }
}

// loss (mean over the minibatch) and batch-SUM gradient (problems/optimize_nn.py:47-52) at the parameters in S.w;
// g[j] = component lane + 32 j
template <int DD, int CC>
__device__ __forceinline__ float eval(const Dev &d, WarpSmem &S, const Batch &b, int lane, float (&g)[PL]) {
    constexpr int DMAX = DD ? DD : tiny::DMAX, CMAX = CC ? CC : tiny::CMAX;      // loop bounds of this instantiation
    const int D = DD ? DD : d.D, C = CC ? CC : d.C, P1 = d.P1;
    float z[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
        float v = 0.f;
        if (c < C) {
#pragma unroll
            for (int k = 0; k < DMAX; ++k) if (k < D) v = fmaf(b.x[k], S.w[k * C + c], v);
            v += S.w[P1 + c];
        }
        z[c] = v;
    }
    float loss = 0.f;
    const bool live = lane < b.cnt;
    if (d.kind == B2E_PROBLEM_SOFTMAX) {
        float m = z[0];
#pragma unroll
        for (int c = 1; c < CMAX; ++c) if (c < C) m = fmaxf(m, z[c]);
        float sum = 0.f, zy = 0.f;
#pragma unroll
        for (int c = 0; c < CMAX; ++c) if (c < C) { sum += expf(z[c] - m); if (c == b.y) zy = z[c]; }
        loss = (m + logf(sum)) - zy;
        const float inv = 1.0f / sum;
#pragma unroll
        for (int c = 0; c < CMAX; ++c) z[c] = (live && c < C) ? expf(z[c] - m) * inv - (c == b.y ? 1.f : 0.f) : 0.f;
    } else {                                                  // utils/utils_math.py:37-48
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
            const float df = (live && c < C) ? z[c] - b.yt[c] : 0.f;
            loss = fmaf(0.5f * df, df, loss);
            z[c] = df;
        }
    }
    if (!live) loss = 0.f;
    // mean loss: the samples in index order, as the fused kernel adds them
    __syncwarp();
#pragma unroll
    for (int k = 0; k < DMAX; ++k) S.xs[lane * tiny::DMAX + k] = b.x[k];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) S.zs[lane * tiny::CMAX + c] = z[c];
    float lsum = 0.f;
    for (int s = 0; s < b.cnt; ++s) lsum += __shfl_sync(0xffffffffu, loss, s);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < PL; ++j) {
        const int p = lane + 32 * j;
        float acc = 0.f;
        if (p < P1) {
            const int k = p / C, c = p - k * C;
            for (int s = 0; s < b.cnt; ++s) acc = fmaf(S.xs[s * tiny::DMAX + k], S.zs[s * tiny::CMAX + c], acc);
        } else if (p < d.P) {
            const int c = p - P1;
            for (int s = 0; s < b.cnt; ++s) acc += S.zs[s * tiny::CMAX + c];
        }
        g[j] = acc;
    }
    return lsum / (float)b.cnt;
}

// InMemoryDataSet.on_epoch_end with the env's permutation (shared shuffle_order, warp version)
__device__ __forceinline__ void warp_shuffle_order(const Dev &d, int e, EnvScalars *sc, int lane) {
    const int sel = sc->ord_sel;
    const int *src = order_ptr(d, e, sel);
    int *dst = d.ord + ((size_t)(sel ^ 1) * d.E + e) * d.N;
    const int *pm = d.perm + (size_t)e * d.perm_stride;
    for (int i = lane; i < d.N; i += 32) dst[i] = src[pm[i]];
    __syncwarp();
    if (lane == 0) sc->ord_sel = sel ^ 1;
    __syncwarp();
}

// base_reset (multioptlrs.py:66-78) of one env by its warp
template <int DD, int CC>
__device__ __noinline__ void reset_one(const Dev &d, const StepArgs &a, WarpSmem &S, int e, int lane) {
    EnvScalars *sc = d.sc + e;
    if (d.index_mode == B2E_INDEX_INTERNAL) {
        warp_shuffle_order(d, e, sc, lane);                   // optimize_nn.py:114-120
        if (lane == 0) sc->cursor = 0;
        __syncwarp();
    }
    Batch b;
    load_batch<DD, CC>(d, a, e, sc, lane, b);
    const int episode = sc->episode;
    float *wE = d.w + (size_t)e * d.Pp;
#pragma unroll
    for (int j = 0; j < PL; ++j) {
        const int p = lane + 32 * j;
        float v = 0.f;
        if (p < d.P) {
            if (a.init_params) v = a.init_params[(size_t)e * d.P + p];
            else if (p < d.P1) v = glorot(d.seed, e + d.env_base, episode, p, d.lim1);      // keras Dense: Glorot kernel, zero bias
        }
        if (p < d.Pp) wE[p] = v;
        S.w[p] = v;
    }
    __syncwarp();
    float g[PL];
    const float loss = eval<DD, CC>(d, S, b, lane, g);
    float gs = 0.f;
    float *gE = d.gprev + (size_t)e * d.Pp;
#pragma unroll
    for (int j = 0; j < PL; ++j) {
        const int p = lane + 32 * j;
        if (p < d.P) { gE[p] = g[j]; gs += g[j]; }
    }
    const double gsum = warp_sum((double)gs);
    if (lane == 0) {
        for (int i = 0; i < RAW_DEPTH; ++i) { sc->raw_loss[i] = 0.f; sc->raw_gsum[i] = 0.0; }
        for (int i = 0; i < B2E_MAX_HISTORY; ++i) sc->adj_loss[i] = 0.f;
        sc->raw_pos = 0;
        sc->raw_loss[0] = loss;
        sc->raw_gsum[0] = gsum;
        sc->loss_prev = loss;
        sc->head = d.H - 1;
        sc->nvalid = 0;
        sc->step = 0;
        sc->episode = episode + 1;
    }
    if (a.obs) {
        float *o = a.obs + (size_t)e * d.P * d.OD;
        for (int i = lane; i < d.P * d.OD; i += 32) o[i] = -1.0f;
    }
    __syncwarp();
}

template <int HT, int DD, int CC>
__global__ void __launch_bounds__(WARPS * 32) tiny_env_kernel(const __grid_constant__ Dev d, const __grid_constant__ StepArgs a) {
    __shared__ WarpSmem smem[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = a.e_begin + blockIdx.x * WARPS + warp;
    if (e >= a.e_begin + a.e_count) return;
    WarpSmem &S = smem[warp];
    if (a.mode == MODE_RESET) {
        if (a.mask == nullptr || a.mask[e]) reset_one<DD, CC>(d, a, S, e, lane);
        return;
    }
    const int H = HT ? HT : d.H, P = d.P, OD = 3 * H;
    EnvScalars *sc = d.sc + e;
    constexpr int HB = HT ? HT : B2E_MAX_HISTORY;
    Batch b;
    load_batch<DD, CC>(d, a, e, sc, lane, b);
    float *wE = d.w + (size_t)e * d.Pp;
    float *gE = d.gprev + (size_t)e * d.Pp;
    float wv[PL], gt[PL];
#pragma unroll
    for (int j = 0; j < PL; ++j) {
        const int p = lane + 32 * j;
        wv[j] = p < P ? wE[p] : 0.f;
        S.w[p] = wv[j];
    }
    __syncwarp();
    const int head_new = (sc->head + 1) % H;
    const int nvalid_new = min(sc->nvalid + 1, H);
    float *rw = d.ringw + (size_t)e * H * d.Pp, *rg = d.ringg + (size_t)e * H * d.Pp;
    float s_absw = 0.f, s_absadjg = 0.f, s_gdiff = 0.f, s_state = 0.f, s_g = 0.f;
    double s_lr = 0.0, s_lr2 = 0.0;
    float aw[PL];
    int row[PL];
    float loss = 0.f;
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {                     // one copy of the eval code serves both evaluations
        loss = eval<DD, CC>(d, S, b, lane, gt);                // multioptlrs.py:85 at w_{t-1}, :88 at w_t (same minibatch)
        if (pass == 0) {
            __syncwarp();
#pragma unroll
            for (int j = 0; j < PL; ++j) {                     // multioptlrs.py:86-87, utils_env.py:158-159
                const int p = lane + 32 * j;
                row[j] = 0; aw[j] = 0.f;
                if (p < P) {
                    row[j] = d.row_lex ? d.row_of_param[p] : p;
                    const float lr = action_to_lr(a.actions[(size_t)e * P + row[j]], d.act_ver);
                    const float wn = fmaf(-gt[j], lr, wv[j]);
                    aw[j] = ratio_nn(wn, wv[j]);
                    s_absw += fabsf(wn);
                    s_lr += (double)lr;
                    s_lr2 += (double)lr * (double)lr;
                    wE[p] = wn;
                    rw[(size_t)head_new * d.Pp + p] = aw[j];
                    S.w[p] = wn;
                }
            }
            __syncwarp();
        }
    }
    const double adjl = nan_to_num_d((double)loss / fabs((double)sc->loss_prev));
    float ol[HB];
    double labs = 0.0;
#pragma unroll
    for (int h = 0; h < HB; ++h) {
        if (h < H) {
            float v = 0.f;
            if (h == 0) v = (float)adjl;
            else if (h < nvalid_new) {
                int slot = head_new - h;
                slot += slot < 0 ? H : 0;
                v = sc->adj_loss[slot];
            }
            ol[h] = clip_m1(v);
            labs += (double)fabsf(v);
        }
    }
#pragma unroll
    for (int j = 0; j < PL; ++j) {                             // utils_env.py:156-157, multioptlrs.py:93-101
        const int p = lane + 32 * j;
        if (p < P) {
            const float gp = gE[p];
            const float ag = ratio_nn(gt[j], gp);
            s_absadjg += fabsf(ag);
            s_gdiff += fabsf(gt[j] - gp);
            s_g += gt[j];
            gE[p] = gt[j];
            rg[(size_t)head_new * d.Pp + p] = ag;
            float *orow = S.obs + row[j] * OD;
#pragma unroll
            for (int h = 0; h < HB; ++h) {
                if (h < H) {
                    float w_h = 0.f, g_h = 0.f;
                    if (h == 0) { w_h = aw[j]; g_h = ag; }
                    else if (h < nvalid_new) {
                        int slot = head_new - h;
                        slot += slot < 0 ? H : 0;
                        w_h = rw[(size_t)slot * d.Pp + p];
                        g_h = rg[(size_t)slot * d.Pp + p];
                    }
                    s_state += fabsf(w_h) + fabsf(g_h);
                    orow[h] = clip_only_m1(w_h);
                    orow[H + h] = ol[h];
                    orow[2 * H + h] = clip_only_m1(g_h);
                }
            }
        }
    }
    __syncwarp();
    {
        float *o = a.obs + (size_t)e * P * OD;
        for (int i = lane; i < P * OD; i += 32) o[i] = S.obs[i];
    }
    const double t_absw = warp_sum((double)s_absw), t_lr = warp_sum(s_lr), t_lr2 = warp_sum(s_lr2);
    const double t_absadjg = warp_sum((double)s_absadjg), t_gdiff = warp_sum((double)s_gdiff);
    const double t_state = warp_sum((double)s_state), t_g = warp_sum((double)s_g);
    int flags = 0;
    if (lane == 0) {                                          // multioptlrs.py:102-128, baseenvironment.py:37-40
        double reward;
        switch (d.rew_ver) {                                  // utils_env.py:71-99
            case 0: reward = -adjl; break;
            case 1: reward = (double)(1.0f / loss); break;
            case 2: reward = -adjl * 100.0; break;
            case 3: reward = (double)(1.0f / loss) * 100.0; break;
            case 4: reward = (double)logf(1.0f / loss); break;
            case 5: reward = -(adjl - 1.0) * (adjl - 1.0); break;
            default: reward = -(adjl - 1.0); break;
        }
        reward = fmin(fmax(reward, -100.0), 100.0);
        const int step = sc->step + 1;
        bool done = step >= d.max_batches;
        if (!done && loss > 1e4f) {
            done = true;
            reward -= (double)(d.max_batches - step);
        }
        const int rp = (sc->raw_pos + 1) % RAW_DEPTH;
        sc->raw_pos = rp;
        sc->raw_loss[rp] = loss;
        sc->raw_gsum[rp] = t_g;
        sc->loss_prev = loss;
        sc->adj_loss[head_new] = (float)adjl;
        sc->head = head_new;
        sc->nvalid = nvalid_new;
        sc->step = step;
        double gsum = 0.0, lsum = 0.0;
        for (int i = 0; i < RAW_DEPTH; ++i) { gsum += sc->raw_gsum[i]; lsum += (double)sc->raw_loss[i]; }
        const double Pd = (double)P, invP = 1.0 / Pd;        // one fp64 division instead of eight
        const double lr_mean = t_lr * invP;
        double lr_var = t_lr2 * invP - lr_mean * lr_mean;
        lr_var = lr_var > 0.0 ? lr_var : 0.0;
        const double ssum = t_state + Pd * labs;
        double *info = a.info + (size_t)e * B2E_INFO_STRIDE;
        info[0] = done ? (double)loss : nan("");
        info[1] = (double)loss;
        info[2] = t_absw * invP;
        info[3] = t_absw;
        info[4] = lr_mean;
        info[5] = sqrt(lr_var);
        info[6] = ssum * invP / (double)OD;
        info[7] = ssum;
        info[8] = gsum * invP * (1.0 / RAW_DEPTH);
        info[9] = gsum;
        info[10] = lsum * (1.0 / RAW_DEPTH);
        info[11] = adjl;
        info[12] = t_absadjg * invP;
        info[13] = t_gdiff * invP;
        info[14] = reward;
        info[15] = (double)step;
        a.reward[e] = (float)reward;
        a.done[e] = done ? 1 : 0;
        flags = done ? 1 : 0;
        if (d.index_mode == B2E_INDEX_INTERNAL) {
            const int cur = sc->cursor + 1;                   // optimize_nn.py:102-112
            if (cur * d.B >= d.N) flags |= 2;
            sc->cursor = (cur * d.B >= d.N) ? 0 : cur;
        }
    }
    flags = __shfl_sync(0xffffffffu, flags, 0);
    __syncwarp();
    if (flags & 2) warp_shuffle_order(d, e, sc, lane);
    if ((flags & 1) && d.auto_reset) reset_one<DD, CC>(d, a, S, e, lane);
}

}  // namespace tiny
}  // namespace

bool b2e_tiny_supported(const void *dev) {
    const Dev &d = *static_cast<const Dev *>(dev);
    return d.env_kind == B2E_ENV_MULTIOPTLRS && !d.split && !d.generic && !d.hidden &&
           (d.kind == B2E_PROBLEM_SOFTMAX || d.kind == B2E_PROBLEM_LINREG) &&
           d.D >= 1 && d.D <= tiny::DMAX && d.C >= 1 && d.C <= tiny::CMAX && d.B <= 32 &&
           d.P <= tiny::PMAX && d.P * 3 * d.H <= tiny::OBS_MAX && d.H <= B2E_MAX_HISTORY && d.OD == 3 * d.H;
}

int b2e_tiny_launch(const void *dev, const void *args, void *stream) {
    const Dev &d = *static_cast<const Dev *>(dev);
    const StepArgs &a = *static_cast<const StepArgs *>(args);
    const int grid = (a.e_count + tiny::WARPS - 1) / tiny::WARPS;
    const cudaStream_t cs = (cudaStream_t)stream;
    if (d.H == 5 && d.D == 4 && d.C == 3) tiny::tiny_env_kernel<5, 4, 3><<<grid, tiny::WARPS * 32, 0, cs>>>(d, a);   // iris
    else if (d.H == 5) tiny::tiny_env_kernel<5, 0, 0><<<grid, tiny::WARPS * 32, 0, cs>>>(d, a);
    else tiny::tiny_env_kernel<0, 0, 0><<<grid, tiny::WARPS * 32, 0, cs>>>(d, a);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}
