// libb200env: fused batched step of custom_envs' optimisation environments for sm_100a.
//
// One CTA owns one env for the whole step.  Per env-step (MultiOptLRs semantics, reference
// envs/multioptlrs.py:80-129) the CTA
//   1. gathers the minibatch rows into shared memory (reference dataset/inmemorydataset.py:24-28),
//   2. forward/backward at w_{t-1}  ->  g0                     (problems/optimize_nn.py:122-126),
//   3. w_t = w_{t-1} - g0 * 10^(a-4), streams w_t back to HBM  (multioptlrs.py:86-87),
//   4. forward/backward at w_t on the same batch -> g_t, L_t   (multioptlrs.py:88),
//   5. ratio history + per-parameter observation rows + reward + the 14 info statistics
//      (utils/utils_env.py:155-164, utils/utils_common.py:188-196, multioptlrs.py:89-127),
//   6. advances the env's minibatch cursor / epoch shuffle     (problems/optimize_nn.py:102-112),
//   7. re-initialises the env if the episode ended             (vectorize/concurrentvecenv.py:32-38).
// The first-layer matrix W1[D,N1] is streamed through a shared-memory tile; everything
// else of the network ("tail": b1, W2, b2) is shared-memory resident.  All arithmetic fp32
// (FFMA), statistics reduced in fp64.  See DESIGN.md for the data layout and traffic model.
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <string>

#include "b200env.h"

#include "b200env_shared.cuh"
#include "b200tc.h"
#include "b200env_internal.h"
#include "b200tiny.h"
#include "b200thin.h"

namespace {

// ---------------------------------------------------------------- minibatch gather
__device__ void load_batch(const Dev &d, float *sm, const int *idx_g, int cnt) {
    float *Xs = sm;
    int *idx_s = reinterpret_cast<int *>(sm + d.off_idx);
    for (int r = threadIdx.x; r < d.B; r += blockDim.x) idx_s[r] = (r < cnt) ? idx_g[r] : 0;
    __syncthreads();
    const int qrow = d.Ds >> 2, qdata = d.Dp >> 2;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int total = d.B * qrow + (d.xslack >> 2);          // + slack after the last row
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int r = i / qrow, c = i - r * qrow;
        float4 v = zero4;
        if (r < cnt && c < qdata)
            v = __ldg(reinterpret_cast<const float4 *>(d.X + (size_t)idx_s[r] * d.Dp) + c);
        reinterpret_cast<float4 *>(Xs)[i] = v;
    }
    if (d.kind == B2E_PROBLEM_SOFTMAX) {
        int *ys = reinterpret_cast<int *>(sm + d.off_y);
        for (int r = threadIdx.x; r < d.B; r += blockDim.x)
            ys[r] = (r < cnt) ? d.labels[idx_s[r]] : 0;
    } else if (d.kind == B2E_PROBLEM_LINREG) {
        float *yt = sm + d.off_y;
        for (int i = threadIdx.x; i < d.B * d.C; i += blockDim.x) {
            const int r = i / d.C, c = i - r * d.C;
            yt[i] = (r < cnt) ? d.targets[(size_t)idx_s[r] * d.C + c] : 0.f;
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------- forward pass
// Hpre[s][c] += sum_{k in tile} Xs[s][k0+k] * T[k][c]; lane = sample, 8 columns per item.
__device__ __forceinline__ void f_accumulate(const Dev &d, const float *Xs, const float *T,
                                             int k0, int krows4, float (&acc)[MAXI][8]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int kslice = d.KT / d.nks;
#pragma unroll
    for (int j = 0; j < MAXI; ++j) {
        const int it = warp + j * nw;
        if (it < d.fitems) {
            const int sc = it % d.nsc, rest = it / d.nsc;
            const int cc = rest % d.ncc, ks = rest / d.ncc;
            int s = sc * 32 + lane;
            s = s < d.B ? s : d.B - 1;
            const float *xrow = Xs + s * d.Ds + k0;
            const float *tcol = T + cc * 8;
            const int kb = ks * kslice;
            int ke = kb + kslice;
            ke = ke < krows4 ? ke : krows4;
            for (int k = kb; k < ke; k += 4) {
                const float4 x = *reinterpret_cast<const float4 *>(xrow + k);
                const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float *t = tcol + (k + kk) * d.N1p;
                    const float4 t0 = *reinterpret_cast<const float4 *>(t);
                    const float4 t1 = *reinterpret_cast<const float4 *>(t + 4);
                    acc[j][0] = fmaf(xv[kk], t0.x, acc[j][0]);
                    acc[j][1] = fmaf(xv[kk], t0.y, acc[j][1]);
                    acc[j][2] = fmaf(xv[kk], t0.z, acc[j][2]);
                    acc[j][3] = fmaf(xv[kk], t0.w, acc[j][3]);
                    acc[j][4] = fmaf(xv[kk], t1.x, acc[j][4]);
                    acc[j][5] = fmaf(xv[kk], t1.y, acc[j][5]);
                    acc[j][6] = fmaf(xv[kk], t1.z, acc[j][6]);
                    acc[j][7] = fmaf(xv[kk], t1.w, acc[j][7]);
                }
            }
        }
    }
}

__device__ void f_store(const Dev &d, float *sm, float (&acc)[MAXI][8]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    float *Hb = sm + d.off_H;
    float *red = sm + d.off_red;
#pragma unroll
    for (int j = 0; j < MAXI; ++j) {
        const int it = warp + j * nw;
        if (it < d.fitems) {
            const int sc = it % d.nsc, rest = it / d.nsc;
            const int cc = rest % d.ncc, ks = rest / d.ncc;
            const int s = sc * 32 + lane;
            if (s < d.B) {
                float *dst = (d.nks == 1 ? Hb : red + (size_t)ks * d.B * d.N1p) + s * d.N1p + cc * 8;
#pragma unroll
                for (int c = 0; c < 8; ++c) dst[c] = acc[j][c];
            }
        }
    }
    __syncthreads();
    if (d.nks > 1) {
        const int n = d.B * d.N1p;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            float v = 0.f;
            for (int ks = 0; ks < d.nks; ++ks) v += red[(size_t)ks * n + i];
            Hb[i] = v;
        }
        __syncthreads();
    }
}

__device__ __forceinline__ void zero_acc(float (&acc)[MAXI][8]) {
#pragma unroll
    for (int j = 0; j < MAXI; ++j)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[j][c] = 0.f;
}

// copy W1 rows [k0, k0+krows) from HBM (natural, stride N1) into the tile (stride N1p);
// rows up to krows4 are zero filled.
__device__ void load_w_tile(const Dev &d, float *T, const float *wE, int k0, int krows,
                            int krows4) {
    if (d.N1p == d.N1) {
        const int nq = (krows * d.N1) >> 2;
        const float4 *src = reinterpret_cast<const float4 *>(wE + (size_t)k0 * d.N1);
        for (int i = threadIdx.x; i < nq; i += blockDim.x)
            reinterpret_cast<float4 *>(T)[i] = src[i];
    } else {
        const int n = krows * d.N1;
        const float *src = wE + (size_t)k0 * d.N1;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int k = i / d.N1, c = i - k * d.N1;
            T[k * d.N1p + c] = src[i];
        }
        for (int i = threadIdx.x; i < krows * (d.N1p - d.N1); i += blockDim.x) {
            const int k = i / (d.N1p - d.N1), c = d.N1 + i - k * (d.N1p - d.N1);
            T[k * d.N1p + c] = 0.f;
        }
    }
    for (int i = krows * d.N1p + threadIdx.x; i < krows4 * d.N1p; i += blockDim.x) T[i] = 0.f;
}

// Hpre = X . W1 with W1 read from HBM
__device__ void forward_from_global(const Dev &d, float *sm, const float *wE) {
    float acc[MAXI][8];
    zero_acc(acc);
    float *T = sm + d.off_T;
    for (int t = 0; t < d.ntiles; ++t) {
        const int k0 = t * d.KT;
        const int krows = min(d.KT, d.D - k0), krows4 = (krows + 3) & ~3;
        load_w_tile(d, T, wE, k0, krows, krows4);
        __syncthreads();
        f_accumulate(d, sm, T, k0, krows4, acc);
        __syncthreads();
    }
    f_store(d, sm, acc);
}

// ------------------------------------------------------------------ backward tile
// T[k][c] = sum_s Xs[s][k0+k] * dPre[s][c] for the rows of one tile (lane = column).
__device__ void g_compute(const Dev &d, const float *sm, float *T, int k0, int cnt) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const float *Xs = sm;
    const float *dP = sm + d.off_dP;
    const int nitems = (d.KT / d.KR) * d.gcc;
    for (int it = warp; it < nitems; it += nw) {
        const int kc = it / d.gcc, c0 = (it - kc * d.gcc) * 32;
        if (k0 + kc * d.KR >= d.D) continue;
        const int r = lane / d.N1g, c = c0 + (lane & (d.N1g - 1));
        const int kl = kc * d.KR + r * 8;
        const int cc = c < d.N1p ? c : d.N1p - 1;
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        const float *xr = Xs + k0 + kl;
        const float *dp = dP + cc;
        for (int s = 0; s < cnt; ++s) {
            const float4 x0 = *reinterpret_cast<const float4 *>(xr + s * d.Ds);
            const float4 x1 = *reinterpret_cast<const float4 *>(xr + s * d.Ds + 4);
            const float dv = dp[s * d.N1p];
            acc[0] = fmaf(x0.x, dv, acc[0]);
            acc[1] = fmaf(x0.y, dv, acc[1]);
            acc[2] = fmaf(x0.z, dv, acc[2]);
            acc[3] = fmaf(x0.w, dv, acc[3]);
            acc[4] = fmaf(x1.x, dv, acc[4]);
            acc[5] = fmaf(x1.y, dv, acc[5]);
            acc[6] = fmaf(x1.z, dv, acc[6]);
            acc[7] = fmaf(x1.w, dv, acc[7]);
        }
        if (c < d.N1) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (k0 + kl + j < d.D) T[(kl + j) * d.N1p + c] = acc[j];
        }
    }
}

// ------------------------------------------------ register-tiled variants (fast path)
// Used when N1 is a multiple of 8 that divides the CTA into column groups (e.g. 64):
// forward : thread = 4 samples x 8 columns, K split over the 4 quarters of the CTA;
// backward: thread = 4 rows x 8 columns of the tile, all samples.
// A thread's 8 columns are two runs of 4, N1/2 apart, so that a warp's float4 accesses
// cover whole 128-byte lines.
// Packed fp32 FMA (FFMA2 on sm_100): two IEEE fmas per instruction, bit-identical to two FFMAs.
// The FMA pipe has the same peak either way (profiles/tools/ffma2_bench.cu: 73 TFLOP/s), but the
// eval kernel is issue bound and FFMA2 halves the issue slots its multiply-adds take.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void ffma2(f32x2 &acc, f32x2 a, f32x2 b) {
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}

// CN1 > 0 fixes the layer width (and B = 32, 256 threads) at compile time so that the strides
// become immediates; CN1 = 0 reads them from the Dev.
template <int CN1 = 0>
__device__ __forceinline__ void f_accumulate_fast(const Dev &d, const float *xbase, int xstride,
                                                  const float *T, int krows4, float (&acc)[4][8]) {
    const int t = threadIdx.x;
    const int N1 = CN1 ? CN1 : d.N1, N1p = CN1 ? CN1 : d.N1p, cg = CN1 ? CN1 / 8 : d.cg;
    const int nB = CN1 ? 32 : d.B, nthreads = CN1 ? 256 : (int)blockDim.x;
    const int per_slice = 8 * cg;                         // threads per K slice
    const int q = t / per_slice, u = t - q * per_slice;
    const int sg = u / cg, cgi = u - sg * cg;
    const int nslices = nthreads / per_slice;
    const int rows_per = ((krows4 / 4 + nslices - 1) / nslices) * 4;
    const int kb = q * rows_per;
    int ke = kb + rows_per;
    ke = ke < krows4 ? ke : krows4;
    const int half = N1 >> 1;
    const float *xr[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int s = sg + 8 * i;
        s = s < nB ? s : nB - 1;
        xr[i] = xbase + s * xstride;
    }
    const float *tc = T + 4 * cgi;
    f32x2 a2[4][4];                                          // accumulators as column pairs
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) a2[i][c] = pack2(acc[i][2 * c], acc[i][2 * c + 1]);
    for (int k = kb; k < ke; k += 4) {
        float xv[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 x = *reinterpret_cast<const float4 *>(xr[i] + k);
            xv[i][0] = x.x; xv[i][1] = x.y; xv[i][2] = x.z; xv[i][3] = x.w;
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const float *tr = tc + (k + kk) * N1p;
            const ulonglong2 t0 = *reinterpret_cast<const ulonglong2 *>(tr);        // (t0,t1) (t2,t3)
            const ulonglong2 t1 = *reinterpret_cast<const ulonglong2 *>(tr + half);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const f32x2 x2 = pack2(xv[i][kk], xv[i][kk]);
                ffma2(a2[i][0], x2, t0.x);
                ffma2(a2[i][1], x2, t0.y);
                ffma2(a2[i][2], x2, t1.x);
                ffma2(a2[i][3], x2, t1.y);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) unpack2(a2[i][c], acc[i][2 * c], acc[i][2 * c + 1]);
}

template <int CN1 = 0>
__device__ __forceinline__ void f_store_fast(const Dev &d, float *sm, float (&acc)[4][8]) {
    const int t = threadIdx.x;
    const int N1 = CN1 ? CN1 : d.N1, N1p = CN1 ? CN1 : d.N1p, cg = CN1 ? CN1 / 8 : d.cg;
    const int nB = CN1 ? 32 : d.B, nthreads = CN1 ? 256 : (int)blockDim.x;
    const int per_slice = 8 * cg;
    const int q = t / per_slice, u = t - q * per_slice;
    const int sg = u / cg, cgi = u - sg * cg;
    const int nslices = nthreads / per_slice;
    const int half = N1 >> 1;
    float *Hb = sm + d.off_H;
    float *red = sm + d.off_red;
    const int n = nB * N1p;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int s = sg + 8 * i;
        if (s < nB) {
            float *dst = red + (size_t)q * n + s * N1p + 4 * cgi;
            *reinterpret_cast<float4 *>(dst) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
            *reinterpret_cast<float4 *>(dst + half) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
        }
    }
    __syncthreads();
    for (int i = t; i < n; i += nthreads) {
        float v = 0.f;
        for (int qq = 0; qq < nslices; ++qq) v += red[(size_t)qq * n + i];
        Hb[i] = v;
    }
    __syncthreads();
}

__device__ void g_compute_fast(const Dev &d, const float *sm, float *T, int k0, int cnt) {
    const int t = threadIdx.x;
    const int rgi = t / d.cg, cgi = t - rgi * d.cg;
    const int kl = rgi * 4;
    if (kl >= d.KT || k0 + kl >= d.D) return;
    const int half = d.N1 >> 1;
    const float *xr = sm + k0 + kl;
    const float *dp = sm + d.off_dP + 4 * cgi;
    float acc[4][8];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[j][c] = 0.f;
    for (int s = 0; s < cnt; ++s) {
        const float4 x = *reinterpret_cast<const float4 *>(xr + s * d.Ds);
        const float4 d0 = *reinterpret_cast<const float4 *>(dp + s * d.N1p);
        const float4 d1 = *reinterpret_cast<const float4 *>(dp + s * d.N1p + half);
        const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            acc[j][0] = fmaf(xv[j], d0.x, acc[j][0]);
            acc[j][1] = fmaf(xv[j], d0.y, acc[j][1]);
            acc[j][2] = fmaf(xv[j], d0.z, acc[j][2]);
            acc[j][3] = fmaf(xv[j], d0.w, acc[j][3]);
            acc[j][4] = fmaf(xv[j], d1.x, acc[j][4]);
            acc[j][5] = fmaf(xv[j], d1.y, acc[j][5]);
            acc[j][6] = fmaf(xv[j], d1.z, acc[j][6]);
            acc[j][7] = fmaf(xv[j], d1.w, acc[j][7]);
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (k0 + kl + j < d.D) {
            float *dst = T + (kl + j) * d.N1p + 4 * cgi;
            *reinterpret_cast<float4 *>(dst) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
            *reinterpret_cast<float4 *>(dst + half) = make_float4(acc[j][4], acc[j][5], acc[j][6], acc[j][7]);
        }
    }
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// Hpre = X . W1, W1 streamed from HBM through two tile buffers with cp.async
__device__ void forward_from_global_fast(const Dev &d, float *sm, const float *wE) {
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;
    float *const T0 = sm + d.off_T, *const T1 = sm + d.off_T2;
    auto issue = [&](int t) {
        const int k0 = t * d.KT;
        const int krows = min(d.KT, d.D - k0);
        const int nq = (krows * d.N1) >> 2;
        const float4 *src = reinterpret_cast<const float4 *>(wE + (size_t)k0 * d.N1);
        float4 *dst = reinterpret_cast<float4 *>((t & 1) ? T1 : T0);
        for (int i = threadIdx.x; i < nq; i += blockDim.x) cp_async16(dst + i, src + i);
        cp_async_commit();
    };
    issue(0);
    for (int t = 0; t < d.ntiles; ++t) {
        const int k0 = t * d.KT;
        const int krows = min(d.KT, d.D - k0), krows4 = (krows + 3) & ~3;
        if (t + 1 < d.ntiles) { issue(t + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
        float *T = (t & 1) ? T1 : T0;
        for (int i = krows * d.N1p + threadIdx.x; i < krows4 * d.N1p; i += blockDim.x) T[i] = 0.f;
        __syncthreads();
        f_accumulate_fast(d, sm + k0, d.Ds, T, krows4, acc);
        __syncthreads();
    }
    f_store_fast(d, sm, acc);
}

// ---------------------------------------------------------------------- the tail
// Everything after the first matmul: bias/relu/second layer/softmax-CE (or MSE, or the
// Rosenbrock function).  Fills dPre [B,N1p] and the tail gradient tg; returns mean loss.
// CN1 / CC > 0 fix the hidden width / class count (and B = 32) at compile time.
template <int CN1 = 0, int CC = 0>
__device__ float tail_eval(const Dev &d, float *sm, int cnt) {
    float *Hb = sm + d.off_H, *dP = sm + d.off_dP, *tw = sm + d.off_tw, *tg = sm + d.off_tg;
    float *Zb = sm + d.off_Z, *lb = sm + d.off_lb, *misc = sm + d.off_misc;
    const int tid = threadIdx.x, nt = blockDim.x;
    if (!CN1 && d.kind == B2E_PROBLEM_FUNC) {         // utils/utils_functions.py:4-6
        if (tid == 0) {
            const float x = tw[0], y = tw[1], t = y - x * x;
            misc[0] = 100.f * t * t + (1.f - x) * (1.f - x);
            tg[0] = -400.f * x * t - 2.f * (1.f - x);
            tg[1] = 200.f * t;
        }
        __syncthreads();
        return misc[0];
    }
    const int N1 = CN1 ? CN1 : d.N1, N1p = CN1 ? CN1 : d.N1p, C = CC ? CC : d.C;
    const int nB = CN1 ? 32 : d.B;
    const bool hidden = CN1 ? true : (d.hidden != 0);
    const float *b1 = tw, *W2 = tw + N1, *b2 = tw + N1 + N1 * C;
    float *Z = hidden ? Zb : Hb;
    const int Zs = hidden ? (CC ? ((CC + 3) & ~3) : d.Cp) : N1p;
    float *dZ = hidden ? Zb : dP;                     // dZ overwrites Z when hidden
    if (hidden) {
        for (int i = tid; i < cnt * N1; i += nt) {
            const int s = i / N1, j = i - s * N1;
            const float v = Hb[s * N1p + j] + b1[j];
            Hb[s * N1p + j] = v > 0.f ? v : 0.f;
        }
        __syncthreads();
        for (int i = tid; i < cnt * C; i += nt) {
            const int s = i / C, c = i - s * C;
            float z = b2[c];
            for (int j = 0; j < N1; ++j) z = fmaf(Hb[s * N1p + j], W2[j * C + c], z);
            Z[s * Zs + c] = z;
        }
    } else {
        for (int i = tid; i < cnt * C; i += nt) {
            const int s = i / C, c = i - s * C;
            Z[s * Zs + c] += tw[c];
        }
    }
    __syncthreads();
    for (int s = tid; s < nB; s += nt) {
        float loss = 0.f;
        if (s < cnt) {
            const float *z = Z + s * Zs;
            float *dz = dZ + s * Zs;
            if (d.kind == B2E_PROBLEM_SOFTMAX) {
                const int y = reinterpret_cast<const int *>(sm + d.off_y)[s];
                float m = z[0];
                for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
                float sum = 0.f;
                for (int c = 0; c < C; ++c) sum += expf(z[c] - m);
                const float zy = z[y];
                loss = (m + logf(sum)) - zy;
                const float inv = 1.0f / sum;
                for (int c = 0; c < C; ++c) {
                    const float p = expf(z[c] - m) * inv;
                    dz[c] = p - (c == y ? 1.f : 0.f);
                }
            } else {
                const float *yt = sm + d.off_y + s * C;
                for (int c = 0; c < C; ++c) {
                    const float df = z[c] - yt[c];
                    loss = fmaf(0.5f * df, df, loss);
                    dz[c] = df;
                }
            }
        } else {
            for (int c = 0; c < C; ++c) dZ[s * Zs + c] = 0.f;
        }
        lb[s] = loss;
    }
    __syncthreads();
    if (tid == 0) {
        float l = 0.f;
        for (int s = 0; s < cnt; ++s) l += lb[s];
        misc[0] = l / (float)cnt;
    }
    if (hidden) {
        float *gb1 = tg, *gW2 = tg + N1, *gb2 = tg + N1 + N1 * C;
        for (int i = tid; i < N1 * C; i += nt) {
            const int j = i / C, c = i - j * C;
            float g = 0.f;
            for (int s = 0; s < cnt; ++s) g = fmaf(Hb[s * N1p + j], dZ[s * Zs + c], g);
            gW2[i] = g;
        }
        for (int c = tid; c < C; c += nt) {
            float g = 0.f;
            for (int s = 0; s < cnt; ++s) g += dZ[s * Zs + c];
            gb2[c] = g;
        }
        for (int i = tid; i < nB * N1; i += nt) {
            const int s = i / N1, j = i - s * N1;
            float v = 0.f;
            if (s < cnt && Hb[s * N1p + j] > 0.f) {
                for (int c = 0; c < C; ++c) v = fmaf(dZ[s * Zs + c], W2[j * C + c], v);
            }
            dP[s * N1p + j] = v;
        }
        __syncthreads();
        for (int j = tid; j < N1; j += nt) {
            float g = 0.f;
            for (int s = 0; s < cnt; ++s) g += dP[s * N1p + j];
            gb1[j] = g;
        }
    } else {
        for (int c = tid; c < C; c += nt) {
            float g = 0.f;
            for (int s = 0; s < cnt; ++s) g += dP[s * N1p + c];
            tg[c] = g;
        }
    }
    __syncthreads();
    return misc[0];
}

// ----------------------------------------------------------- elementwise epilogues
struct EpiCtx {
    int e;
    int head_new, nvalid_new;
    float *wE, *gE, *rwE, *rgE;      // this env's slices
    const float *gnewE;              // split path: g_t in HBM (written by the compute kernel)
    const float *obsL;               // [H] clipped adjusted-loss columns
};

constexpr int SPAN_CAP = 160;        // rows a warp's 128-parameter chunk may span when staged by row

__device__ __forceinline__ float ratio_nn(float num, float den) {    // nan_to_num(num / |den|)
    return nan_to_num_f(num / fabsf(den));       // IEEE division: huge / denormal denominators behave as in numpy
}
__device__ __forceinline__ float clip_only_m1(float x) {             // x already nan_to_num'ed
    return fminf(fmaxf(x, -100.0f), 100.0f) - 1.0f;
}
__device__ __forceinline__ int div_small(int n, float inv) {         // exact n / OD for n < 2^15
    return (int)(((float)n + 0.5f) * inv);
}

// Warp writes the observation rows staged for its chunk.
//  dense: rows staged at (row - rlo) * OD (+ phase shift); holes flagged in valid_s; 16-byte
//         stores wherever the four words belong to valid rows;
//  else : rows staged in natural slot order, scattered word by word.
__device__ __forceinline__ void emit_obs(const Dev &d, const StepArgs &a, const EpiCtx &cx,
                                         const float *st, const int *rows_s, const int *valid_s,
                                         bool dense, int rlo, int rhi, int soff) {
    const int lane = threadIdx.x & 31;
    const int OD = d.OD;
    if (rhi < rlo) return;
    if (dense) {
        const int span_words = (rhi - rlo + 1) * OD;
        const size_t g_lo = ((size_t)cx.e * d.P + rlo) * OD;
        const size_t x0 = g_lo - soff;                       // multiple of 4
        const float inv = 1.0f / (float)OD;
        for (int u = lane * 4; u < span_words + soff; u += 128) {
            const int w0 = u - soff;                         // first word of this unit in the span
            const int wa = w0 > 0 ? w0 : 0;
            const int wb = w0 + 3 < span_words ? w0 + 3 : span_words - 1;
            const int ra = div_small(wa, inv), rb = div_small(wb, inv);
            const int va = valid_s[ra], vb = valid_s[rb];
            if (w0 >= 0 && w0 + 3 < span_words && va && vb) {
                *reinterpret_cast<float4 *>(a.obs + x0 + u) = *reinterpret_cast<const float4 *>(st + u);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int w = w0 + j;
                    if (w >= 0 && w < span_words) {
                        const int ok = (w < rb * OD) ? va : vb;
                        if (ok) a.obs[x0 + u + j] = st[u + j];
                    }
                }
            }
        }
    } else {
        float *base = a.obs + (size_t)cx.e * d.P * OD;
        const int q32 = 32 / OD, r32 = 32 - q32 * OD;
        int pl = lane / OD, col = lane - pl * OD;
        for (int wd = lane; wd < 128 * OD; wd += 32) {
            const int row = rows_s[pl];
            if (row >= 0) base[(size_t)row * OD + col] = st[wd];
            pl += q32; col += r32;
            if (col >= OD) { col -= OD; ++pl; }
        }
    }
}

template <int PASS, int HT>
__device__ void epilogue(const Dev &d, const StepArgs &a, float *sm, const EpiCtx &cx,
                         int p_begin, int p_end, float *gsrc, bool tile_mode, int k0,
                         Stats &st) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (p_end <= p_begin) return;
    const int q0 = p_begin >> 2, q1 = (p_end + 3) >> 2;
    const int nchunks = (q1 - q0 + 31) >> 5;
    float *stage = sm + d.off_stage + warp * d.stage_stride;
    int *rows_s = reinterpret_cast<int *>(sm + d.off_rows) + warp * (128 + SPAN_CAP);
    int *valid_s = rows_s + 128;
    const int H = HT > 0 ? HT : d.H, OD = d.OD;
    for (int ch = warp; ch < nchunks; ch += nw) {
        const int p = (q0 + ch * 32 + lane) * 4;
        bool in[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) in[i] = (p + i >= p_begin) && (p + i < p_end);
        const bool any = in[0] || in[1] || in[2] || in[3];
        const bool all = in[0] && in[1] && in[2] && in[3];
        int gi[4];
        if (tile_mode) {
            int k = p / d.N1, c = p - k * d.N1;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                gi[i] = (k - k0) * d.N1p + c;
                if (++c == d.N1) { c = 0; ++k; }
            }
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) gi[i] = p + i - p_begin;
        }
        int rows[4] = {p, p + 1, p + 2, p + 3};
        float g[4] = {0.f, 0.f, 0.f, 0.f};
        if (any) {
            if (d.row_lex && (PASS == PASS_U || PASS == PASS_G)) {
                const int4 r4 = *reinterpret_cast<const int4 *>(d.row_of_param + p);
                rows[0] = r4.x; rows[1] = r4.y; rows[2] = r4.z; rows[3] = r4.w;
            }
            if (PASS == PASS_G && cx.gnewE) {
                const float4 g4 = *reinterpret_cast<const float4 *>(cx.gnewE + p);
                g[0] = g4.x; g[1] = g4.y; g[2] = g4.z; g[3] = g4.w;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (in[i]) g[i] = gsrc[gi[i]];
            }
        }
        if (PASS == PASS_U) {
            if (any) {
                const float4 w4 = *reinterpret_cast<const float4 *>(cx.wE + p);
                const float *act = a.actions + (size_t)cx.e * d.P;
                float av[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) av[i] = in[i] ? act[rows[i]] : 0.f;
                const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
                float wn[4], aw[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float lr = action_to_lr(av[i], d.act_ver);
                    wn[i] = fmaf(-g[i], lr, wv[i]);                 // multioptlrs.py:87
                    aw[i] = ratio_nn(wn[i], wv[i]);                 // utils_env.py:158-159
                    if (in[i]) {
                        st.f[ST_ABSW] += fabsf(wn[i]);
                        st.lr += (double)lr;
                        st.lr2 += (double)lr * (double)lr;
                        gsrc[gi[i]] = wn[i];
                    }
                }
                float *rw = cx.rwE + (size_t)cx.head_new * d.Pp + p;
                if (all) {
                    *reinterpret_cast<float4 *>(cx.wE + p) = make_float4(wn[0], wn[1], wn[2], wn[3]);
                    *reinterpret_cast<float4 *>(rw) = make_float4(aw[0], aw[1], aw[2], aw[3]);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (in[i]) { cx.wE[p + i] = wn[i]; rw[i] = aw[i]; }
                }
            }
        } else if (PASS == PASS_R || PASS == PASS_E || PASS == PASS_S) {
            if (any && PASS == PASS_R && d.g2) {               // raw History keeps the older gradient
                float *g2p = d.g2 + (size_t)cx.e * d.Pp + p;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (in[i]) g2p[i] = cx.gE[p + i];
            }
            if (any) {
                float *dst = (PASS == PASS_R) ? cx.gE + p
                           : (PASS == PASS_S) ? d.gnext + (size_t)cx.e * d.Pp + p
                                              : a.grad_out + (size_t)cx.e * d.P + p;
                if (all && PASS != PASS_E) {
                    *reinterpret_cast<float4 *>(dst) = make_float4(g[0], g[1], g[2], g[3]);
                    st.f[ST_G] += (g[0] + g[1]) + (g[2] + g[3]);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (in[i]) { dst[i] = g[i]; st.f[ST_G] += g[i]; }
                }
            }
        } else {   // PASS_G
            // ---- issue every global load of this quad first
            constexpr int HB = HT > 0 ? HT : 1;
            float4 gp4 = make_float4(1.f, 1.f, 1.f, 1.f);
            float4 rw4[HB], rg4[HB];
            if (HT > 0) {
#pragma unroll
                for (int h = 0; h < HB; ++h) rw4[h] = rg4[h] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (any) {
                gp4 = *reinterpret_cast<const float4 *>(cx.gE + p);
                if (HT > 0) {
#pragma unroll
                    for (int h = 0; h < HB; ++h) {
                        if (h < cx.nvalid_new) {
                            int slot = cx.head_new - h;
                            slot += slot < 0 ? HB : 0;
                            rw4[h] = *reinterpret_cast<const float4 *>(cx.rwE + (size_t)slot * d.Pp + p);
                            if (h > 0)
                                rg4[h] = *reinterpret_cast<const float4 *>(cx.rgE + (size_t)slot * d.Pp + p);
                        }
                    }
                }
            }
            // ---- row span of this warp's chunk
            int rlo = 0x7fffffff, rhi = -1;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (in[i]) { rlo = min(rlo, rows[i]); rhi = max(rhi, rows[i]); }
            rlo = __reduce_min_sync(0xffffffffu, rlo);
            rhi = __reduce_max_sync(0xffffffffu, rhi);
            const bool dense = (rhi - rlo) < SPAN_CAP;
            const int soff = dense ? (int)((((size_t)cx.e * d.P + rlo) * OD) & 3) : 0;
            if (dense) {
                for (int i = lane; i < SPAN_CAP; i += 32) valid_s[i] = 0;
                __syncwarp();
            }
            if (any) {
                const float gp[4] = {gp4.x, gp4.y, gp4.z, gp4.w};
                float ag[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    ag[i] = ratio_nn(g[i], gp[i]);                  // utils_env.py:156-157
                    if (in[i]) {
                        st.f[ST_G] += g[i];
                        st.f[ST_ABSADJG] += fabsf(ag[i]);
                        st.f[ST_GDIFF] += fabsf(g[i] - gp[i]);
                    }
                }
                float *rg = cx.rgE + (size_t)cx.head_new * d.Pp + p;
                const bool keep_g = cx.gnewE == nullptr;   // split path ping-pongs the g buffers
                if (all) {
                    if (keep_g)
                        *reinterpret_cast<float4 *>(cx.gE + p) = make_float4(g[0], g[1], g[2], g[3]);
                    *reinterpret_cast<float4 *>(rg) = make_float4(ag[0], ag[1], ag[2], ag[3]);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (in[i]) { if (keep_g) cx.gE[p + i] = g[i]; rg[i] = ag[i]; }
                }
                // observation rows: [adj_w newest..oldest | adj_L | adj_g newest..oldest]
                float *srow[4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    srow[i] = stage + soff + (dense ? (in[i] ? rows[i] - rlo : 0) : lane * 4 + i) * OD;
                float sabs = 0.f;
                if (HT > 0) {
#pragma unroll
                    for (int h = 0; h < HB; ++h) {
                        const float wv[4] = {rw4[h].x, rw4[h].y, rw4[h].z, rw4[h].w};
                        const float gv[4] = {h ? rg4[h].x : ag[0], h ? rg4[h].y : ag[1],
                                             h ? rg4[h].z : ag[2], h ? rg4[h].w : ag[3]};
                        const float ol = cx.obsL[h];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            if (in[i]) {
                                sabs += fabsf(wv[i]) + fabsf(gv[i]);
                                srow[i][h] = clip_only_m1(wv[i]);
                                srow[i][HB + h] = ol;
                                srow[i][2 * HB + h] = clip_only_m1(gv[i]);
                            }
                        }
                    }
                } else {
                    for (int h = 0; h < H; ++h) {
                        float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f), g4 = w4;
                        if (h < cx.nvalid_new) {
                            int slot = cx.head_new - h;
                            slot += slot < 0 ? H : 0;
                            w4 = *reinterpret_cast<const float4 *>(cx.rwE + (size_t)slot * d.Pp + p);
                            if (h > 0)
                                g4 = *reinterpret_cast<const float4 *>(cx.rgE + (size_t)slot * d.Pp + p);
                            else
                                g4 = make_float4(ag[0], ag[1], ag[2], ag[3]);
                        }
                        const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
                        const float gv[4] = {g4.x, g4.y, g4.z, g4.w};
                        const float ol = cx.obsL[h];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            if (in[i]) {
                                sabs += fabsf(wv[i]) + fabsf(gv[i]);
                                srow[i][h] = clip_only_m1(wv[i]);
                                srow[i][H + h] = ol;
                                srow[i][2 * H + h] = clip_only_m1(gv[i]);
                            }
                        }
                    }
                }
                st.f[ST_STATE] += sabs;
                if (dense) {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (in[i]) valid_s[rows[i] - rlo] = 1;
                }
            }
            if (!dense) {
#pragma unroll
                for (int i = 0; i < 4; ++i) rows_s[lane * 4 + i] = in[i] ? rows[i] : -1;
            }
            __syncwarp();
            emit_obs(d, a, cx, stage, rows_s, valid_s, dense, rlo, rhi, soff);
            __syncwarp();
        }
    }
}


__device__ void load_tail(const Dev &d, float *sm, const float *wE) {
    float *tw = sm + d.off_tw;
    for (int i = threadIdx.x; i < d.tailP; i += blockDim.x) tw[i] = wE[d.P1 + i];
    __syncthreads();
}

// gradient of all parameters at the parameters currently in HBM / tw; PASS_R or PASS_E
template <int PASS, bool BIG>
__device__ float eval_current(const Dev &d, const StepArgs &a, float *sm, const EpiCtx &cx,
                              int cnt, Stats &st) {
    load_tail(d, sm, cx.wE);
    if (d.ntiles) { if (BIG && d.fast) forward_from_global_fast(d, sm, cx.wE); else forward_from_global(d, sm, cx.wE); }
    const float loss = tail_eval(d, sm, cnt);
    float *T = sm + d.off_T;
    epilogue<PASS, 0>(d, a, sm, cx, d.P1, d.P, sm + d.off_tg, false, 0, st);
    for (int t = 0; t < d.ntiles; ++t) {
        const int k0 = t * d.KT;
        if (BIG && d.fast) g_compute_fast(d, sm, T, k0, cnt); else g_compute(d, sm, T, k0, cnt);
        __syncthreads();
        epilogue<PASS, 0>(d, a, sm, cx, k0 * d.N1, min(d.D, k0 + d.KT) * d.N1, T, true, k0, st);
        __syncthreads();
    }
    return loss;
}

__device__ void make_ctx(const Dev &d, int e, EpiCtx &cx) {
    cx.e = e;
    cx.wE = d.w + (size_t)e * d.Pp;
    cx.gE = d.gprev + (size_t)e * d.Pp;
    cx.rwE = d.ringw + (size_t)e * d.H * d.Pp;
    cx.rgE = d.ringg + (size_t)e * d.H * d.Pp;
    cx.gnewE = nullptr;
    cx.head_new = 0;
    cx.nvalid_new = 0;
    cx.obsL = nullptr;
}

// base_reset (multioptlrs.py:66-78) of one env
template <bool BIG>
__device__ void reset_env(const Dev &d, const StepArgs &a, float *sm, int e) {
    EnvScalars *sc = d.sc + e;
    EpiCtx cx;
    make_ctx(d, e, cx);
    if (d.kind != B2E_PROBLEM_FUNC && d.index_mode == B2E_INDEX_INTERNAL) {
        shuffle_order(d, e, sc);                                  // optimize_nn.py:114-120
        if (threadIdx.x == 0) sc->cursor = 0;
        __syncthreads();
    }
    const int *idx; int cnt;
    current_batch(d, a, e, sc, idx, cnt);
    if (d.kind != B2E_PROBLEM_FUNC) load_batch(d, sm, idx, cnt);
    const int episode = sc->episode;
    for (int p = threadIdx.x; p < d.Pp; p += blockDim.x) {
        float v = 0.f;
        if (p < d.P) {
            if (a.init_params) v = a.init_params[(size_t)e * d.P + p];
            else if (d.kind == B2E_PROBLEM_FUNC) v = p == 0 ? -1.9f : 2.0f;   // optimize_function.py:37
            else if (p < d.P1) v = glorot(d.seed, e + d.env_base, episode, p, d.lim1);
            else if (d.hidden && p >= d.P1 + d.N1 && p < d.P1 + d.N1 + d.N1 * d.C)
                v = glorot(d.seed, e + d.env_base, episode, p, d.lim2);
        }
        if (d.w2) d.w2[(size_t)e * d.Pp + p] = cx.wE[p];         // raw History keeps the older weights
        cx.wE[p] = v;
    }
    __syncthreads();
    Stats st;
    zero_stats(st);
    const float loss = eval_current<PASS_R, BIG>(d, a, sm, cx, cnt, st);
    Totals tot;
    block_reduce(st, tot, reinterpret_cast<double *>(sm + d.off_red2));
    const bool lrs = d.env_kind == B2E_ENV_MULTIOPTLRS;
    if (threadIdx.x == 0) {
        // MultiOptLRs clears its raw History (multioptlrs.py:69), MultiOptimize only the adjusted
        // one (multioptimize.py:78-88): there the reset evaluation is one more raw entry
        if (lrs) {
            for (int i = 0; i < RAW_DEPTH; ++i) { sc->raw_loss[i] = 0.f; sc->raw_gsum[i] = 0.0; }
            sc->raw_pos = 0;
        } else {
            sc->raw_pos = (sc->raw_pos + 1) % RAW_DEPTH;
        }
        for (int i = 0; i < B2E_MAX_HISTORY; ++i) sc->adj_loss[i] = 0.f;
        sc->raw_loss[sc->raw_pos] = loss;
        sc->raw_gsum[sc->raw_pos] = tot.v[ST_G];
        sc->loss_prev = loss;
        sc->head = d.H - 1;
        sc->nvalid = 0;
        sc->step = 0;
        sc->episode = episode + 1;
    }
    if (a.obs) {                        // MultiOptLRs: clip(0) - 1 = -1; MultiOptimize: the zero history
        float *o = a.obs + (size_t)e * d.P * d.OD;
        const size_t n = (size_t)d.P * d.OD;
        const float fill = lrs ? -1.0f : 0.0f;
        for (size_t i = threadIdx.x; i < n; i += blockDim.x) o[i] = fill;
    }
    __syncthreads();
}

template <int HT, bool BIG>
__device__ void step_env(const Dev &d, const StepArgs &a, float *sm, int e) {
    EnvScalars *sc = d.sc + e;
    EpiCtx cx;
    make_ctx(d, e, cx);
    float *misc = sm + d.off_misc;
    float *T = sm + d.off_T;
    const int *idx; int cnt;
    current_batch(d, a, e, sc, idx, cnt);
    if (d.kind != B2E_PROBLEM_FUNC) load_batch(d, sm, idx, cnt);
    const int head_new = (sc->head + 1) % d.H;
    const int nvalid_new = min(sc->nvalid + 1, d.H);
    cx.head_new = head_new;
    cx.nvalid_new = nvalid_new;
    cx.obsL = misc + 8;
    Stats st;
    zero_stats(st);

    // ---- gradient at w_{t-1}, update, forward at w_t (fused per tile)
    load_tail(d, sm, cx.wE);
    if (d.ntiles) { if (BIG && d.fast) forward_from_global_fast(d, sm, cx.wE); else forward_from_global(d, sm, cx.wE); }
    tail_eval(d, sm, cnt);
    epilogue<PASS_U, 0>(d, a, sm, cx, d.P1, d.P, sm + d.off_tg, false, 0, st);
    __syncthreads();
    {   // tail: tg now holds w_t of the tail; make it the live tail parameters
        float *tw = sm + d.off_tw, *tg = sm + d.off_tg;
        for (int i = threadIdx.x; i < d.tailP; i += blockDim.x) tw[i] = tg[i];
    }
    float acc[MAXI][8];
    zero_acc(acc);
    for (int t = 0; t < d.ntiles; ++t) {
        const int k0 = t * d.KT;
        const int krows = min(d.KT, d.D - k0), krows4 = (krows + 3) & ~3;
        if (BIG && d.fast) g_compute_fast(d, sm, T, k0, cnt); else g_compute(d, sm, T, k0, cnt);
        __syncthreads();
        epilogue<PASS_U, 0>(d, a, sm, cx, k0 * d.N1, (k0 + krows) * d.N1, T, true, k0, st);
        for (int i = krows * d.N1p + threadIdx.x; i < krows4 * d.N1p; i += blockDim.x) T[i] = 0.f;
        if (d.N1p != d.N1)
            for (int i = threadIdx.x; i < krows * (d.N1p - d.N1); i += blockDim.x) {
                const int k = i / (d.N1p - d.N1), c = d.N1 + i - k * (d.N1p - d.N1);
                T[k * d.N1p + c] = 0.f;
            }
        __syncthreads();
        if (BIG && d.fast) f_accumulate_fast(d, sm + k0, d.Ds, T, krows4, acc); else f_accumulate(d, sm, T, k0, krows4, acc);
        __syncthreads();
    }
    if (d.ntiles) { if (BIG && d.fast) f_store_fast(d, sm, acc); else f_store(d, sm, acc); }
    __syncthreads();

    // ---- gradient and loss at w_t
    const float loss = tail_eval(d, sm, cnt);
    if (threadIdx.x == 0) {
        const double adjl = nan_to_num_d((double)loss / fabs((double)sc->loss_prev));
        reinterpret_cast<double *>(misc + 2)[0] = adjl;          // misc[2..3]
        float *obsL = misc + 8;
        for (int h = 0; h < d.H; ++h) {
            float v = 0.f;
            if (h == 0) v = (float)adjl;
            else if (h < nvalid_new) {
                int slot = head_new - h;
                slot += slot < 0 ? d.H : 0;
                v = sc->adj_loss[slot];
            }
            obsL[h] = clip_m1(v);
            misc[8 + B2E_MAX_HISTORY + h] = fabsf(v);
        }
    }
    __syncthreads();
    if (d.split) {      // g_t goes to HBM; the observation kernel takes it from there
        epilogue<PASS_S, 0>(d, a, sm, cx, d.P1, d.P, sm + d.off_tg, false, 0, st);
        for (int t = 0; t < d.ntiles; ++t) {
            const int k0 = t * d.KT;
            if (BIG && d.fast) g_compute_fast(d, sm, T, k0, cnt); else g_compute(d, sm, T, k0, cnt);
            __syncthreads();
            epilogue<PASS_S, 0>(d, a, sm, cx, k0 * d.N1, min(d.D, k0 + d.KT) * d.N1, T, true, k0, st);
            __syncthreads();
        }
    } else {
        epilogue<PASS_G, HT>(d, a, sm, cx, d.P1, d.P, sm + d.off_tg, false, 0, st);
        for (int t = 0; t < d.ntiles; ++t) {
            const int k0 = t * d.KT;
            if (BIG && d.fast) g_compute_fast(d, sm, T, k0, cnt); else g_compute(d, sm, T, k0, cnt);
            __syncthreads();
            epilogue<PASS_G, HT>(d, a, sm, cx, k0 * d.N1, min(d.D, k0 + d.KT) * d.N1, T, true, k0, st);
            __syncthreads();
        }
    }
    Totals tot;
    block_reduce(st, tot, reinterpret_cast<double *>(sm + d.off_red2));

    // ---- scalars: reward, done, info, history bookkeeping (thread 0)
    bool done = false;
    if (threadIdx.x == 0) {
        const double adjl = reinterpret_cast<double *>(misc + 2)[0];
        const double L = (double)loss;
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
        reward = fmin(fmax(reward, -100.0), 100.0);                // multioptlrs.py:103
        const int step = sc->step + 1;                             // baseenvironment.py:37
        done = step >= d.max_batches;
        if (!done && loss > 1e4f) {                                // multioptlrs.py:105-107
            done = true;
            reward -= (double)(d.max_batches - step);
        }
        const int rp = (sc->raw_pos + 1) % RAW_DEPTH;
        sc->raw_pos = rp;
        sc->raw_loss[rp] = loss;
        sc->raw_gsum[rp] = tot.v[ST_G];
        sc->loss_prev = loss;
        sc->adj_loss[head_new] = (float)adjl;
        sc->head = head_new;
        sc->nvalid = nvalid_new;
        sc->step = step;
        double gsum = 0.0, lsum = 0.0, labs = 0.0;
        for (int i = 0; i < RAW_DEPTH; ++i) { gsum += sc->raw_gsum[i]; lsum += (double)sc->raw_loss[i]; }
        for (int h = 0; h < d.H; ++h) labs += (double)misc[8 + B2E_MAX_HISTORY + h];
        const double P = (double)d.P;
        const double lr_mean = tot.v[ST_LR] / P;
        double lr_var = tot.v[ST_LR2] / P - lr_mean * lr_mean;
        lr_var = lr_var > 0.0 ? lr_var : 0.0;
        const double ssum = tot.v[ST_STATE] + P * labs;
        double *info = a.info + (size_t)e * B2E_INFO_STRIDE;
        info[0] = done ? L : nan("");                              // multioptlrs.py:108-110
        info[1] = L;
        info[2] = tot.v[ST_ABSW] / P;
        info[3] = tot.v[ST_ABSW];
        info[4] = lr_mean;
        info[5] = sqrt(lr_var);
        info[6] = ssum / (P * (double)d.OD);
        info[7] = ssum;
        info[8] = gsum / (RAW_DEPTH * P);
        info[9] = gsum;
        info[10] = lsum / RAW_DEPTH;
        info[11] = adjl;
        info[12] = tot.v[ST_ABSADJG] / P;
        info[13] = tot.v[ST_GDIFF] / P;
        info[14] = reward;                                         // baseenvironment.py:40
        info[15] = (double)step;
        a.reward[e] = (float)reward;
        a.done[e] = done ? 1 : 0;
        misc[1] = done ? 1.f : 0.f;
        if (d.kind != B2E_PROBLEM_FUNC && d.index_mode == B2E_INDEX_INTERNAL) {
            const int cur = sc->cursor + 1;                        // optimize_nn.py:102-112
            misc[4] = (cur * d.B >= d.N) ? 1.f : 0.f;
            sc->cursor = (cur * d.B >= d.N) ? 0 : cur;
        } else {
            misc[4] = 0.f;
        }
    }
    __syncthreads();
    const bool wrap = misc[4] != 0.f;
    done = misc[1] != 0.f;
    __syncthreads();
    if (wrap) shuffle_order(d, e, sc);
    if (done && d.auto_reset && !d.split) reset_env<BIG>(d, a, sm, e);
}


// pipeline stage "evaluate at w_t" for problems the eval kernel does not cover: g_t to HBM,
// then the step's scalars
template <bool BIG>
__device__ void eval_step_env(const Dev &d, const StepArgs &a, float *sm, int e) {
    EnvScalars *sc = d.sc + e;
    EpiCtx cx;
    make_ctx(d, e, cx);
    const int *idx; int cnt;
    current_batch(d, a, e, sc, idx, cnt);
    if (d.kind != B2E_PROBLEM_FUNC) load_batch(d, sm, idx, cnt);
    Stats st;
    zero_stats(st);
    const float loss = eval_current<PASS_S, BIG>(d, a, sm, cx, cnt, st);
    Totals tot;
    block_reduce(st, tot, reinterpret_cast<double *>(sm + d.off_red2));
    float *misc = sm + d.off_misc;
    if (threadIdx.x == 0) step_scalars(d, a, sc, e, loss, tot.v[ST_G], misc);
    __syncthreads();
    const bool wrap = misc[4] != 0.f;
    __syncthreads();
    if (wrap) shuffle_order(d, e, sc);
}

template <bool BIG>
__device__ void eval_env(const Dev &d, const StepArgs &a, float *sm, int e) {
    EnvScalars *sc = d.sc + e;
    EpiCtx cx;
    make_ctx(d, e, cx);
    const int *idx; int cnt;
    current_batch(d, a, e, sc, idx, cnt);
    if (d.kind != B2E_PROBLEM_FUNC) load_batch(d, sm, idx, cnt);
    Stats st;
    zero_stats(st);
    const float loss = eval_current<PASS_E, BIG>(d, a, sm, cx, cnt, st);
    if (threadIdx.x == 0) a.loss_out[e] = loss;
    __syncthreads();
}

template <int HT, bool BIG>
__global__ void __launch_bounds__(256, BIG ? 1 : 2) optenv_kernel(const __grid_constant__ Dev d,
                                                     const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int e_end = a.e_begin + a.e_count;
    for (int e = a.e_begin + blockIdx.x; e < e_end; e += gridDim.x) {
        if (a.mode == MODE_STEP) {
            step_env<HT, BIG>(d, a, sm, e);
        } else if (a.mode == MODE_RESET) {
            if (a.mask == nullptr || a.mask[e]) reset_env<BIG>(d, a, sm, e);
        } else if (a.mode == MODE_EVAL_STEP) {
            eval_step_env<BIG>(d, a, sm, e);
        } else {
            eval_env<BIG>(d, a, sm, e);
        }
        __syncthreads();
    }
}

// ------------------------------------------------- split path: observation kernel
// Row-space streaming kernel: lane = one agent row (= one parameter, through the row
// table).  Reads g_t, g_{t-1} and the ratio rings of that parameter, appends the new
// gradient ratio, builds the observation row in shared memory and the warp writes its 32
// rows as one contiguous block.  Consecutive rows are (runs of) consecutive parameters in
// lexicographic order, so the 4-byte gathers stay sector efficient.
constexpr int OBS_WARPS = 8;
constexpr int OBS_ITERS = 8;
constexpr int SEG_ROWS = OBS_WARPS * OBS_ITERS * 32;

template <int HT>
__global__ void __launch_bounds__(OBS_WARPS * 32) obs_kernel(const __grid_constant__ Dev d,
                                                             const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    __shared__ double red[OBS_WARPS * 4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int H = HT > 0 ? HT : d.H, OD = d.OD;
    constexpr int HB = HT > 0 ? HT : 1;
    float *obsL_s = sm;                                       // [B2E_MAX_HISTORY]
    float *stage = sm + B2E_MAX_HISTORY + warp * (32 * OD + 8);
    const int nitems = a.e_count * d.nseg;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int eo = item / d.nseg;
        const int e = a.e_begin + eo;
        const int seg = item - eo * d.nseg;
        const EnvScalars *sc = d.sc + e;
        const int head = sc->head, nvalid = sc->nvalid;      // already advanced by the second eval
        __syncthreads();
        if (threadIdx.x < H) {
            const int h = threadIdx.x;
            float v = 0.f;
            if (h < nvalid) {
                int slot = head - h;
                slot += slot < 0 ? H : 0;
                v = sc->adj_loss[slot];
            }
            obsL_s[h] = clip_m1(v);
        }
        __syncthreads();
        const float *gnew = d.gnext + (size_t)e * d.Pp;
        const float *gold = d.gprev + (size_t)e * d.Pp;
        const float *rw = d.ringw + (size_t)e * H * d.Pp;
        float *rg = d.ringg + (size_t)e * H * d.Pp;
        float *rg_new = rg + (size_t)head * d.Pp;
        float *obs_env = a.obs + (size_t)e * d.P * OD;
        // per-history-slot base pointers and loss columns (uniform across the CTA)
        const float *rwh[HB], *rgh[HB];
        float ol[HB];
        if (HT > 0) {
#pragma unroll
            for (int h = 0; h < HB; ++h) {
                int slot = head - h;
                slot += slot < 0 ? HB : 0;
                rwh[h] = rw + (size_t)slot * d.Pp;
                rgh[h] = rg + (size_t)slot * d.Pp;
                ol[h] = obsL_s[h];
            }
        }
        float s_absadjg = 0.f, s_gdiff = 0.f, s_state = 0.f;
        for (int it = 0; it < OBS_ITERS; ++it) {
            const int rbase = seg * SEG_ROWS + (it * OBS_WARPS + warp) * 32;
            if (rbase >= d.P) break;
            const int r = rbase + lane;
            const bool ok = r < d.P;
            const int p = ok ? (d.row_lex ? d.param_of_row[r] : r) : 0;
            const float g = gnew[p], gp = gold[p];
            float wv[HB], gv[HB];
            if (HT > 0) {
#pragma unroll
                for (int h = 0; h < HB; ++h) {
                    wv[h] = 0.f; gv[h] = 0.f;
                    if (h < nvalid) {
                        wv[h] = rwh[h][p];
                        if (h > 0) gv[h] = rgh[h][p];
                    }
                }
            }
            // stage so that shared and global memory share their 16-byte phase
            const unsigned w_lo = (unsigned)rbase * OD;           // word offset inside this env's block
            const unsigned sh = (unsigned)((((size_t)e * d.P * OD) + w_lo) & 3);
            float *srow = stage + sh + lane * OD;
            const float ag = ratio_nn(g, gp);                     // utils_env.py:156-157
            if (ok) {
                rg_new[p] = ag;
                s_absadjg += fabsf(ag);
                s_gdiff += fabsf(g - gp);
            }
            if (HT > 0) {
                gv[0] = ag;
#pragma unroll
                for (int h = 0; h < HB; ++h) {
                    if (ok) s_state += fabsf(wv[h]) + fabsf(gv[h]);
                    srow[h] = clip_only_m1(wv[h]);
                    srow[HB + h] = ol[h];
                    srow[2 * HB + h] = clip_only_m1(gv[h]);
                }
            } else {
                for (int h = 0; h < H; ++h) {
                    float w1 = 0.f, g1 = 0.f;
                    if (h < nvalid) {
                        int slot = head - h;
                        slot += slot < 0 ? H : 0;
                        w1 = rw[(size_t)slot * d.Pp + p];
                        g1 = h > 0 ? rg[(size_t)slot * d.Pp + p] : ag;
                    }
                    if (ok) s_state += fabsf(w1) + fabsf(g1);
                    srow[h] = clip_only_m1(w1);
                    srow[H + h] = obsL_s[h];
                    srow[2 * H + h] = clip_only_m1(g1);
                }
            }
            __syncwarp();
            // contiguous write of this warp's rows: words [0, nw) of `dst`, stage word i at stage[sh + i]
            const unsigned nw = (unsigned)min(32, d.P - rbase) * OD;
            float *dst = obs_env + w_lo;
            const float *src = stage + sh;
            const unsigned head_w = min(nw, (4u - sh) & 3u);      // scalars up to the first aligned word
            const unsigned body_e = head_w + ((nw - head_w) & ~3u);
            if (lane < head_w) dst[lane] = src[lane];
            for (unsigned i = head_w + lane * 4; i < body_e; i += 128)
                *reinterpret_cast<float4 *>(dst + i) = *reinterpret_cast<const float4 *>(src + i);
            if (body_e + lane < nw) dst[body_e + lane] = src[body_e + lane];
            __syncwarp();
        }
        // per-segment partials (deterministic: fixed order inside the CTA, summed per env later)
        const double v0 = warp_sum((double)s_absadjg), v1 = warp_sum((double)s_gdiff);
        const double v2 = warp_sum((double)s_state);
        if (lane == 0) { red[warp * 4] = v0; red[warp * 4 + 1] = v1; red[warp * 4 + 2] = v2; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double *out = d.part + ((size_t)e * d.nseg + seg) * 4;
            for (int i = 0; i < 3; ++i) {
                double v = 0.0;
                for (int w = 0; w < OBS_WARPS; ++w) v += red[w * 4 + i];
                out[i] = v;
            }
        }
    }
}

// ------------------------------------------- observation kernel, asynchronous gathers
// Same work as obs_kernel, organised for memory-level parallelism: a WARP owns 32 units of
// 32 consecutive agent rows of one env and runs a private S-stage pipeline over them.  The
// 2H+1 four-byte gathers of a row (g_t, g_{t-1}, H adjusted-weight slots, H-1 adjusted-gradient
// slots) are cp.async copies into the warp's shared-memory stage, so S units of loads are in
// flight per warp without holding registers or scoreboard slots; no CTA-wide barrier exists.
// The 32 finished rows (32 * 3H words, contiguous in HBM) leave either through 16-byte stores
// or as one cp.async.bulk shared->global copy issued by lane 0.
constexpr int O2_WARPS = 4;
constexpr int O2_UNITS = 32;

__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void bulk_store(void *gmem_dst, const void *smem_src, unsigned bytes) {
    const unsigned src = (unsigned)__cvta_generic_to_shared(smem_src);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n"
                 ::"l"(gmem_dst), "r"(src), "r"(bytes) : "memory");
}

template <int H, int S, bool BULK>
__global__ void __launch_bounds__(O2_WARPS * 32) obs_kernel2(const __grid_constant__ Dev d,
                                                             const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    constexpr int OD = 3 * H, NPL = 2 * H + 1, NPL1 = NPL + 1;   // + the row's parameter index
    constexpr int STG = 32 * OD + 8;
    constexpr int PER_WARP = S * NPL1 * 32 + (BULK ? 2 : 1) * STG;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item = blockIdx.x * O2_WARPS + warp;
    if (item >= a.e_count * d.nseg) return;                  // nseg = 32-unit chunks per env
    float *gat = sm + warp * PER_WARP;
    float *stage0 = gat + S * NPL1 * 32;
    const int eo = item / d.nseg, chunk = item - eo * d.nseg;
    const int e = a.e_begin + eo;
    const EnvScalars *sc = d.sc + e;
    const int head = sc->head, nvalid = sc->nvalid;          // already advanced by the second eval
    float ol[H];
    const float *src[NPL];
    src[0] = d.gnext + (size_t)e * d.Pp;
    src[1] = d.gprev + (size_t)e * d.Pp;
#pragma unroll
    for (int h = 0; h < H; ++h) {
        int slot = head - h;
        slot += slot < 0 ? H : 0;
        ol[h] = clip_m1(h < nvalid ? sc->adj_loss[slot] : 0.f);
        src[2 + h] = d.ringw + ((size_t)e * H + slot) * d.Pp;
        if (h > 0) src[2 + H + h - 1] = d.ringg + ((size_t)e * H + slot) * d.Pp;
    }
    float *rg_new = d.ringg + ((size_t)e * H + head) * d.Pp;
    float *obs_env = a.obs + (size_t)e * d.P * OD;
    const int nblk = (d.P + 31) >> 5;
    const int u0 = chunk * d.obs_units;
    const int nu = min(d.obs_units, nblk - u0);
    auto row_param = [&](int it) -> int {
        const int r = (u0 + it) * 32 + lane;
        return r < d.P ? (d.row_lex ? d.param_of_row[r] : r) : 0;
    };
    auto issue = [&](int it, int p) {
        float *dst = gat + (it % S) * (NPL1 * 32) + lane;
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int h = k < 2 ? 0 : (k < 2 + H ? k - 2 : k - 1 - H);
            if (h < nvalid) cp_async4(dst + k * 32, src[k] + p);
        }
        reinterpret_cast<int *>(dst)[NPL * 32] = p;
    };
#pragma unroll
    for (int it = 0; it < S; ++it) {
        if (it < nu) issue(it, row_param(it));
        cp_async_commit();
    }
    int p_next = S < nu ? row_param(S) : 0;
    float s_absadjg = 0.f, s_gdiff = 0.f, s_state = 0.f;
    for (int it = 0; it < nu; ++it) {
        cp_async_wait<S - 1>();
        const float *gs = gat + (it % S) * (NPL1 * 32) + lane;
        const float g = gs[0], gp = gs[32];
        const int p = reinterpret_cast<const int *>(gs)[NPL * 32];
        float wv[H], gv[H];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            wv[h] = h < nvalid ? gs[(2 + h) * 32] : 0.f;
            gv[h] = (h > 0 && h < nvalid) ? gs[(2 + H + h - 1) * 32] : 0.f;
        }
        if (it + S < nu) issue(it + S, p_next);              // refill the stage just consumed
        cp_async_commit();
        if (it + S + 1 < nu) p_next = row_param(it + S + 1);
        const int rbase = (u0 + it) * 32;
        const bool ok = rbase + lane < d.P;
        const float ag = ratio_nn(g, gp);                    // utils_env.py:156-157
        if (ok) {
            rg_new[p] = ag;
            s_absadjg += fabsf(ag);
            s_gdiff += fabsf(g - gp);
        }
        gv[0] = ag;
        // stage so that shared and global memory share their 16-byte phase
        const unsigned w_lo = (unsigned)rbase * OD;
        const unsigned sh = (unsigned)((((size_t)e * d.P * OD) + w_lo) & 3);
        float *stage = stage0 + (BULK ? (it & 1) * STG : 0);
        if (BULK) {
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory");
            __syncwarp();
        }
        float *srow = stage + sh + lane * OD;
#pragma unroll
        for (int h = 0; h < H; ++h) {
            if (ok) s_state += fabsf(wv[h]) + fabsf(gv[h]);
            srow[h] = clip_only_m1(wv[h]);
            srow[H + h] = ol[h];
            srow[2 * H + h] = clip_only_m1(gv[h]);
        }
        if (BULK) asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        const unsigned nw = (unsigned)min(32, d.P - rbase) * OD;
        float *dst = obs_env + w_lo;
        const float *srcw = stage + sh;
        const unsigned head_w = min(nw, (4u - sh) & 3u);     // scalars up to the first aligned word
        const unsigned body_e = head_w + ((nw - head_w) & ~3u);
        if (lane < head_w) dst[lane] = srcw[lane];
        if (BULK) {
            if (lane == 0) {
                if (body_e > head_w) bulk_store(dst + head_w, srcw + head_w, (body_e - head_w) * 4u);
                asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
            }
        } else {
            for (unsigned i = head_w + lane * 4; i < body_e; i += 128)
                *reinterpret_cast<float4 *>(dst + i) = *reinterpret_cast<const float4 *>(srcw + i);
        }
        if (body_e + lane < nw) dst[body_e + lane] = srcw[body_e + lane];
        if (!BULK) __syncwarp();
    }
    if (BULK && lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
    const double v0 = warp_sum((double)s_absadjg), v1 = warp_sum((double)s_gdiff);
    const double v2 = warp_sum((double)s_state);
    if (lane == 0) {
        double *out = d.part + ((size_t)e * d.nseg + chunk) * 4;
        out[0] = v0; out[1] = v1; out[2] = v2;
    }
}

// ------------------------------------------- observation kernel, register-batched gathers
// As obs_kernel2, but the loads stay in registers: every lane issues the 2H+1 gathers of R
// rows (R units of 32 rows per warp iteration) back to back before the first use, so a warp
// has R*(2H+1) loads in flight at the LSU cost of plain LDG.
template <int H, int R, bool BULK>
__global__ void __launch_bounds__(O2_WARPS * 32) obs_kernel3(const __grid_constant__ Dev d,
                                                             const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    constexpr int OD = 3 * H;
    constexpr int STG = 32 * OD + 8;
    constexpr int PER_WARP = (BULK ? 2 : 1) * STG;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item = blockIdx.x * O2_WARPS + warp;
    if (item >= a.e_count * d.nseg) return;
    float *stage0 = sm + warp * PER_WARP;
    const int eo = item / d.nseg, chunk = item - eo * d.nseg;
    const int e = a.e_begin + eo;
    const EnvScalars *sc = d.sc + e;
    const int head = sc->head, nvalid = sc->nvalid;
    float ol[H];
    const float *rwh[H], *rgh[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        int slot = head - h;
        slot += slot < 0 ? H : 0;
        ol[h] = clip_m1(h < nvalid ? sc->adj_loss[slot] : 0.f);
        rwh[h] = d.ringw + ((size_t)e * H + slot) * d.Pp;
        rgh[h] = d.ringg + ((size_t)e * H + slot) * d.Pp;
    }
    const float *gnew = d.gnext + (size_t)e * d.Pp;
    const float *gold = d.gprev + (size_t)e * d.Pp;
    float *rg_new = d.ringg + ((size_t)e * H + head) * d.Pp;
    float *obs_env = a.obs + (size_t)e * d.P * OD;
    const int nblk = (d.P + 31) >> 5;
    const int u0 = chunk * d.obs_units;
    const int nu = min(d.obs_units, nblk - u0);
    float s_absadjg = 0.f, s_gdiff = 0.f, s_state = 0.f;
    int pn[R];
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const int r = (u0 + j) * 32 + lane;
        pn[j] = (j < nu && r < d.P) ? (d.row_lex ? d.param_of_row[r] : r) : 0;
    }
    int nstore = 0;
    for (int it = 0; it < nu; it += R) {
        int p[R];
        float g[R], gp[R], wv[R][H], gv[R][H];
#pragma unroll
        for (int j = 0; j < R; ++j) {
            p[j] = pn[j];
            g[j] = gnew[p[j]];
            gp[j] = gold[p[j]];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                wv[j][h] = h < nvalid ? rwh[h][p[j]] : 0.f;
                gv[j][h] = (h > 0 && h < nvalid) ? rgh[h][p[j]] : 0.f;
            }
        }
#pragma unroll
        for (int j = 0; j < R; ++j) {                        // row indices of the next iteration
            const int r = (u0 + it + R + j) * 32 + lane;
            pn[j] = (it + R + j < nu && r < d.P) ? (d.row_lex ? d.param_of_row[r] : r) : 0;
        }
#pragma unroll
        for (int j = 0; j < R; ++j) {
            if (it + j >= nu) break;
            const int rbase = (u0 + it + j) * 32;
            const bool ok = rbase + lane < d.P;
            const float ag = ratio_nn(g[j], gp[j]);          // utils_env.py:156-157
            if (ok) {
                rg_new[p[j]] = ag;
                s_absadjg += fabsf(ag);
                s_gdiff += fabsf(g[j] - gp[j]);
            }
            gv[j][0] = ag;
            const unsigned w_lo = (unsigned)rbase * OD;
            const unsigned sh = (unsigned)((((size_t)e * d.P * OD) + w_lo) & 3);
            float *stage = stage0 + (BULK ? (nstore & 1) * STG : 0);
            ++nstore;
            if (BULK) {
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory");
                __syncwarp();
            }
            float *srow = stage + sh + lane * OD;
#pragma unroll
            for (int h = 0; h < H; ++h) {
                if (ok) s_state += fabsf(wv[j][h]) + fabsf(gv[j][h]);
                srow[h] = clip_only_m1(wv[j][h]);
                srow[H + h] = ol[h];
                srow[2 * H + h] = clip_only_m1(gv[j][h]);
            }
            if (BULK) asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            __syncwarp();
            const unsigned nw = (unsigned)min(32, d.P - rbase) * OD;
            float *dst = obs_env + w_lo;
            const float *srcw = stage + sh;
            const unsigned head_w = min(nw, (4u - sh) & 3u);
            const unsigned body_e = head_w + ((nw - head_w) & ~3u);
            if (lane < head_w) dst[lane] = srcw[lane];
            if (BULK) {
                if (lane == 0) {
                    if (body_e > head_w) bulk_store(dst + head_w, srcw + head_w, (body_e - head_w) * 4u);
                    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
                }
            } else {
                for (unsigned i = head_w + lane * 4; i < body_e; i += 128)
                    *reinterpret_cast<float4 *>(dst + i) = *reinterpret_cast<const float4 *>(srcw + i);
            }
            if (body_e + lane < nw) dst[body_e + lane] = srcw[body_e + lane];
            if (!BULK) __syncwarp();
        }
    }
    if (BULK && lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
    const double v0 = warp_sum((double)s_absadjg), v1 = warp_sum((double)s_gdiff);
    const double v2 = warp_sum((double)s_state);
    if (lane == 0) {
        double *out = d.part + ((size_t)e * d.nseg + chunk) * 4;
        out[0] = v0; out[1] = v1; out[2] = v2;
    }
}

// =========================================================================================
// Large problems: the step is a pipeline of four kernels on the caller's stream
//   eval_kernel<false> : g0 = grad(batch, w_{t-1})                      (2 CTAs/SM, FFMA bound)
//   update_kernel      : w_t = w_{t-1} - g0*lr(a); adj_w ring; stats    (streaming, HBM bound)
//   eval_kernel<true>  : g_t, L_t = grad/loss(batch, w_t); scalars      (2 CTAs/SM, FFMA bound)
//   obs_kernel         : adj_g ring + observation rows + stats          (streaming, HBM bound)
// The eval kernel streams BOTH operands through double-buffered shared-memory tiles
// (cp.async), so it needs ~110 KB per CTA and is insensitive to HBM latency.
// =========================================================================================
// CN1 / CKT > 0: layer width and tile length fixed at compile time (config 4: 64 / 112), which
// turns a quarter of the kernel's instructions (address arithmetic on runtime strides) into
// immediates; 0 = read them from the Dev.
template <bool SECOND, int CN1 = 0, int CKT = 0>
__global__ void __launch_bounds__(256, 2) eval_kernel(const __grid_constant__ Dev d,
                                                      const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x;
    float *const X0 = sm + d.ev_X0, *const X1 = sm + d.ev_X1;
    float *const W0 = sm + d.ev_W0, *const W1 = sm + d.ev_W1;
    float *misc = sm + d.off_misc;
    const int cN1 = CN1 ? CN1 : d.N1, cN1p = CN1 ? CN1 : d.N1p, cKT = CKT ? CKT : d.KT;
    const int XS = CKT ? (((CKT >> 2) & 1) ? CKT : CKT + 4) : d.ev_XS;
    const int e_end = a.e_begin + a.e_count;
    for (int e = a.e_begin + blockIdx.x; e < e_end; e += gridDim.x) {
        EnvScalars *sc = d.sc + e;
        const float *wE = d.w + (size_t)e * d.Pp;
        float *gout = d.gnext + (size_t)e * d.Pp;
        const int *idx; int cnt;
        current_batch(d, a, e, sc, idx, cnt);
        int *idx_s = reinterpret_cast<int *>(sm + d.off_idx);
        int *ys = reinterpret_cast<int *>(sm + d.off_y);
        for (int r = tid; r < d.B; r += blockDim.x) {
            const int row = (r < cnt) ? idx[r] : 0;
            idx_s[r] = row;
            if (d.kind == B2E_PROBLEM_SOFTMAX) ys[r] = (r < cnt) ? d.labels[row] : 0;
        }
        if (d.kind == B2E_PROBLEM_LINREG) {
            float *yt = sm + d.off_y;
            for (int i = tid; i < d.B * d.C; i += blockDim.x) {
                const int r = i / d.C, c = i - r * d.C;
                yt[i] = (r < cnt) ? d.targets[(size_t)idx[r] * d.C + c] : 0.f;
            }
        }
        for (int i = tid; i < 2 * d.B * XS; i += blockDim.x) X0[i] = 0.f;    // X0, X1 contiguous
        for (int i = tid; i < d.tailP; i += blockDim.x) sm[d.off_tw + i] = wE[d.P1 + i];
        __syncthreads();

        auto issue_x = [&](int t) {
            const int k0 = t * cKT;
            // 16-byte chunks per row; the fixed-shape instantiation is only used when CKT divides D
            const int kq = CKT ? CKT / 4 : (min(cKT, d.Dp - k0)) >> 2;
            float *dst = (t & 1) ? X1 : X0;
            for (int i = tid; i < cnt * kq; i += blockDim.x) {
                const int r = i / kq, c = i - r * kq;
                cp_async16(dst + r * XS + 4 * c, d.X + (size_t)idx_s[r] * d.Dp + k0 + 4 * c);
            }
        };
        auto issue_w = [&](int t) {
            const int k0 = t * cKT;
            const int nq = (CKT && CN1) ? CKT * CN1 / 4 : (min(cKT, d.D - k0) * cN1) >> 2;
            const float4 *src = reinterpret_cast<const float4 *>(wE + (size_t)k0 * cN1);
            float4 *dst = reinterpret_cast<float4 *>((t & 1) ? W1 : W0);
            for (int i = tid; i < nq; i += blockDim.x) cp_async16(dst + i, src + i);
        };

        // ---- forward: Hpre = X . W1
        float acc[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;
        issue_x(0); issue_w(0); cp_async_commit();
        for (int t = 0; t < d.ntiles; ++t) {
            const int krows = min(cKT, d.D - t * cKT), krows4 = (krows + 3) & ~3;
            if (t + 1 < d.ntiles) { issue_x(t + 1); issue_w(t + 1); cp_async_commit(); cp_async_wait<1>(); }
            else cp_async_wait<0>();
            float *T = (t & 1) ? W1 : W0;
            for (int i = krows * cN1p + tid; i < krows4 * cN1p; i += blockDim.x) T[i] = 0.f;
            __syncthreads();
            f_accumulate_fast<CN1>(d, (t & 1) ? X1 : X0, XS, T, krows4, acc);
            __syncthreads();
        }
        f_store_fast<CN1>(d, sm, acc);                       // partials reduced through the W tiles
        // the first X tile of the backward pass can already travel
        issue_x(0); cp_async_commit();
        const float loss = (CN1 == 64 && d.C == 10) ? tail_eval<CN1, 10>(d, sm, cnt) : tail_eval(d, sm, cnt);

        // ---- backward: tail gradient, then g = X^T . dPre tile by tile, straight to HBM
        float gsum = 0.f;
        for (int i = tid; i < d.tailP; i += blockDim.x) {
            const float g = sm[d.off_tg + i];
            gout[d.P1 + i] = g;
            gsum += g;
        }
        const int ccg = cN1 >> 3;
        const int rgi = tid / ccg, cgi = tid - rgi * ccg, kl = rgi * 4;
        const int half = cN1 >> 1;
        const float *dp = sm + d.off_dP + 4 * cgi;
        for (int t = 0; t < d.ntiles; ++t) {
            const int k0 = t * cKT;
            if (t + 1 < d.ntiles) { issue_x(t + 1); cp_async_commit(); cp_async_wait<1>(); }
            else cp_async_wait<0>();
            __syncthreads();
            if (kl < cKT && k0 + kl < d.D) {
                const float *xr = ((t & 1) ? X1 : X0) + kl;
                float g[4][8];
                f32x2 g2[4][4];                                  // column pairs, packed FMAs
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) g2[j][c] = 0ull;
                for (int s = 0; s < cnt; ++s) {
                    const float4 x = *reinterpret_cast<const float4 *>(xr + s * XS);
                    const ulonglong2 d0 = *reinterpret_cast<const ulonglong2 *>(dp + s * cN1p);
                    const ulonglong2 d1 = *reinterpret_cast<const ulonglong2 *>(dp + s * cN1p + half);
                    const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const f32x2 x2 = pack2(xv[j], xv[j]);
                        ffma2(g2[j][0], x2, d0.x);
                        ffma2(g2[j][1], x2, d0.y);
                        ffma2(g2[j][2], x2, d1.x);
                        ffma2(g2[j][3], x2, d1.y);
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) unpack2(g2[j][c], g[j][2 * c], g[j][2 * c + 1]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (k0 + kl + j < d.D) {
                        float *dst = gout + (size_t)(k0 + kl + j) * cN1 + 4 * cgi;
                        *reinterpret_cast<float4 *>(dst) = make_float4(g[j][0], g[j][1], g[j][2], g[j][3]);
                        *reinterpret_cast<float4 *>(dst + half) = make_float4(g[j][4], g[j][5], g[j][6], g[j][7]);
                        gsum += ((g[j][0] + g[j][1]) + (g[j][2] + g[j][3])) + ((g[j][4] + g[j][5]) + (g[j][6] + g[j][7]));
                    }
                }
            }
            __syncthreads();
        }
        if (!SECOND) continue;

        // ---- scalars of the step (thread 0): history bookkeeping, reward, done, info
        const double gtot = block_sum((double)gsum, reinterpret_cast<double *>(sm + d.off_red2));
        if (tid == 0) step_scalars(d, a, sc, e, loss, gtot, misc);
        __syncthreads();
        const bool wrap = misc[4] != 0.f;
        __syncthreads();
        if (wrap) shuffle_order(d, e, sc);
    }
}

// ------------------------------------------------ tensor-core eval kernel (tcgen05, 3xTF32)
// The two per-env GEMMs of the one-hidden-layer MLP (BASELINE config 4: D = 784, N1 = 64,
// B = 32) on the 5th-generation tensor cores:
//   forward : Hpre^T[j][s] = sum_f W1[f][j] X[s][f]     M = 64 hidden, N = 32 samples, K = D
//   backward: G[f][j]      = sum_s X[s][f] dPre[s][j]   M = 128 features per tile, N = 64, K = 32
// fp32 parity (1e-5) is kept with the 3xTF32 split a = hi + lo (hi = the 19 leading bits, which
// is what the tensor core reads of an fp32 word anyway: profiles/r1_tc_probe.txt):
// a.b ~ lo.hi + hi.lo + hi.hi, accumulated in fp32 in TMEM; measured error 1.3e-6 of
// sum|terms| (profiles/r1_tc_fb_probe_v4.txt).  Operands are staged by the threads (global ->
// registers, one tile ahead -> 4x4 transpose, split -> shared memory) in the K-major
// no-swizzle canonical layout (core matrix = 8 rows x 16 bytes, K chunks 128 bytes apart,
// 8-row groups SBO apart; MN-major no-swizzle descriptors do not work for tf32).  One thread
// issues the MMAs; tcgen05.commit arrives on an mbarrier when the stage may be overwritten.
// One operand stage per CTA, two CTAs per SM overlap each other.  The tail of the network
// (bias, relu, second layer, softmax-CE) is the shared-memory code of the FFMA kernels.
namespace tc {
constexpr int N1 = 64, B = 32, KT = 56, MT = 128;
constexpr int SBO_FA = (KT / 4) * 128 + 16;           // forward A = W1^T tile [64 j  x 56 f]
constexpr int SBO_FB = (KT / 4) * 128;                // forward B = X tile    [32 s  x 56 f]
constexpr int SBO_BA = (B / 4) * 128 + 16;            // backward A = X^T tile [128 f x 32 s]
constexpr int SBO_BB = (B / 4) * 128 + 16;            // backward B = dPre^T   [64 j  x 32 s]
constexpr int A_F = (N1 / 8) * SBO_FA, B_F = (B / 8) * SBO_FB, A_B = (MT / 8) * SBO_BA;
constexpr int STAGE = 2 * A_F + 2 * B_F;              // 43264 bytes >= 2 * A_B
constexpr int DP_B = (N1 / 8) * SBO_BB;
constexpr int OPERAND_BYTES = 2 * STAGE + 2 * DP_B;   // two operand stages + the dPre operand; float region follows
constexpr int TMEM_COLS = 256;                        // forward 32 columns, backward 2 x 64

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}"
                 ::"r"(tmem), "l"(ad), "l"(bd), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool elect_one() {        // one lane of a converged warp (issues the MMAs)
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void split_store(unsigned char *hi, unsigned char *lo, int off, float4 v) {
    float4 h, l;
    // hi = fp32 rounded to nearest at tf32 precision (the tensor core truncates, so the rounding
    // is done here); lo = exact remainder, |lo| <= 2^-12 |v|
    h.x = __uint_as_float((__float_as_uint(v.x) + 0x1000u) & 0xFFFFE000u); l.x = v.x - h.x;
    h.y = __uint_as_float((__float_as_uint(v.y) + 0x1000u) & 0xFFFFE000u); l.y = v.y - h.y;
    h.z = __uint_as_float((__float_as_uint(v.z) + 0x1000u) & 0xFFFFE000u); l.z = v.z - h.z;
    h.w = __uint_as_float((__float_as_uint(v.w) + 0x1000u) & 0xFFFFE000u); l.w = v.w - h.w;
    *reinterpret_cast<float4 *>(hi + off) = h;
    *reinterpret_cast<float4 *>(lo + off) = l;
}
// 4x4 transpose (rows of v = 4 consecutive K indices, columns = 4 consecutive operand rows)
__device__ __forceinline__ void split_store_t(unsigned char *hi, unsigned char *lo, int off, const float4 (&v)[4]) {
    split_store(hi, lo, off, make_float4(v[0].x, v[1].x, v[2].x, v[3].x));
    split_store(hi, lo, off + 16, make_float4(v[0].y, v[1].y, v[2].y, v[3].y));
    split_store(hi, lo, off + 32, make_float4(v[0].z, v[1].z, v[2].z, v[3].z));
    split_store(hi, lo, off + 48, make_float4(v[0].w, v[1].w, v[2].w, v[3].w));
}
#define B2E_TMEM_LD32(taddr, v) \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, " \
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];" \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), \
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), \
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]) \
                 : "r"(taddr))
struct Pre { float4 w[4]; float4 x[2]; };            // one tile of global loads held in registers
}  // namespace tc

template <bool SECOND>
__global__ void __launch_bounds__(256, 2) tc_eval_kernel(const __grid_constant__ Dev d,
                                                         const __grid_constant__ StepArgs a) {
    using namespace tc;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(8) uint64_t bar[2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *sm = reinterpret_cast<float *>(smem_raw);              // Dev offsets (floats) index from here
    unsigned char *dPhi = smem_raw + 2 * STAGE, *dPlo = dPhi + DP_B;
    // row-major Hpre / dPre scratch of the tail lives in stage 1 (idle between the two passes);
    // in the backward pass the same region stages the gradient rows for coalesced stores
    float *Hb = sm + d.off_H, *dPs = sm + d.off_dP, *misc = sm + d.off_misc;
    int *idx_s = reinterpret_cast<int *>(sm + d.off_idx);
    int *ys = reinterpret_cast<int *>(sm + d.off_y);
    const int D = d.D, NT_F = D / KT, NT_B = (D + MT - 1) / MT;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_slot;
    uint32_t uses0 = 0, uses1 = 0;                    // commits issued to each stage barrier (uniform)
    // forward: ONE 128x64x8 MMA per K step, A = [W_hi ; W_lo] rows, B = [X_hi ; X_lo] rows;
    // backward: x_hi.[dP_hi ; dP_lo] (128x128x8) and x_lo.dP_hi (128x64x8)
    const uint32_t idesc_f = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(2 * B >> 3) << 17) | ((uint32_t)(2 * N1 >> 4) << 24);
    const uint32_t idesc_b = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N1 >> 3) << 17) | ((uint32_t)(MT >> 4) << 24);
    const uint32_t idesc_b2 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(2 * N1 >> 3) << 17) | ((uint32_t)(MT >> 4) << 24);
    const uint64_t stage_step = (uint64_t)(STAGE >> 4);
    const uint64_t dFA = make_desc(smem_u32(smem_raw), 128, SBO_FA);
    const uint64_t dFB = make_desc(smem_u32(smem_raw + 2 * A_F), 128, SBO_FB);
    const uint64_t dBAhi = make_desc(smem_u32(smem_raw), 128, SBO_BA), dBAlo = make_desc(smem_u32(smem_raw + A_B), 128, SBO_BA);
    const uint64_t dBB = make_desc(smem_u32(dPhi), 128, SBO_BB);
    const int r8 = lane & 7, q4 = lane >> 3;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    auto wait_stage = [&](int b) {
        const uint32_t u = b ? uses1 : uses0;
        if (u) mbar_wait(&bar[b], (u - 1) & 1);
    };
    const int e_end = a.e_begin + a.e_count;

    for (int e = a.e_begin + blockIdx.x; e < e_end; e += gridDim.x) {
        EnvScalars *sc = d.sc + e;
        const float *We = d.w + (size_t)e * d.Pp;
        float *gout = d.gnext + (size_t)e * d.Pp;
        const int *idx; int cnt;
        current_batch(d, a, e, sc, idx, cnt);
        __syncthreads();
        if (tid < B) {
            const int row = (tid < cnt) ? idx[tid] : -1;          // ragged last batch: missing rows are zeros
            idx_s[tid] = row;
            ys[tid] = row >= 0 ? d.labels[row] : 0;
        }
        for (int i = tid; i < d.tailP; i += blockDim.x) sm[d.off_tw + i] = We[d.P1 + i];
        __syncthreads();
        Pre pre;
        auto load_fwd = [&](int t) {
            const int f0 = t * KT;
            if (tid < (KT / 4) * (N1 / 4)) {
                const int jq = tid & 15, f4 = tid >> 4;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    pre.w[i] = *reinterpret_cast<const float4 *>(We + (size_t)(f0 + 4 * f4 + i) * N1 + 4 * jq);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int c = warp + 8 * u, sg = c >> 2, f4 = (c & 3) * 4 + q4;
                if (f4 < KT / 4) {
                    const int row = idx_s[sg * 8 + r8];
                    pre.x[u] = row >= 0 ? *reinterpret_cast<const float4 *>(d.X + (size_t)row * d.Dp + f0 + 4 * f4) : zero4;
                }
            }
        };
        auto store_fwd = [&](int b) {
            unsigned char *FAhi = smem_raw + b * STAGE, *FAlo = FAhi + A_F, *FBhi = FAlo + A_F, *FBlo = FBhi + B_F;
            if (tid < (KT / 4) * (N1 / 4)) {
                const int jq = tid & 15, f4 = tid >> 4;
                split_store_t(FAhi, FAlo, (jq >> 1) * SBO_FA + f4 * 128 + (jq & 1) * 64, pre.w);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int c = warp + 8 * u, sg = c >> 2, f4 = (c & 3) * 4 + q4;
                if (f4 < KT / 4) split_store(FBhi, FBlo, sg * SBO_FB + f4 * 128 + r8 * 16, pre.x[u]);
            }
        };
        auto load_bwd = [&](int m) {
            const int f0 = m * MT, f4 = tid & 31, sq = tid >> 5;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int row = idx_s[4 * sq + i];
                pre.w[i] = (row >= 0 && f0 + 4 * f4 < D)
                               ? *reinterpret_cast<const float4 *>(d.X + (size_t)row * d.Dp + f0 + 4 * f4) : zero4;
            }
        };
        auto store_bwd = [&]() {
            const int f4 = tid & 31, sq = tid >> 5;
            split_store_t(smem_raw, smem_raw + A_B, (f4 >> 1) * SBO_BA + sq * 128 + (f4 & 1) * 64, pre.w);
        };

        // ================= forward: two operand stages; accumulators: even K steps at TMEM columns
        // [0, 64), odd K steps at [64, 128); rows 0..63 = W_hi, 64..127 = W_lo; columns 0..31 = X_hi
        load_fwd(0);
        for (int t = 0; t < NT_F; ++t) {
            const int b = t & 1;
            wait_stage(b);                                        // MMAs of tile t-2 done: stage b is free
            store_fwd(b);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            if (warp == 0 && elect_one()) {
                // the barrier made every thread's st.shared visible to this thread; one proxy fence
                // orders them before the tensor core's (async proxy) reads
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t so = b ? stage_step : 0;
#pragma unroll
                for (int ks = 0; ks < KT / 8; ++ks) {                        // 8 features = two 16-byte chunks
                    const uint64_t ko = so + (uint64_t)(ks * 256 >> 4);
                    mma_tf32(tmem + 64 * (ks & 1), dFA + ko, dFB + ko, idesc_f, (t == 0 && ks < 2) ? 0u : 1u);
                }
                mma_commit(&bar[b]);
            }
            if (b) uses1++; else uses0++;
            if (t + 1 < NT_F) load_fwd(t + 1); else load_bwd(0);     // in flight while the tensor core works
        }
        wait_stage(0);
        wait_stage(1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (warp < 4) {   // M = 128: accumulator row r sits in TMEM lane r
            float acc[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {                         // small products first: X_lo columns, then X_hi
                const int col = (k < 2 ? 32 : 0) + ((k & 1) ? 0 : 64);
                uint32_t v[32];
                B2E_TMEM_LD32(tmem + ((uint32_t)(warp * 32) << 16) + col, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int i = 0; i < 32; ++i) acc[i] += __uint_as_float(v[i]);
            }
            const int j = (warp & 1) * 32 + lane;
            if (warp >= 2) {                                       // W_lo rows: hand the partial sums over
#pragma unroll
                for (int s = 0; s < B; ++s) dPs[s * N1 + j] = acc[s];
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (warp < 2) {
#pragma unroll
                for (int s = 0; s < B; ++s) Hb[s * N1 + j] = acc[s] + dPs[s * N1 + j];
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        // ================= tail: bias, relu, second layer, softmax-CE -> dPre [B][N1], tail gradient
        const float loss = d.C == 10 ? tail_eval<64, 10>(d, sm, cnt) : tail_eval(d, sm, cnt);
        float gsum = 0.f;
        for (int i = tid; i < d.tailP; i += blockDim.x) {
            const float g = sm[d.off_tg + i];
            gout[d.P1 + i] = g;
            gsum += g;
        }
        // dPre -> B operand (N = hidden j, K = sample s): thread = 4 samples x 4 hidden units
        if (tid < (B / 4) * (N1 / 4)) {
            const int jq = tid & 15, sq = tid >> 4;
            float4 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = *reinterpret_cast<const float4 *>(dPs + (4 * sq + i) * N1 + 4 * jq);
            split_store_t(dPhi, dPlo, (jq >> 1) * SBO_BB + sq * 128 + (jq & 1) * 64, v);
        }
        __syncthreads();                                          // the scratch in stage 1 is dead from here
        // ================= backward: one operand stage (stage 0); accumulators P = x_hi.[dP_hi ; dP_lo]
        // at TMEM columns [0, 128), Q = x_lo.dP_hi at [128, 192); G = P[:, 0:64] + P[:, 64:128] + Q
        float *scr = reinterpret_cast<float *>(smem_raw + STAGE) + warp * (32 * 33);
        auto readout = [&](int m) {
            wait_stage(0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int q = warp & 3, half = warp >> 2;                 // lanes 32q.., columns 32*half.. of each block
            float acc[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = 0.f;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int col = (k == 0 ? 128 : k == 1 ? 64 : 0) + 32 * half;
                uint32_t v[32];
                B2E_TMEM_LD32(tmem + ((uint32_t)(q * 32) << 16) + col, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int i = 0; i < 32; ++i) acc[i] += __uint_as_float(v[i]);
            }
            // lane = feature row; transpose through shared memory so that a warp store covers one row
#pragma unroll
            for (int i = 0; i < 32; ++i) scr[lane * 33 + i] = acc[i];
            __syncwarp();
            const int fbase = m * MT + q * 32;
            for (int r = 0; r < 32; ++r) {
                if (fbase + r < D) {
                    const float g = scr[r * 33 + lane];
                    gout[(size_t)(fbase + r) * N1 + 32 * half + lane] = g;
                    gsum += g;
                }
            }
            __syncwarp();
        };
        for (int m = 0; m < NT_B; ++m) {
            wait_stage(0);                                        // tile m-1 multiplied: stage and accumulators free
            store_bwd();
            if (m >= 1) readout(m - 1);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            if (warp == 0 && elect_one()) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int ks = 0; ks < B / 8; ++ks) {                     // 8 samples = two 16-byte chunks
                    const uint64_t ko = (uint64_t)(ks * 256 >> 4);
                    mma_tf32(tmem, dBAhi + ko, dBB + ko, idesc_b2, ks ? 1u : 0u);
                    mma_tf32(tmem + 128, dBAlo + ko, dBB + ko, idesc_b, ks ? 1u : 0u);
                }
                mma_commit(&bar[0]);
            }
            uses0++;
            if (m + 1 < NT_B) load_bwd(m + 1);
        }
        readout(NT_B - 1);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        if (!SECOND) continue;
        // ---- scalars of the step (thread 0): history bookkeeping, reward, done, info
        __syncthreads();                                          // the reduction scratch shares stage 1
        const double gtot = block_sum((double)gsum, reinterpret_cast<double *>(sm + d.off_red2));
        if (tid == 0) step_scalars(d, a, sc, e, loss, gtot, misc);
        __syncthreads();
        const bool wrap = misc[4] != 0.f;
        __syncthreads();
        if (wrap) shuffle_order(d, e, sc);
    }
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS));
}

// ------------------------------------------------ eval kernel, bulk-copy operand pipeline
// eval_kernel<., 64, 112> with the operand tiles moved by the copy engine instead of the threads:
// per tile ONE cp.async.bulk for the contiguous 28 KB W1 tile and one per minibatch row piece
// (448 B), completing on an mbarrier ("full"); the eight warps arrive on a second mbarrier
// ("empty") when they have consumed a stage and warp 0 then refills it two tiles ahead.  This
// removes the per-thread cp.async issue loops and the two CTA barriers per tile.
namespace bk {
constexpr int N1 = 64, KT = 112, B = 32, XS = 116;
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(tc::smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(tc::smem_u32(bar)) : "memory");
}
}  // namespace bk

// FUSED (first eval only): the update w_t = w_{t-1} - g0 * lr(action) (update_kernel's work) happens in
// the backward epilogue while the gradient tile is still in registers: the W1 tile is bulk-copied
// a second time into the W stage that idles during the backward pass (an L2 hit mostly: this CTA
// read it a few microseconds ago), so g0 is never written, and w / g0 are not re-read from HBM by a
// separate kernel.  Saves 3 of the step's 35 words per parameter and one launch -- but no time:
// measured 1.54 ms against 0.84 + 0.70 ms for the two kernels (profiles/r1_notes.md): the epilogue's
// dependent chain (row lookup -> action gather -> arithmetic -> stores) is appended to each CTA's
// timeline with nothing running underneath it, while the separate update kernel streams at 90 % of
// the HBM rate.  Opt-in (B2E_FUSE_UPDATE=1).
template <bool SECOND, bool FUSED = false>
__global__ void __launch_bounds__(256, 2) eval_bulk_kernel(const __grid_constant__ Dev d,
                                                           const __grid_constant__ StepArgs a) {
    using namespace bk;
    constexpr int PRODUCER = 7;       // the warp that refills the stages: idle in the backward tiles (kl >= KT)
    extern __shared__ __align__(16) float sm[];
    __shared__ __align__(8) uint64_t full[2], empty[2], wfull[2];
    static_assert(!(SECOND && FUSED), "the update belongs to the first eval");
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *const X0 = sm + d.ev_X0, *const W0 = sm + d.ev_W0;
    const int xstep = d.ev_X1 - d.ev_X0, wstep = d.ev_W1 - d.ev_W0;   // stage s at X0 + s * xstep
    float *misc = sm + d.off_misc;
    int *idx_s = reinterpret_cast<int *>(sm + d.off_idx);
    int *ys = reinterpret_cast<int *>(sm + d.off_y);
    const int NT = d.ntiles;                                  // D / 112
    if (tid == 0) {
        mbar_init(&full[0], 1); mbar_init(&full[1], 1);
        mbar_init(&empty[0], 8); mbar_init(&empty[1], 8);
        mbar_init(&wfull[0], 1); mbar_init(&wfull[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    unsigned fph = 0, eph = 0, wph = 0;                       // bit s: phase parity of stage s (warp-uniform)
    const int e_end = a.e_begin + a.e_count;
    for (int e = a.e_begin + blockIdx.x; e < e_end; e += gridDim.x) {
        EnvScalars *sc = d.sc + e;
        const float *wE = d.w + (size_t)e * d.Pp;
        float *gout = d.gnext + (size_t)e * d.Pp;
        float *wOut = d.w + (size_t)e * d.Pp;                                                  // FUSED: updated in place
        float *rw = d.ringw + ((size_t)e * d.H + (sc->head + 1) % d.H) * d.Pp;                 // FUSED: adjusted weights
        const float *act = a.actions + (size_t)e * d.P;
        float s_absw = 0.f;
        double s_lr = 0.0, s_lr2 = 0.0;
        const int *idx; int cnt;
        current_batch(d, a, e, sc, idx, cnt);
        __syncthreads();
        if (tid < B) {
            const int row = (tid < cnt) ? idx[tid] : 0;
            idx_s[tid] = row;
            ys[tid] = (tid < cnt) ? d.labels[row] : 0;
        }
        // rows the minibatch does not have (ragged last batch) read as zeros; the copies never touch them
        for (int i = cnt * XS + tid; i < B * XS; i += blockDim.x) { X0[i] = 0.f; X0[xstep + i] = 0.f; }
        for (int i = tid; i < d.tailP; i += blockDim.x) sm[d.off_tw + i] = wE[d.P1 + i];
        __syncthreads();
        // q = 0..NT-1: forward tiles (W1 and X), q = NT..2NT-1: backward tiles (X only); stage = q & 1
        auto issue = [&](int q) {                              // producer warp only
            const int s = q & 1, t = q < NT ? q : q - NT, k0 = t * KT;
            const bool with_w = q < NT;
            if (lane == 0) mbar_expect(&full[s], (with_w ? KT * N1 * 4 : 0) + cnt * KT * 4);
            __syncwarp();
            if (lane < cnt) bulk_load(X0 + s * xstep + lane * XS, d.X + (size_t)idx_s[lane] * d.Dp + k0, KT * 4, &full[s]);
            if (with_w && lane == 0) bulk_load(W0 + s * wstep, wE + (size_t)k0 * N1, KT * N1 * 4, &full[s]);
        };
        // FUSED: old weights of backward tile q into the idle W stage (own barrier: the first two are
        // requested only after the forward partials have left the W stages)
        auto issue_w = [&](int q) {                            // producer warp only
            const int s = q & 1, k0 = (q - NT) * KT;
            if (lane == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect(&wfull[s], KT * N1 * 4);
                bulk_load(W0 + s * wstep, wE + (size_t)k0 * N1, KT * N1 * 4, &wfull[s]);
            }
        };
        auto wait_full = [&](int s) {
            tc::mbar_wait(&full[s], (fph >> s) & 1u);
            fph ^= 1u << s;
        };
        // This warp is done with the stage of tile q.  The producer warp then waits until every warp
        // is and requests tile q + 2 into it; it runs the forward tiles a little behind the others
        // because of that, which the one-tile lookahead absorbs.  (Requesting from inside its FMA
        // loop instead, with mbarrier.test_wait, measured slower: profiles/r1_notes.md.)
        auto release = [&](int q) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[q & 1]);
            if (warp == PRODUCER) {
                const int s = q & 1;
                tc::mbar_wait(&empty[s], (eph >> s) & 1u);
                eph ^= 1u << s;
                if (q + 2 < 2 * NT) {
                    issue(q + 2);
                    if (FUSED && q >= NT) issue_w(q + 2);
                }
            }
        };
        if (warp == PRODUCER) { issue(0); issue(1); }

        // ---- forward: Hpre = X . W1
        float acc[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;
        for (int t = 0; t < NT; ++t) {
            wait_full(t & 1);
            f_accumulate_fast<N1>(d, X0 + (t & 1) * xstep, XS, W0 + (t & 1) * wstep, KT, acc);
            release(t);
        }
        __syncthreads();                                      // every warp is done with the W tiles
        f_store_fast<N1>(d, sm, acc);                         // partials reduced through the W tiles
        if (FUSED && warp == PRODUCER) { issue_w(NT); if (NT > 1) issue_w(NT + 1); }
        const float loss = d.C == 10 ? tail_eval<N1, 10>(d, sm, cnt) : tail_eval<N1, 0>(d, sm, cnt);

        // ---- backward: tail gradient, then g = X^T . dPre tile by tile, straight to HBM
        float gsum = 0.f;
        for (int i = tid; i < d.tailP; i += blockDim.x) {
            const float g = sm[d.off_tg + i];
            if (FUSED) {                                      // b1, W2, b2: same update, one parameter at a time
                const int p = d.P1 + i;
                const float wo = wE[p];
                const float lr = action_to_lr(act[d.row_lex ? d.row_of_param[p] : p], d.act_ver);
                const float wn = fmaf(-g, lr, wo);
                wOut[p] = wn;
                rw[p] = ratio_nn(wn, wo);
                s_absw += fabsf(wn);
                s_lr += (double)lr;
                s_lr2 += (double)lr * (double)lr;
            } else {
                gout[d.P1 + i] = g;
            }
            gsum += g;
        }
        const int rgi = tid >> 3, cgi = tid & 7, kl = rgi * 4;
        constexpr int half = N1 >> 1;
        const float *dp = sm + d.off_dP + 4 * cgi;
        for (int t = 0; t < NT; ++t) {
            const int q = NT + t, k0 = t * KT;
            wait_full(q & 1);
            if (kl < KT) {
                const float *xr = X0 + (q & 1) * xstep + kl;
                float g[4][8];
                f32x2 g2[4][4];                                  // column pairs, packed FMAs
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) g2[j][c] = 0ull;
                for (int s = 0; s < cnt; ++s) {
                    const float4 x = *reinterpret_cast<const float4 *>(xr + s * XS);
                    const ulonglong2 d0 = *reinterpret_cast<const ulonglong2 *>(dp + s * N1);
                    const ulonglong2 d1 = *reinterpret_cast<const ulonglong2 *>(dp + s * N1 + half);
                    const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const f32x2 x2 = pack2(xv[j], xv[j]);
                        ffma2(g2[j][0], x2, d0.x);
                        ffma2(g2[j][1], x2, d0.y);
                        ffma2(g2[j][2], x2, d1.x);
                        ffma2(g2[j][3], x2, d1.y);
                    }
                }
                if (!FUSED) release(q);                       // the tile is in registers now
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c) unpack2(g2[j][c], g[j][2 * c], g[j][2 * c + 1]);
                if (FUSED) {
                    // rows of the agents first (the only dependent loads), all in flight at once
                    const int pbase = (k0 + kl) * N1 + 4 * cgi;
                    int4 r4[4][2];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            const int p = pbase + j * N1 + hh * half;
                            r4[j][hh] = d.row_lex ? *reinterpret_cast<const int4 *>(d.row_of_param + p)
                                                  : make_int4(p, p + 1, p + 2, p + 3);
                        }
                    float av[4][8];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            av[j][4 * hh + 0] = act[r4[j][hh].x]; av[j][4 * hh + 1] = act[r4[j][hh].y];
                            av[j][4 * hh + 2] = act[r4[j][hh].z]; av[j][4 * hh + 3] = act[r4[j][hh].w];
                        }
                    tc::mbar_wait(&wfull[q & 1], (wph >> (q & 1)) & 1u);
                    wph ^= 1u << (q & 1);
                    const float *ws = W0 + (q & 1) * wstep + kl * N1 + 4 * cgi;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            const float4 wo4 = *reinterpret_cast<const float4 *>(ws + j * N1 + hh * half);
                            const float wo[4] = {wo4.x, wo4.y, wo4.z, wo4.w};
                            float wn[4], aw[4];
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const float lr = action_to_lr(av[j][4 * hh + c], d.act_ver);
                                wn[c] = fmaf(-g[j][4 * hh + c], lr, wo[c]);
                                aw[c] = ratio_nn(wn[c], wo[c]);          // utils_env.py:158-159
                                s_absw += fabsf(wn[c]);
                                s_lr += (double)lr;
                                s_lr2 += (double)lr * (double)lr;
                            }
                            const int p = pbase + j * N1 + hh * half;
                            *reinterpret_cast<float4 *>(wOut + p) = make_float4(wn[0], wn[1], wn[2], wn[3]);
                            *reinterpret_cast<float4 *>(rw + p) = make_float4(aw[0], aw[1], aw[2], aw[3]);
                        }
                    release(q);                               // the old weights have been read
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        gsum += ((g[j][0] + g[j][1]) + (g[j][2] + g[j][3])) + ((g[j][4] + g[j][5]) + (g[j][6] + g[j][7]));
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float *dst = gout + (size_t)(k0 + kl + j) * N1 + 4 * cgi;
                        *reinterpret_cast<float4 *>(dst) = make_float4(g[j][0], g[j][1], g[j][2], g[j][3]);
                        *reinterpret_cast<float4 *>(dst + half) = make_float4(g[j][4], g[j][5], g[j][6], g[j][7]);
                        gsum += ((g[j][0] + g[j][1]) + (g[j][2] + g[j][3])) + ((g[j][4] + g[j][5]) + (g[j][6] + g[j][7]));
                    }
                }
            } else {                                          // the producer warp has no rows here
                if (FUSED) {
                    tc::mbar_wait(&wfull[q & 1], (wph >> (q & 1)) & 1u);
                    wph ^= 1u << (q & 1);
                }
                release(q);
            }
        }
        if (FUSED) {                                          // update_kernel's statistics, whole env in segment 0
            double *red = reinterpret_cast<double *>(sm + d.off_red2);
            const double t0 = block_sum((double)s_absw, red), t1 = block_sum(s_lr, red), t2 = block_sum(s_lr2, red);
            if (tid == 0) {
                double *out = d.part_u + (size_t)e * d.nsegU * 4;
                out[0] = t0; out[1] = t1; out[2] = t2;
                for (int seg = 1; seg < d.nsegU; ++seg) { out[seg * 4] = 0.0; out[seg * 4 + 1] = 0.0; out[seg * 4 + 2] = 0.0; }
            }
        }
        if (!SECOND) continue;

        // ---- scalars of the step (thread 0): history bookkeeping, reward, done, info
        const double gtot = block_sum((double)gsum, reinterpret_cast<double *>(sm + d.off_red2));
        if (tid == 0) step_scalars(d, a, sc, e, loss, gtot, misc);
        __syncthreads();
        const bool wrap = misc[4] != 0.f;
        __syncthreads();
        if (wrap) shuffle_order(d, e, sc);
    }
}

// ------------------------------------------------ thin eval kernel: no hidden layer
// Softmax regression (BASELINE config 3: 784 -> 10): logits Z = X.W + b with at most 16
// classes.  There is almost no arithmetic (1 MFLOP per env); the kernel is the minibatch
// gather, so the feature axis is cut into chunks of KC <= 128 features that stream through
// two small shared-memory buffers with 16-byte cp.async (X rows and the contiguous W chunk):
// ~50 KB per CTA, four CTAs per SM hide each other's latencies.
//   forward : warp = 4 samples, lanes stride over the chunk's features, logits accumulate in
//             registers across the chunks, one shuffle reduction at the end
//   backward: second pass over the chunks (L2 hits); thread = (feature, half of the samples);
//             the chunk's gradient rows are contiguous in HBM and leave as 16-byte stores
constexpr int THIN_CMAX = 16;
constexpr int THIN_KC = 128;
constexpr int THIN_STAGES = 4;                     // chunks in flight: the kernel is bound by load latency

// CC > 0 fixes the class count at compile time (config 3: 10), 0 reads it from the Dev.
template <bool SECOND, int CC = 0>
__global__ void __launch_bounds__(256) thin_eval_kernel(const __grid_constant__ Dev d,
                                                        const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    __shared__ float misc[8];
    __shared__ double red[NSTAT * 8];
    __shared__ int idx_s[64], ys[64];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int D = d.D, C = CC ? CC : d.C, B = d.B, KC = d.KT;     // KT = chunk length here
    constexpr int CU = CC ? CC : THIN_CMAX;                       // unrolled class loops
    const int XS = KC + 4;                                        // row stride of an X chunk (16-byte rows)
    const int nch = (D + KC - 1) / KC;
    float *Xb0 = sm;                                              // [THIN_STAGES][B][XS]
    float *Wb0 = Xb0 + THIN_STAGES * B * XS;                      // [THIN_STAGES][KC][C]
    float *Gs = Wb0 + THIN_STAGES * KC * C;                       // [2][KC][C] partial gradients of the chunk
    float *Zs = Gs + 2 * KC * C;                                  // [B][16] logits, then dZ
    float *lb = Zs + B * THIN_CMAX;                               // [B]
    float *bs = lb + B;                                           // [16]
    const int e_end = a.e_begin + a.e_count;
    for (int e = a.e_begin + blockIdx.x; e < e_end; e += gridDim.x) {
        EnvScalars *sc = d.sc + e;
        const float *wE = d.w + (size_t)e * d.Pp;
        float *gout = d.gnext + (size_t)e * d.Pp;
        const int *idx; int cnt;
        current_batch(d, a, e, sc, idx, cnt);
        __syncthreads();
        for (int r = tid; r < B; r += blockDim.x) {
            const int row = (r < cnt) ? idx[r] : -1;
            idx_s[r] = row;
            ys[r] = row >= 0 ? d.labels[row] : 0;
        }
        if (tid < THIN_CMAX) bs[tid] = tid < C ? wE[d.P1 + tid] : 0.f;
        __syncthreads();
        auto issue = [&](int ch, bool with_w) {
            const int k0 = ch * KC, krows = min(KC, D - k0), kq = (krows + 3) >> 2;
            float *xb = Xb0 + (ch % THIN_STAGES) * B * XS;
            for (int r = warp; r < B; r += 8) {                   // warp = row, lanes = its 16-byte pieces
                const int row = idx_s[r];
                for (int c = lane; c < kq; c += 32) {
                    if (row >= 0) cp_async16(xb + r * XS + 4 * c, d.X + (size_t)row * d.Dp + k0 + 4 * c);
                    else *reinterpret_cast<float4 *>(xb + r * XS + 4 * c) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            if (with_w) {
                float *wb = Wb0 + (ch % THIN_STAGES) * KC * C;
                const float *src = wE + (size_t)k0 * C;
                const int n = krows * C, nq = n >> 2;             // k0 * C is a multiple of 4 (KC * C % 4 == 0)
                for (int i = tid; i < nq; i += blockDim.x) cp_async16(wb + 4 * i, src + 4 * i);
                for (int i = 4 * nq + tid; i < n; i += blockDim.x) wb[i] = src[i];
            }
            cp_async_commit();
        };
        // ---- forward: Z[s][c] accumulated over the chunks, warp = 4 samples per pass
        float acc[4][THIN_CMAX];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int c = 0; c < THIN_CMAX; ++c) acc[i][c] = 0.f;
        const int s0 = warp * 4;                                  // B <= 32: one pass of 8 warps x 4 samples
        for (int ch = 0; ch < THIN_STAGES - 1; ++ch) { if (ch < nch) issue(ch, true); else cp_async_commit(); }
        for (int ch = 0; ch < nch; ++ch) {
            if (ch + THIN_STAGES - 1 < nch) issue(ch + THIN_STAGES - 1, true); else cp_async_commit();
            cp_async_wait<THIN_STAGES - 1>();                     // chunk ch has landed
            __syncthreads();
            const int krows = min(KC, D - ch * KC);
            const float *xb = Xb0 + (ch % THIN_STAGES) * B * XS, *wb = Wb0 + (ch % THIN_STAGES) * KC * C;
            if (s0 < B) {
                const float *x0 = xb + min(s0, B - 1) * XS, *x1 = xb + min(s0 + 1, B - 1) * XS;
                const float *x2 = xb + min(s0 + 2, B - 1) * XS, *x3 = xb + min(s0 + 3, B - 1) * XS;
                if (CC && CC % 2 == 0) {
                    // even compile-time class count: W row as 8-byte pairs, packed FMAs (FFMA2)
                    f32x2 a2[4][CU / 2 + 1];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int c = 0; c < CU / 2; ++c) a2[i][c] = pack2(acc[i][2 * c], acc[i][2 * c + 1]);
                    for (int k = lane; k < krows; k += 32) {
                        const f32x2 xx[4] = {pack2(x0[k], x0[k]), pack2(x1[k], x1[k]), pack2(x2[k], x2[k]), pack2(x3[k], x3[k])};
                        const f32x2 *wr = reinterpret_cast<const f32x2 *>(wb + k * C);
#pragma unroll
                        for (int c = 0; c < CU / 2; ++c) {
                            const f32x2 w2 = wr[c];
#pragma unroll
                            for (int i = 0; i < 4; ++i) ffma2(a2[i][c], xx[i], w2);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int c = 0; c < CU / 2; ++c) unpack2(a2[i][c], acc[i][2 * c], acc[i][2 * c + 1]);
                } else {
                    for (int k = lane; k < krows; k += 32) {
                        const float xv[4] = {x0[k], x1[k], x2[k], x3[k]};
                        const float *wr = wb + k * C;
#pragma unroll
                        for (int c = 0; c < CU; ++c) {
                            if (CC || c < C) {
                                const float w = wr[c];
#pragma unroll
                                for (int i = 0; i < 4; ++i) acc[i][c] = fmaf(xv[i], w, acc[i][c]);
                            }
                        }
                    }
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int c = 0; c < CU; ++c) {
                if (CC || c < C) {
                    float v = acc[i][c];
                    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                    if (lane == 0 && s0 + i < B) Zs[(s0 + i) * THIN_CMAX + c] = v + bs[c];
                }
            }
        __syncthreads();
        for (int ch = 0; ch < THIN_STAGES - 1; ++ch) { if (ch < nch) issue(ch, false); else cp_async_commit(); }   // backward pass travels
        // ---- softmax cross-entropy per sample, dZ in place (problems/optimize_nn.py:47-50)
        for (int s = tid; s < B; s += blockDim.x) {
            float *z = Zs + s * THIN_CMAX;
            float loss = 0.f;
            if (s < cnt) {
                const int y = ys[s];
                float m = z[0];
                for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
                float sum = 0.f;
                for (int c = 0; c < C; ++c) sum += expf(z[c] - m);
                loss = (m + logf(sum)) - z[y];
                const float inv = 1.0f / sum;
                for (int c = 0; c < C; ++c) z[c] = expf(z[c] - m) * inv - (c == y ? 1.f : 0.f);
                for (int c = C; c < THIN_CMAX; ++c) z[c] = 0.f;
            } else {
                for (int c = 0; c < THIN_CMAX; ++c) z[c] = 0.f;
            }
            lb[s] = loss;
        }
        __syncthreads();
        if (warp == 0) {                                          // mean loss, summed in sample order by one lane
            float l = 0.f;
            if (lane == 0) { for (int s = 0; s < cnt; ++s) l += lb[s]; misc[0] = l / (float)cnt; }
        }
        __syncthreads();
        const float loss = misc[0];
        // ---- backward: thread = (feature k of the chunk, half h of the samples)
        float gsum = 0.f;
        const int kk = tid & (THIN_KC - 1), hh = tid >> 7;
        const int s_lo = hh * ((B + 1) >> 1), s_hi = hh ? B : ((B + 1) >> 1);
        for (int ch = 0; ch < nch; ++ch) {
            if (ch + THIN_STAGES - 1 < nch) issue(ch + THIN_STAGES - 1, false); else cp_async_commit();
            cp_async_wait<THIN_STAGES - 1>();
            __syncthreads();
            const int k0 = ch * KC, krows = min(KC, D - k0);
            const float *xb = Xb0 + (ch % THIN_STAGES) * B * XS;
            if (kk < krows) {
                float g[THIN_CMAX];
#pragma unroll
                for (int c = 0; c < THIN_CMAX; ++c) g[c] = 0.f;
                for (int s = s_lo; s < s_hi; ++s) {
                    const float x = xb[s * XS + kk];
                    const float4 *dz = reinterpret_cast<const float4 *>(Zs + s * THIN_CMAX);
#pragma unroll
                    for (int q = 0; q < (CU + 3) / 4; ++q) {
                        if (CC || 4 * q < C) {
                            const float4 d4 = dz[q];
                            g[4 * q] = fmaf(x, d4.x, g[4 * q]);
                            g[4 * q + 1] = fmaf(x, d4.y, g[4 * q + 1]);
                            g[4 * q + 2] = fmaf(x, d4.z, g[4 * q + 2]);
                            g[4 * q + 3] = fmaf(x, d4.w, g[4 * q + 3]);
                        }
                    }
                }
#pragma unroll
                for (int c = 0; c < CU; ++c)
                    if (CC || c < C) Gs[(hh * KC + kk) * C + c] = g[c];
            }
            __syncthreads();
            // the chunk's gradient rows [k0, k0 + krows) x C are contiguous in HBM
            const int n = krows * C;
            float *dst = gout + (size_t)k0 * C;
            for (int i = tid * 4; i < n; i += blockDim.x * 4) {
                if (i + 3 < n) {
                    const float4 u = *reinterpret_cast<const float4 *>(Gs + i);
                    const float4 v = *reinterpret_cast<const float4 *>(Gs + KC * C + i);
                    const float4 g4 = make_float4(u.x + v.x, u.y + v.y, u.z + v.z, u.w + v.w);
                    *reinterpret_cast<float4 *>(dst + i) = g4;
                    gsum += (g4.x + g4.y) + (g4.z + g4.w);
                } else {
                    for (int j = i; j < n; ++j) { const float g = Gs[j] + Gs[KC * C + j]; dst[j] = g; gsum += g; }
                }
            }
            // no barrier needed here: the next iteration's barrier orders these reads of Gs before its writes
        }
        __syncthreads();
        if (tid < C) {
            float g = 0.f;
            for (int s = 0; s < cnt; ++s) g += Zs[s * THIN_CMAX + tid];
            gout[d.P1 + tid] = g;
            gsum += g;
        }
        if (!SECOND) continue;
        const double gtot = block_sum((double)gsum, red);
        if (tid == 0) step_scalars(d, a, sc, e, loss, gtot, misc);
        __syncthreads();
        const bool wrap = misc[4] != 0.f;
        __syncthreads();
        if (wrap) shuffle_order(d, e, sc);
    }
}

// w_t = w_{t-1} - g0 * lr(action)  (multioptlrs.py:86-87), adjusted-weight ring, statistics.
constexpr int UPD_QUADS = 4;                      // float4 groups per thread
constexpr int UPD_SEG = 256 * UPD_QUADS * 4;      // parameters per CTA

__global__ void __launch_bounds__(256) update_kernel(const __grid_constant__ Dev d,
                                                     const __grid_constant__ StepArgs a) {
    const int e = a.e_begin + blockIdx.y;
    const int seg = blockIdx.x;
    const EnvScalars *sc = d.sc + e;
    const int head_new = (sc->head + 1) % d.H;
    float *wE = d.w + (size_t)e * d.Pp;
    const float *gE = d.gnext + (size_t)e * d.Pp;             // g0, left there by the first eval
    float *rw = d.ringw + ((size_t)e * d.H + head_new) * d.Pp;
    const float *act = a.actions + (size_t)e * d.P;
    float4 w4[UPD_QUADS], g4[UPD_QUADS];
    int4 r4[UPD_QUADS];
    int pq[UPD_QUADS];
#pragma unroll
    for (int i = 0; i < UPD_QUADS; ++i) {
        pq[i] = seg * UPD_SEG + (i * 256 + threadIdx.x) * 4;
        if (pq[i] < d.P) {
            w4[i] = *reinterpret_cast<const float4 *>(wE + pq[i]);
            g4[i] = *reinterpret_cast<const float4 *>(gE + pq[i]);
            r4[i] = d.row_lex ? *reinterpret_cast<const int4 *>(d.row_of_param + pq[i])
                              : make_int4(pq[i], pq[i] + 1, pq[i] + 2, pq[i] + 3);
        }
    }
    float av[UPD_QUADS][4];
#pragma unroll
    for (int i = 0; i < UPD_QUADS; ++i) {
        const int rows[4] = {r4[i].x, r4[i].y, r4[i].z, r4[i].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) av[i][j] = (pq[i] + j < d.P) ? act[rows[j]] : 0.f;
    }
    float s_absw = 0.f, s_absaw = 0.f;
    double s_lr = 0.0, s_lr2 = 0.0;
#pragma unroll
    for (int i = 0; i < UPD_QUADS; ++i) {
        if (pq[i] >= d.P) continue;
        const float wv[4] = {w4[i].x, w4[i].y, w4[i].z, w4[i].w};
        const float gv[4] = {g4[i].x, g4[i].y, g4[i].z, g4[i].w};
        float wn[4], aw[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float lr = action_to_lr(av[i][j], d.act_ver);
            wn[j] = fmaf(-gv[j], lr, wv[j]);
            aw[j] = ratio_nn(wn[j], wv[j]);                      // utils_env.py:158-159
            if (pq[i] + j < d.P) {
                s_absw += fabsf(wn[j]);
                s_absaw += fabsf(aw[j]);
                s_lr += (double)lr;
                s_lr2 += (double)lr * (double)lr;
            } else {
                wn[j] = 0.f; aw[j] = 0.f;
            }
        }
        *reinterpret_cast<float4 *>(wE + pq[i]) = make_float4(wn[0], wn[1], wn[2], wn[3]);
        *reinterpret_cast<float4 *>(rw + pq[i]) = make_float4(aw[0], aw[1], aw[2], aw[3]);
    }
    __shared__ double red[8 * 4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double v0 = warp_sum((double)s_absw), v1 = warp_sum(s_lr), v2 = warp_sum(s_lr2);
    const double v3 = warp_sum((double)s_absaw);             // sum |adjusted weights| of the new ring slot
    if (lane == 0) { red[warp * 4] = v0; red[warp * 4 + 1] = v1; red[warp * 4 + 2] = v2; red[warp * 4 + 3] = v3; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double *out = d.part_u + ((size_t)e * d.nsegU + seg) * 4;
        for (int i = 0; i < 4; ++i) {
            double v = 0.0;
            for (int w = 0; w < 8; ++w) v += red[w * 4 + i];
            out[i] = v;
        }
    }
}

// Ring-only step (b2e_step with obs_out = NULL; SURVEY 8f.2): what obs_kernel does minus the observation
// rows -- the adjusted gradient g_t / |g_{t-1}| (utils_env.py:156-157) into the newest ring slot and the
// partial sums of adjusted_grad / grad_diff.  Parameter space, float4, fully coalesced: 2 words read and
// 1 written per parameter instead of 26.  A consumer reads the rings in place (b2p_act_env).
__global__ void __launch_bounds__(256) ring_adjg_kernel(const __grid_constant__ Dev d,
                                                        const __grid_constant__ StepArgs a) {
    const int e = a.e_begin + blockIdx.y;
    const int seg = blockIdx.x;
    const EnvScalars *sc = d.sc + e;
    const float *gnew = d.gnext + (size_t)e * d.Pp;
    const float *gold = d.gprev + (size_t)e * d.Pp;
    float *rg = d.ringg + ((size_t)e * d.H + sc->head) * d.Pp;    // eval<w_new> has advanced the head
    float4 gn[UPD_QUADS], go[UPD_QUADS];
    int pq[UPD_QUADS];
#pragma unroll
    for (int i = 0; i < UPD_QUADS; ++i) {
        pq[i] = seg * UPD_SEG + (i * 256 + threadIdx.x) * 4;
        if (pq[i] < d.P) {
            gn[i] = *reinterpret_cast<const float4 *>(gnew + pq[i]);
            go[i] = *reinterpret_cast<const float4 *>(gold + pq[i]);
        }
    }
    float s_absadjg = 0.f, s_gdiff = 0.f;
#pragma unroll
    for (int i = 0; i < UPD_QUADS; ++i) {
        if (pq[i] >= d.P) continue;
        const float g1[4] = {gn[i].x, gn[i].y, gn[i].z, gn[i].w};
        const float g0[4] = {go[i].x, go[i].y, go[i].z, go[i].w};
        float ag[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            ag[j] = ratio_nn(g1[j], g0[j]);
            if (pq[i] + j < d.P) {
                s_absadjg += fabsf(ag[j]);
                s_gdiff += fabsf(g1[j] - g0[j]);
            } else {
                ag[j] = 0.f;
            }
        }
        *reinterpret_cast<float4 *>(rg + pq[i]) = make_float4(ag[0], ag[1], ag[2], ag[3]);
    }
    __shared__ double red[8 * 2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double v0 = warp_sum((double)s_absadjg), v1 = warp_sum((double)s_gdiff);
    if (lane == 0) { red[warp * 2] = v0; red[warp * 2 + 1] = v1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double *out = d.part_r + ((size_t)e * d.nsegU + seg) * 4;
        for (int i = 0; i < 2; ++i) {
            double v = 0.0;
            for (int w = 0; w < 8; ++w) v += red[w * 2 + i];
            out[i] = v;
        }
    }
}

// sum |x| of every ring slot after b2e_set_state wrote the rings (ring-only steps rebuild states_sum from these)
__global__ void __launch_bounds__(256) slot_abs_kernel(Dev d) {
    const int e = blockIdx.x / d.H, slot = blockIdx.x - e * d.H;
    const float *rw = d.ringw + ((size_t)e * d.H + slot) * d.Pp, *rg = d.ringg + ((size_t)e * d.H + slot) * d.Pp;
    double sw = 0.0, sg = 0.0;
    for (int p = threadIdx.x; p < d.P; p += blockDim.x) { sw += (double)fabsf(rw[p]); sg += (double)fabsf(rg[p]); }
    __shared__ double red[8];
    sw = block_sum(sw, red);
    sg = block_sum(sg, red);
    if (threadIdx.x == 0) { d.slot_abs[((size_t)e * d.H + slot) * 2] = sw; d.slot_abs[((size_t)e * d.H + slot) * 2 + 1] = sg; }
}

// info entries that need the streaming kernels' partial sums (states_*, adjusted_grad, grad_diff)
__global__ void info_finalize_kernel(Dev d, StepArgs a) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= d.E) return;
    const EnvScalars *sc = d.sc + e;
    const bool ring_only = a.obs == nullptr;
    double absadjg = 0.0, gdiff = 0.0, state = 0.0;
    if (ring_only) {
        for (int s = 0; s < d.nsegU; ++s) {
            const double *in = d.part_r + ((size_t)e * d.nsegU + s) * 4;
            absadjg += in[0]; gdiff += in[1];
        }
    } else {
        for (int s = 0; s < d.nseg; ++s) {
            const double *in = d.part + ((size_t)e * d.nseg + s) * 4;
            absadjg += in[0]; gdiff += in[1]; state += in[2];
        }
    }
    if (d.slot_abs) {
        // every step records sum |.| of the two planes it appended; a ring-only step, which never visits
        // the older slots, adds those up for states_mean / states_sum (multioptlrs.py:119-120)
        double absaw = 0.0;
        for (int s = 0; s < d.nsegU; ++s) absaw += d.part_u[((size_t)e * d.nsegU + s) * 4 + 3];
        double *sa = d.slot_abs + (size_t)e * d.H * 2;
        sa[sc->head * 2] = absaw;
        sa[sc->head * 2 + 1] = absadjg;
        if (ring_only) {
            for (int h = 0; h < d.H && h < sc->nvalid; ++h) {
                int slot = sc->head - h;
                slot += slot < 0 ? d.H : 0;
                state += sa[slot * 2] + sa[slot * 2 + 1];
            }
        }
    }
    double labs = 0.0;
    for (int h = 0; d.col_l >= 0 && h < d.H && h < sc->nvalid; ++h) {
        int slot = sc->head - h;
        slot += slot < 0 ? d.H : 0;
        labs += (double)fabsf(sc->adj_loss[slot]);
    }
    double absw = 0.0, lr = 0.0, lr2 = 0.0;
    for (int s = 0; s < d.nsegU; ++s) {
        const double *in = d.part_u + ((size_t)e * d.nsegU + s) * 4;
        absw += in[0]; lr += in[1]; lr2 += in[2];
    }
    const double P = (double)d.P;
    const double ssum = state + P * labs;
    double *info = a.info + (size_t)e * B2E_INFO_STRIDE;
    const double lr_mean = lr / P;
    double lr_var = lr2 / P - lr_mean * lr_mean;
    lr_var = lr_var > 0.0 ? lr_var : 0.0;
    info[2] = absw / P;
    info[3] = absw;
    info[4] = lr_mean;
    info[5] = sqrt(lr_var);
    info[6] = ssum / (P * (double)d.OD);
    info[7] = ssum;
    info[12] = absadjg / P;
    info[13] = gdiff / P;
}


// =========================================================================================
// Reset pipeline of the tcgen05 path (MultiOptLRs, BASELINE config 4 / 5): base_reset
// (envs/multioptlrs.py:66-78) as
//   reset_list_kernel    : the envs to reset (mask / done flags, or all), ascending, + their count
//   reset_prepare_kernel : reshuffle (optimize_nn.py:114-120), cursor 0, fresh parameters
//   tc2 eval kernel      : loss and gradient of the listed envs at the fresh parameters (b200tc.cu)
//   reset_finish_kernel  : histories / counters, the raw-history gradient sum, the all -1 observation rows
// instead of the one-CTA-per-SM fused kernel in reset mode (10.4 ms for 4096 envs; this takes ~3 ms).  With no env
// to reset (the usual auto-reset launch of a step) every kernel finds an empty list and returns.
// =========================================================================================
__global__ void __launch_bounds__(1024) reset_list_kernel(const unsigned char *mask, int E, int *list, int *count) {
    __shared__ int warp_tot[32];
    __shared__ int base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int e0 = 0; e0 < E; e0 += 1024) {
        const int e = e0 + threadIdx.x;
        const bool flag = e < E && (!mask || mask[e]);
        const unsigned ballot = __ballot_sync(0xffffffffu, flag);
        if (lane == 0) warp_tot[warp] = __popc(ballot);
        __syncthreads();
        int off = base;
        for (int w = 0; w < warp; ++w) off += warp_tot[w];
        if (flag) list[off + __popc(ballot & ((1u << lane) - 1u))] = e;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < 32; ++w) t += warp_tot[w];
            base += t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

__global__ void __launch_bounds__(256) reset_prepare_kernel(const __grid_constant__ Dev d, const __grid_constant__ StepArgs a) {
    const int n = *a.env_count;
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
        const int e = a.env_list[i];
        EnvScalars *sc = d.sc + e;
        if (d.index_mode == B2E_INDEX_INTERNAL) {
            // InMemoryDataSet.on_epoch_end (shuffle_order) with eight independent gathers in flight per thread
            const int sel = sc->ord_sel;
            const int *src = order_ptr(d, e, sel);
            int *dst = d.ord + ((size_t)(sel ^ 1) * d.E + e) * d.N;
            const int *pm = d.perm + (size_t)e * d.perm_stride;
            if ((d.N & 3) == 0 && (d.perm_stride & 3) == 0) {
                const int nq = d.N >> 2;
                for (int q = threadIdx.x; q < nq; q += 2 * blockDim.x) {
                    const int q2 = q + blockDim.x;
                    const int4 a4 = reinterpret_cast<const int4 *>(pm)[q];
                    const int4 b4 = q2 < nq ? reinterpret_cast<const int4 *>(pm)[q2] : make_int4(0, 0, 0, 0);
                    const int4 ra = make_int4(src[a4.x], src[a4.y], src[a4.z], src[a4.w]);
                    const int4 rb = make_int4(src[b4.x], src[b4.y], src[b4.z], src[b4.w]);
                    reinterpret_cast<int4 *>(dst)[q] = ra;
                    if (q2 < nq) reinterpret_cast<int4 *>(dst)[q2] = rb;
                }
            } else {
                for (int i = threadIdx.x; i < d.N; i += blockDim.x) dst[i] = src[pm[i]];
            }
            __syncthreads();
            if (threadIdx.x == 0) { sc->ord_sel = sel ^ 1; sc->cursor = 0; }
            __syncthreads();
        }
        const int episode = sc->episode;
        float *wE = d.w + (size_t)e * d.Pp;
        for (int p = threadIdx.x; p < d.Pp; p += blockDim.x) {
            float v = 0.f;
            if (p < d.P) {
                if (a.init_params) v = a.init_params[(size_t)e * d.P + p];
                else if (p < d.P1) v = glorot(d.seed, e + d.env_base, episode, p, d.lim1);
                else if (d.hidden && p >= d.P1 + d.N1 && p < d.P1 + d.N1 + d.N1 * d.C) v = glorot(d.seed, e + d.env_base, episode, p, d.lim2);
            }
            wE[p] = v;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) reset_finish_kernel(const __grid_constant__ Dev d, const __grid_constant__ StepArgs a) {
    __shared__ double red[8];
    const int n = *a.env_count;
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
        const int e = a.env_list[i];
        EnvScalars *sc = d.sc + e;
        const float *gE = d.gprev + (size_t)e * d.Pp;           // the eval kernel left the reset gradient here
        double gs = 0.0;
        for (int p = threadIdx.x; p < d.P; p += blockDim.x) gs += (double)gE[p];
        gs = block_sum(gs, red);
        if (threadIdx.x == 0) {
            const float loss = a.loss_out[e];
            for (int k = 0; k < RAW_DEPTH; ++k) { sc->raw_loss[k] = 0.f; sc->raw_gsum[k] = 0.0; }   // multioptlrs.py:69
            for (int k = 0; k < B2E_MAX_HISTORY; ++k) sc->adj_loss[k] = 0.f;
            sc->raw_pos = 0;
            sc->raw_loss[0] = loss;
            sc->raw_gsum[0] = gs;
            sc->loss_prev = loss;
            sc->head = d.H - 1;
            sc->nvalid = 0;
            sc->step = 0;
            sc->episode = sc->episode + 1;
        }
        if (a.obs) {                                            // clip(0) - 1 = -1 in every column (multioptlrs.py:70-78)
            float *o = a.obs + (size_t)e * d.P * d.OD;
            const size_t total = (size_t)d.P * d.OD;
            const size_t head = min(total, (size_t)((4 - ((reinterpret_cast<uintptr_t>(o) >> 2) & 3)) & 3));
            const size_t quads = (total - head) >> 2;
            if (threadIdx.x < head) o[threadIdx.x] = -1.0f;
            float4 *o4 = reinterpret_cast<float4 *>(o + head);
            const float4 m1 = make_float4(-1.f, -1.f, -1.f, -1.f);
            for (size_t q = threadIdx.x; q < quads; q += blockDim.x) o4[q] = m1;
            for (size_t t = head + (quads << 2) + threadIdx.x; t < total; t += blockDim.x) o[t] = -1.0f;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- MultiOptimize
// envs/multioptimize.py:90-154 as a pipeline for every problem size:
//   mo_update_kernel : w_t = w_{t-1} - delta(a); adjusted-weight ring; raw weight planes
//   eval             : g_t, L_t and the step's scalars (eval_kernel<true> / MODE_EVAL_STEP)
//   mo_obs_kernel    : adjusted-gradient ring, raw gradient planes, observation rows
__global__ void __launch_bounds__(256) mo_update_kernel(const __grid_constant__ Dev d,
                                                        const __grid_constant__ StepArgs a) {
    const int e = a.e_begin + blockIdx.y;
    const int seg = blockIdx.x;
    const EnvScalars *sc = d.sc + e;
    const int head_new = (sc->head + 1) % d.H;
    float *wE = d.w + (size_t)e * d.Pp;
    float *w2E = d.w2 ? d.w2 + (size_t)e * d.Pp : nullptr;
    float *rw = d.col_w >= 0 ? d.ringw + ((size_t)e * d.H + head_new) * d.Pp : nullptr;
    const float *act = a.actions + (size_t)e * d.P;
    float s_absw = 0.f;
    double s_lr = 0.0, s_lr2 = 0.0;
    for (int i = 0; i < UPD_QUADS; ++i) {
        const int p = seg * UPD_SEG + (i * 256 + threadIdx.x) * 4;
        if (p >= d.P) continue;
        const float4 w4 = *reinterpret_cast<const float4 *>(wE + p);
        float4 o4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (w2E) o4 = *reinterpret_cast<const float4 *>(w2E + p);
        const int4 r4 = d.row_lex ? *reinterpret_cast<const int4 *>(d.row_of_param + p)
                                  : make_int4(p, p + 1, p + 2, p + 3);
        const int rows[4] = {r4.x, r4.y, r4.z, r4.w};
        const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
        const float ov[4] = {o4.x, o4.y, o4.z, o4.w};
        float wn[4], aw[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            wn[j] = 0.f; aw[j] = 0.f;
            if (p + j < d.P) {
                const float delta = action_to_delta(act[rows[j]], d.act_ver);   // multioptimize.py:95-102
                wn[j] = wv[j] - delta;                                          // :103
                aw[j] = adjust_w(d.obs_ver, wn[j], wv[j], ov[j]);
                s_absw += fabsf(wn[j]);
                s_lr += (double)delta;
                s_lr2 += (double)delta * (double)delta;
            }
        }
        *reinterpret_cast<float4 *>(wE + p) = make_float4(wn[0], wn[1], wn[2], wn[3]);
        if (w2E) *reinterpret_cast<float4 *>(w2E + p) = w4;
        if (rw) *reinterpret_cast<float4 *>(rw + p) = make_float4(aw[0], aw[1], aw[2], aw[3]);
    }
    __shared__ double red[8 * 4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double v0 = warp_sum((double)s_absw), v1 = warp_sum(s_lr), v2 = warp_sum(s_lr2);
    if (lane == 0) { red[warp * 4] = v0; red[warp * 4 + 1] = v1; red[warp * 4 + 2] = v2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double *out = d.part_u + ((size_t)e * d.nsegU + seg) * 4;
        for (int i = 0; i < 3; ++i) {
            double v = 0.0;
            for (int w = 0; w < 8; ++w) v += red[w * 4 + i];
            out[i] = v;
        }
    }
}

// Row-space observation kernel for every history layout / observation version
// (utils/utils_env.py:9-47, 126-164; utils/utils_common.py:188-196): rows are
// [key blocks in insertion order][depth values newest first], not clipped.
__global__ void __launch_bounds__(OBS_WARPS * 32) mo_obs_kernel(const __grid_constant__ Dev d,
                                                                const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    __shared__ double red[OBS_WARPS * 4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int H = d.H, OD = d.OD;
    float *obsL_s = sm;                                       // [B2E_MAX_HISTORY]
    float *stage = sm + B2E_MAX_HISTORY + warp * (32 * OD + 8);
    const int nitems = a.e_count * d.nseg;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int eo = item / d.nseg;
        const int e = a.e_begin + eo;
        const int seg = item - eo * d.nseg;
        const EnvScalars *sc = d.sc + e;
        const int head = sc->head, nvalid = sc->nvalid;      // already advanced by the eval stage
        __syncthreads();
        if (threadIdx.x < H) {
            const int h = threadIdx.x;
            float v = 0.f;
            if (h < nvalid) {
                int slot = head - h;
                slot += slot < 0 ? H : 0;
                v = sc->adj_loss[slot];
            }
            obsL_s[h] = v;
        }
        __syncthreads();
        const float *gnew = d.gnext + (size_t)e * d.Pp;
        float *gold = d.gprev + (size_t)e * d.Pp;
        float *g2E = d.g2 ? d.g2 + (size_t)e * d.Pp : nullptr;
        const float *rw = d.ringw + (size_t)e * H * d.Pp;
        float *rg = d.ringg + (size_t)e * H * d.Pp;
        float *rg_new = rg + (size_t)head * d.Pp;
        float *obs_env = a.obs + (size_t)e * d.P * OD;
        float s_absadjg = 0.f, s_gdiff = 0.f, s_state = 0.f;
        for (int it = 0; it < OBS_ITERS; ++it) {
            const int rbase = seg * SEG_ROWS + (it * OBS_WARPS + warp) * 32;
            if (rbase >= d.P) break;
            const int r = rbase + lane;
            const bool ok = r < d.P;
            const int p = ok ? (d.row_lex ? d.param_of_row[r] : r) : 0;
            const float g = gnew[p], gp = gold[p];
            const float g2 = g2E ? g2E[p] : 0.f;
            const float ag = adjust_g(d.obs_ver, g, gp, g2);
            if (ok) {
                rg_new[p] = ag;
                gold[p] = g;                                  // raw History shift
                if (g2E) g2E[p] = gp;
                s_absadjg += fabsf(ag);
                s_gdiff += fabsf(g - gp);
            }
            const unsigned w_lo = (unsigned)rbase * OD;
            const unsigned sh = (unsigned)((((size_t)e * d.P * OD) + w_lo) & 3);
            float *srow = stage + sh + lane * OD;
            for (int h = 0; h < H; ++h) {
                float w1 = 0.f, g1 = 0.f;
                if (h < nvalid) {
                    int slot = head - h;
                    slot += slot < 0 ? H : 0;
                    if (d.col_w >= 0) w1 = rw[(size_t)slot * d.Pp + p];
                    g1 = h > 0 ? rg[(size_t)slot * d.Pp + p] : ag;
                }
                if (ok) s_state += fabsf(w1) + fabsf(g1);
                if (d.col_w >= 0) srow[d.col_w + h] = w1;
                if (d.col_l >= 0) srow[d.col_l + h] = obsL_s[h];
                srow[d.col_g + h] = g1;
            }
            __syncwarp();
            const unsigned nw = (unsigned)min(32, d.P - rbase) * OD;
            float *dst = obs_env + w_lo;
            const float *src = stage + sh;
            const unsigned head_w = min(nw, (4u - sh) & 3u);
            const unsigned body_e = head_w + ((nw - head_w) & ~3u);
            if (lane < head_w) dst[lane] = src[lane];
            for (unsigned i = head_w + lane * 4; i < body_e; i += 128)
                *reinterpret_cast<float4 *>(dst + i) = *reinterpret_cast<const float4 *>(src + i);
            if (body_e + lane < nw) dst[body_e + lane] = src[body_e + lane];
            __syncwarp();
        }
        const double v0 = warp_sum((double)s_absadjg), v1 = warp_sum((double)s_gdiff);
        const double v2 = warp_sum((double)s_state);
        if (lane == 0) { red[warp * 4] = v0; red[warp * 4 + 1] = v1; red[warp * 4 + 2] = v2; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double *out = d.part + ((size_t)e * d.nseg + seg) * 4;
            for (int i = 0; i < 3; ++i) {
                double v = 0.0;
                for (int w = 0; w < OBS_WARPS; ++w) v += red[w * 4 + i];
                out[i] = v;
            }
        }
    }
}

// ---------------------------------------------------------------- generic dense stack
// Any `layers` tuple of the reference's create_neural_net (utils/utils_tf.py:74-86; default
// (256, 256)) and any minibatch size (MultiOptimize's batch_size=None is the whole data set):
// one CTA per env, activations and deltas in a per-CTA HBM/L2 workspace, every matmul a
// 64x64x16 shared-memory tiled FFMA GEMM with 4x4 register tiles.  Slower than the
// single-hidden-layer kernels above but shape-agnostic; it plugs into the same pipeline
// (eval -> update -> eval -> observations).
constexpr int GT_M = 64, GT_N = 64, GT_K = 16, GT_LD = 68;

// C(m,n) = sum_k A(m,k) * B(k,n) with A(m,k) = A[m*am + k*ak], B(k,n) = Bm[k*bk + n*bn]
template <class Epi>
__device__ void gemm_tiled(int M, int N, int K, const float *A, long am, long ak, const float *Bm,
                           long bk, long bn, float *smA, float *smB, Epi epi) {
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    for (int m0 = 0; m0 < M; m0 += GT_M) {
        for (int n0 = 0; n0 < N; n0 += GT_N) {
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
            f32x2 acc2[4][2];
#pragma unroll
            for (int i = 0; i < 4; ++i) acc2[i][0] = acc2[i][1] = 0ull;
            // the global loads of K step k0 + GT_K are in flight while step k0 is multiplied
            float ra[4], rb[4];
            auto fetch = [&](int k0) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int i = tid + j * 256;
                    int mm, kk;
                    if (ak == 1) { kk = i & 15; mm = i >> 4; } else { mm = i & 63; kk = i >> 6; }
                    const int m = m0 + mm, k = k0 + kk;
                    ra[j] = (m < M && k < K) ? A[m * am + k * ak] : 0.f;
                    int nn, kb;
                    if (bn == 1) { nn = i & 63; kb = i >> 6; } else { kb = i & 15; nn = i >> 4; }
                    const int n = n0 + nn, k2 = k0 + kb;
                    rb[j] = (n < N && k2 < K) ? Bm[k2 * bk + n * bn] : 0.f;
                }
            };
            fetch(0);
            for (int k0 = 0; k0 < K; k0 += GT_K) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int i = tid + j * 256;
                    int mm, kk;
                    if (ak == 1) { kk = i & 15; mm = i >> 4; } else { mm = i & 63; kk = i >> 6; }
                    smA[kk * GT_LD + mm] = ra[j];
                    int nn, kb;
                    if (bn == 1) { nn = i & 63; kb = i >> 6; } else { kb = i & 15; nn = i >> 4; }
                    smB[kb * GT_LD + nn] = rb[j];
                }
                __syncthreads();
                if (k0 + GT_K < K) fetch(k0 + GT_K);
#pragma unroll
                for (int kk = 0; kk < GT_K; ++kk) {
                    const float4 a4 = *reinterpret_cast<const float4 *>(smA + kk * GT_LD + ty * 4);
                    const ulonglong2 b2 = *reinterpret_cast<const ulonglong2 *>(smB + kk * GT_LD + tx * 4);
                    const float av[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {                  // packed FMAs over column pairs
                        const f32x2 a2 = pack2(av[i], av[i]);
                        ffma2(acc2[i][0], a2, b2.x);
                        ffma2(acc2[i][1], a2, b2.y);
                    }
                }
                __syncthreads();
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                unpack2(acc2[i][0], acc[i][0], acc[i][1]);
                unpack2(acc2[i][1], acc[i][2], acc[i][3]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
                    if (m < M && n < N) epi(m, n, acc[i][j]);
                }
        }
    }
}

__global__ void __launch_bounds__(256, 2) gen_eval_kernel(const __grid_constant__ Dev d,
                                                       const __grid_constant__ StepArgs a) {
    __shared__ __align__(16) float smA[GT_K * GT_LD];
    __shared__ __align__(16) float smB[GT_K * GT_LD];
    __shared__ double red[8];
    __shared__ float misc[8];
    const int tid = threadIdx.x, nt = blockDim.x;
    const int L = d.nlayers, B = d.B, C = d.C;
    float *ws = d.ws + (size_t)blockIdx.x * d.ws_stride;
    const int e_end = a.e_begin + a.e_count;
    for (int e = a.e_begin + blockIdx.x; e < e_end; e += gridDim.x) {
        if (a.mode == MODE_RESET && a.mask != nullptr && !a.mask[e]) continue;
        EnvScalars *sc = d.sc + e;
        float *wE = d.w + (size_t)e * d.Pp;
        const bool lrs = d.env_kind == B2E_ENV_MULTIOPTLRS;
        __syncthreads();
        if (a.mode == MODE_RESET) {                                   // base_reset
            if (d.index_mode == B2E_INDEX_INTERNAL) {
                shuffle_order(d, e, sc);                              // optimize_nn.py:114-120
                if (tid == 0) sc->cursor = 0;
                __syncthreads();
            }
            const int episode = sc->episode;
            for (int l = 0; l < L; ++l) {                             // keras Dense defaults
                const int nin = d.dims[l], nout = d.dims[l + 1];
                const float limit = sqrtf(6.0f / (float)(nin + nout));
                const int lo = d.woff[l], hi = d.boff[l] + nout;
                for (int p = lo + tid; p < hi; p += nt) {
                    float v = 0.f;
                    if (a.init_params) v = a.init_params[(size_t)e * d.P + p];
                    else if (p < d.boff[l]) v = glorot(d.seed, e + d.env_base, episode, p, limit);
                    if (d.w2) d.w2[(size_t)e * d.Pp + p] = wE[p];
                    wE[p] = v;
                }
            }
            __syncthreads();
        }
        const int *idx; int cnt;
        current_batch(d, a, e, sc, idx, cnt);
        // ---- inputs
        float *act0 = ws + d.aoff[0];
        for (int i = tid; i < B * d.D; i += nt) {
            const int s = i / d.D, k = i - s * d.D;
            act0[i] = s < cnt ? d.X[(size_t)idx[s] * d.Dp + k] : 0.f;
        }
        __syncthreads();
        // ---- forward (problems/optimize_nn.py:35-44)
        for (int l = 0; l < L; ++l) {
            const int nin = d.dims[l], nout = d.dims[l + 1];
            const float *in = ws + d.aoff[l];
            float *out = ws + d.aoff[l + 1];
            const float *Wl = wE + d.woff[l], *bl = wE + d.boff[l];
            const bool relu = l + 1 < L;
            gemm_tiled(B, nout, nin, in, nin, 1, Wl, nout, 1, smA, smB,
                       [&](int m, int n, float v) {
                           v += bl[n];
                           out[(size_t)m * nout + n] = relu ? fmaxf(v, 0.f) : v;
                       });
            __syncthreads();
        }
        // ---- softmax cross-entropy per sample (:47), delta of the logits
        float *dl = ws + d.doff0;
        const float *Z = ws + d.aoff[L];
        double lsum = 0.0;
        for (int s = tid; s < B; s += nt) {
            float *dz = dl + (size_t)s * C;
            if (s < cnt) {
                const float *z = Z + (size_t)s * C;
                const int y = d.labels[idx[s]];
                float m = z[0];
                for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
                float sum = 0.f;
                for (int c = 0; c < C; ++c) sum += expf(z[c] - m);
                lsum += (double)((m + logf(sum)) - z[y]);
                const float inv = 1.0f / sum;
                for (int c = 0; c < C; ++c) dz[c] = expf(z[c] - m) * inv - (c == y ? 1.f : 0.f);
            } else {
                for (int c = 0; c < C; ++c) dz[c] = 0.f;
            }
        }
        const float loss = (float)(block_sum(lsum, red) / (double)cnt);     // reduce_mean (:50)
        // ---- backward: gradient of the batch SUM (:49)
        float *gdst;
        if (a.mode == MODE_RESET) gdst = d.gprev + (size_t)e * d.Pp;
        else if (a.mode == MODE_EVAL) gdst = a.grad_out + (size_t)e * d.P;
        else gdst = d.gnext + (size_t)e * d.Pp;
        float *g2E = (a.mode == MODE_RESET && d.g2) ? d.g2 + (size_t)e * d.Pp : nullptr;
        float gpart = 0.f;
        for (int l = L - 1; l >= 0; --l) {
            const int nin = d.dims[l], nout = d.dims[l + 1];
            const float *in = ws + d.aoff[l];
            float *gW = gdst + d.woff[l], *gb = gdst + d.boff[l];
            const int wo = d.woff[l], bo = d.boff[l];
            // kernel gradient: in^T . delta
            gemm_tiled(nin, nout, B, in, 1, nin, dl, nout, 1, smA, smB,
                       [&](int m, int n, float v) {
                           const int p = m * nout + n;
                           if (g2E) g2E[wo + p] = gW[p];
                           gW[p] = v;
                           gpart += v;
                       });
            for (int j = tid; j < nout; j += nt) {
                float g = 0.f;
                for (int s = 0; s < cnt; ++s) g += dl[(size_t)s * nout + j];
                if (g2E) g2E[bo + j] = gb[j];
                gb[j] = g;
                gpart += g;
            }
            if (l > 0) {                                              // delta of the layer below
                float *dn = ws + (dl == ws + d.doff0 ? d.doff1 : d.doff0);
                const float *Wl = wE + d.woff[l];
                gemm_tiled(B, nin, nout, dl, nout, 1, Wl, 1, nout, smA, smB,
                           [&](int m, int n, float v) {
                               dn[(size_t)m * nin + n] = in[(size_t)m * nin + n] > 0.f ? v : 0.f;
                           });
                dl = dn;
            }
            __syncthreads();
        }
        const double gsum = block_sum((double)gpart, red);
        // ---- what the caller asked for
        if (a.mode == MODE_EVAL) {
            if (tid == 0) a.loss_out[e] = loss;
        } else if (a.mode == MODE_EVAL_STEP) {
            if (tid == 0) step_scalars(d, a, sc, e, loss, gsum, misc);
            __syncthreads();
            const bool wrap = misc[4] != 0.f;
            __syncthreads();
            if (wrap) shuffle_order(d, e, sc);
        } else if (a.mode == MODE_RESET) {
            if (tid == 0) {
                if (lrs) {
                    for (int i = 0; i < RAW_DEPTH; ++i) { sc->raw_loss[i] = 0.f; sc->raw_gsum[i] = 0.0; }
                    sc->raw_pos = 0;
                } else {
                    sc->raw_pos = (sc->raw_pos + 1) % RAW_DEPTH;
                }
                for (int i = 0; i < B2E_MAX_HISTORY; ++i) sc->adj_loss[i] = 0.f;
                sc->raw_loss[sc->raw_pos] = loss;
                sc->raw_gsum[sc->raw_pos] = gsum;
                sc->loss_prev = loss;
                sc->head = d.H - 1;
                sc->nvalid = 0;
                sc->step = 0;
                sc->episode = sc->episode + 1;
            }
            if (a.obs) {
                float *o = a.obs + (size_t)e * d.P * d.OD;
                const size_t n = (size_t)d.P * d.OD;
                const float fill = lrs ? -1.0f : 0.0f;
                for (size_t i = tid; i < n; i += nt) o[i] = fill;
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------ utility kernels
__global__ void pad_rows_kernel(const float *src, float *dst, int n, int dcols, int dpad) {
    const size_t total = (size_t)n * dpad;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total;
         i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / dpad;
        const int c = (int)(i - r * dpad);
        dst[i] = c < dcols ? src[r * dcols + c] : 0.f;
    }
}

__global__ void init_order_kernel(int *ord, const int *init, int e_count, int n) {
    const size_t total = (size_t)e_count * n;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total;
         i += (size_t)gridDim.x * blockDim.x)
        ord[i] = init ? init[i] : (int)(i % n);
}

// ring <-> newest-first conversion for b2e_get_state / b2e_set_state
__global__ void ring_copy_kernel(Dev d, int which, float *user, int to_user) {
    const int e = blockIdx.x;
    EnvScalars *sc = d.sc + e;
    const int H = d.H;
    if (which == B2E_STATE_ADJ_LOSSES) {
        for (int h = threadIdx.x; h < H; h += blockDim.x) {
            int slot = sc->head - h; slot += slot < 0 ? H : 0;
            if (to_user) user[(size_t)e * H + h] = h < sc->nvalid ? sc->adj_loss[slot] : 0.f;
            else sc->adj_loss[slot] = user[(size_t)e * H + h];
        }
        return;
    }
    float *ring = (which == B2E_STATE_ADJ_WEIGHTS ? d.ringw : d.ringg) + (size_t)e * H * d.Pp;
    for (int h = 0; h < H; ++h) {
        int slot = sc->head - h; slot += slot < 0 ? H : 0;
        float *u = user + ((size_t)e * H + h) * d.P;
        for (int p = threadIdx.x; p < d.P; p += blockDim.x) {
            if (to_user) u[p] = h < sc->nvalid ? ring[(size_t)slot * d.Pp + p] : 0.f;
            else ring[(size_t)slot * d.Pp + p] = u[p];
        }
    }
}

__global__ void scalars_copy_kernel(Dev d, int which, void *user, int to_user) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= d.E) return;
    EnvScalars *sc = d.sc + e;
    if (which == B2E_STATE_RAW_LOSSES || which == B2E_STATE_RAW_GSUMS) {
        for (int i = 0; i < RAW_DEPTH; ++i) {
            int slot = sc->raw_pos - i; slot += slot < 0 ? RAW_DEPTH : 0;
            if (which == B2E_STATE_RAW_LOSSES) {
                float *u = (float *)user + (size_t)e * RAW_DEPTH + i;
                if (to_user) *u = sc->raw_loss[slot];
                else { sc->raw_loss[slot] = *u; if (i == 0) sc->loss_prev = *u; }
            } else {
                double *u = (double *)user + (size_t)e * RAW_DEPTH + i;
                if (to_user) *u = sc->raw_gsum[slot]; else sc->raw_gsum[slot] = *u;
            }
        }
    } else if (which == B2E_STATE_STEP) {
        int *u = (int *)user + e;
        if (to_user) *u = sc->step; else sc->step = *u;
    } else if (which == B2E_STATE_CURSOR) {
        int *u = (int *)user + e;
        if (to_user) *u = sc->cursor; else sc->cursor = *u;
    }
}

// marks every adjusted-history slot valid (after b2e_set_state of a history)
__global__ void set_nvalid_kernel(Dev d, int nvalid) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < d.E) d.sc[e].nvalid = nvalid;
}

__global__ void strided_copy_kernel(float *state, float *user, int e_count, int p, int pp,
                                    int to_user) {
    const size_t total = (size_t)e_count * p;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total;
         i += (size_t)gridDim.x * blockDim.x) {
        const size_t e = i / p, c = i - e * p;
        if (to_user) user[i] = state[e * pp + c]; else state[e * pp + c] = user[i];
    }
}

__global__ void order_copy_kernel(Dev d, int *user, int to_user) {
    const int e = blockIdx.x;
    int *cur = d.ord + ((size_t)d.sc[e].ord_sel * d.E + e) * d.N;
    for (int i = threadIdx.x; i < d.N; i += blockDim.x) {
        if (to_user) user[(size_t)e * d.N + i] = cur[i]; else cur[i] = user[(size_t)e * d.N + i];
    }
}

__global__ void batch_indices_kernel(Dev d, int *idx_out, int *cnt_out) {
    const int e = blockIdx.x;
    const EnvScalars *sc = d.sc + e;
    const int lo = sc->cursor * d.B;
    const int cnt = min(d.B, d.N - lo);
    const int *cur = d.ord + ((size_t)sc->ord_sel * d.E + e) * d.N + lo;
    for (int r = threadIdx.x; r < d.B; r += blockDim.x) idx_out[(size_t)e * d.B + r] = r < cnt ? cur[r] : 0;
    if (threadIdx.x == 0) cnt_out[e] = cnt;
}

// BaseProblem.next() for the masked envs (problems/optimize_nn.py:102-112)
__global__ void next_batch_kernel(Dev d, const unsigned char *mask) {
    const int e = blockIdx.x;
    if (mask && !mask[e]) return;
    EnvScalars *sc = d.sc + e;
    __shared__ int wrap;
    if (threadIdx.x == 0) {
        const int cur = sc->cursor + 1;
        wrap = cur * d.B >= d.N;
        sc->cursor = wrap ? 0 : cur;
    }
    __syncthreads();
    if (wrap) shuffle_order(d, e, sc);
}

__global__ void init_scalars_kernel(Dev d) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= d.E) return;
    EnvScalars *sc = d.sc + e;
    memset(sc, 0, sizeof(EnvScalars));
    sc->head = d.H - 1;
}

thread_local std::string g_create_error;

}  // namespace

// =============================================================== host side / C ABI
struct b2e_env {
    b2e_config cfg;
    Dev d;
    int nthreads, grid, num_sms;
    size_t smem_bytes;
    float *X, *targets_f;
    int *labels, *ord, *perm, *row_of_param, *param_of_row;
    float *w, *gprev, *gnext, *ringw, *ringg;
    double *part;
    EnvScalars *sc;
    size_t smem_obs;
    int chunk_envs, obs_grid;
    bool use_eval_kernel;            // first layer fits the streamed-operand eval kernel
    bool eval_c;                     // eval_kernel instantiated for N1 = 64, KT = 112 (config 4)
    bool fuse_update;                // first eval applies the update itself (eval_bulk_kernel<false, true>; opt-in with B2E_FUSE_UPDATE=1)
    bool eval_bulk;                  // ... and its bulk-copy / mbarrier pipelined form (B2E_EVAL_BULK=0 disables)
    int nchunks, eval_ctas_per_sm;   // B2E_CHUNKS experiment
    bool use_thin;                   // softmax regression: thin_eval_kernel
    bool thin_fused;                 // ... whose cluster form runs eval / update / eval of a MultiOptLRs step as ONE launch (opt-in: B2E_THIN_FUSE=1)
    bool use_thin2;                  // ... its shared-memory-resident successor for 10 classes (b200thin.cu; B2E_THIN2=0 disables)
    size_t smem_thin;
    int thin_kc;
    bool use_tc;                     // tcgen05 eval kernel replaces eval_kernel
    Dev d_tc;                        // Dev with the tensor-core kernel's shared-memory layout
    size_t smem_tc;
    int tc_grid;
    bool use_tc2;                    // warp-specialised tcgen05 eval kernel (b200tc.cu)
    b2e_tc2_ctx *tc2;                // its context: tensor map, watchdog word, grid
    bool tc2_check;                  // B2E_TC_CHECK=1: synchronise and test the watchdog after every step
    float *w2, *g2, *ws;
    int obs_stages, obs_regs, obs_bulk;        // obs_kernel2 variant (0 stages = obs_kernel)
    size_t smem_obs2;
    Dev d_eval;                      // Dev with the eval kernel's shared-memory layout
    size_t smem_eval;
    int eval_grid;
    double *part_u;
    int *reset_list, *reset_count;   // reset pipeline of the tcgen05 path: work list, its length, losses of the reset evals
    float *reset_loss;
    bool reset_pipeline;
    bool use_tiny;                   // warp-per-env kernel for tiny problems (b200tiny.cu; B2E_TINY=0 disables)
    double *part_r, *slot_abs;       // ring-only steps: ring_adjg_kernel's partial sums, per-slot sums of |adjusted x|
    cudaStream_t side;               // the observation kernel runs here (lowest priority) ...
    cudaStream_t hi;                 // ... next to the compute kernel (highest priority)
    cudaEvent_t ev_fork, ev_join;
    cudaEvent_t ev_chunk[64];
    bool dataset_bound, stream_bound;
    bool trace;                      // record per-kernel events in b2e_step
    cudaEvent_t tr[8];
    int tr_count;
    int64_t launches;
    std::string error;
};

namespace {

int fail(b2e_handle h, const std::string &msg) {
    if (h) h->error = msg; else g_create_error = msg;
    return 1;
}

#define CUDA_TRY(h, expr)                                                             \
    do {                                                                              \
        cudaError_t err__ = (expr);                                                   \
        if (err__ != cudaSuccess)                                                     \
            return fail(h, std::string(#expr) + ": " + cudaGetErrorString(err__));    \
    } while (0)

int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Every entry point runs on the handle's device whatever the caller's current device is, and
// leaves the caller's device selected afterwards.
struct DeviceGuard {
    int prev;
    bool switched;
    explicit DeviceGuard(int device) : prev(-1), switched(false) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != device) switched = cudaSetDevice(device) == cudaSuccess;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

int pow2_ceil(int v) { int p = 1; while (p < v) p <<= 1; return p; }

std::string lex_rows(int num_params, int *row_of_param_host) {
    // row of parameter p = rank of the string "%d" % p among 0..P-1 (DFS over the digit trie
    // enumerates them in lexicographic order).
    int next_row = 0;
    struct Frame { long long v; int digit; };
    Frame *stack = new (std::nothrow) Frame[16];
    if (!stack) return "out of memory";
    // iterative pre-order: roots are 0..9 ("0" has no children)
    for (int root = 0; root <= 9 && root < num_params; ++root) {
        int depth = 0;
        stack[0] = {root, 0};
        row_of_param_host[root] = next_row++;
        if (root == 0) continue;
        while (depth >= 0) {
            Frame &f = stack[depth];
            if (f.digit > 9) { --depth; continue; }
            const long long child = f.v * 10 + f.digit;
            ++f.digit;
            if (child >= num_params) { f.digit = 10; continue; }
            row_of_param_host[child] = next_row++;
            stack[++depth] = {child, 0};
        }
    }
    delete[] stack;
    return next_row == num_params ? "" : "internal error in lexicographic row table";
}

const void *obs2_fn(int stages, int regs, int bulk) {
    if (regs) {
        switch (regs * 2 + (bulk ? 1 : 0)) {
            case 2: return (const void *)obs_kernel3<5, 1, false>;
            case 3: return (const void *)obs_kernel3<5, 1, true>;
            case 4: return (const void *)obs_kernel3<5, 2, false>;
            case 5: return (const void *)obs_kernel3<5, 2, true>;
            case 8: return (const void *)obs_kernel3<5, 4, false>;
            default: return (const void *)obs_kernel3<5, 4, true>;
        }
    }
    switch (stages * 2 + (bulk ? 1 : 0)) {
        case 6: return (const void *)obs_kernel2<5, 3, false>;
        case 7: return (const void *)obs_kernel2<5, 3, true>;
        case 8: return (const void *)obs_kernel2<5, 4, false>;
        case 9: return (const void *)obs_kernel2<5, 4, true>;
        case 12: return (const void *)obs_kernel2<5, 6, false>;
        default: return (const void *)obs_kernel2<5, 6, true>;
    }
}

int configure(b2e_handle h) {
    const b2e_config &c = h->cfg;
    Dev &d = h->d;
    memset(&d, 0, sizeof(d));
    d.env_kind = c.env_kind;
    d.kind = c.problem_kind;
    d.hidden = c.num_hidden > 0;
    d.E = c.num_envs; d.H = c.max_history; d.max_batches = c.max_batches;
    d.act_ver = c.action_version; d.rew_ver = c.reward_version; d.obs_ver = c.observation_version;
    d.row_lex = c.row_order == B2E_ROWS_LEXICOGRAPHIC;
    d.index_mode = c.index_mode; d.auto_reset = c.auto_reset; d.seed = c.init_seed; d.env_base = c.env_base;
    if (d.kind == B2E_PROBLEM_FUNC) {
        d.D = 0; d.N1 = 8; d.C = 0; d.N = 0; d.B = 1; d.P1 = 0; d.tailP = 2; d.P = 2;
    } else {
        d.D = c.num_features; d.C = c.num_outputs; d.N = c.num_rows; d.B = c.batch_size;
        d.N1 = d.hidden ? c.num_hidden : d.C;
        d.P1 = d.D * d.N1;
        d.tailP = d.hidden ? d.N1 + d.N1 * d.C + d.C : d.C;
        d.P = d.P1 + d.tailP;
        d.lim1 = sqrtf(6.0f / (float)(d.D + d.N1));
        d.lim2 = d.hidden ? sqrtf(6.0f / (float)(d.N1 + d.C)) : 0.f;
    }
    // dense stack of the classifier; more than one hidden layer (or a shape the fused kernels
    // cannot hold) runs the generic pipeline
    int nhid = 0;
    if (d.kind != B2E_PROBLEM_FUNC) {
        d.dims[0] = d.D;
        if (c.num_hidden > 0) {
            d.dims[++nhid] = c.num_hidden;
            for (int i = 0; i < B2E_MAX_LAYERS - 2 && c.hidden_more[i] > 0; ++i) d.dims[++nhid] = c.hidden_more[i];
        }
        d.dims[nhid + 1] = d.C;
        d.nlayers = nhid + 1;
        int p = 0;
        for (int l = 0; l < d.nlayers; ++l) {
            d.woff[l] = p; p += d.dims[l] * d.dims[l + 1];
            d.boff[l] = p; p += d.dims[l + 1];
        }
        const char *force = getenv("B2E_FORCE_GENERIC");
        d.generic = (nhid > 1 || (force && atoi(force) != 0 && d.kind == B2E_PROBLEM_SOFTMAX)) ? 1 : 0;
        if (d.generic) d.P = p;
    }
    d.Pp = round_up(d.P, 4);
    d.col_w = 0; d.col_l = d.H; d.col_g = 2 * d.H;
    d.OD = 3 * d.H;
    if (c.env_kind == B2E_ENV_MULTIOPTIMIZE) {                 // utils/utils_env.py:22-44
        const int hv = c.history_version;
        if (hv == 0 || hv == 2) d.H = 1;                       // History(1, ...)
        const bool has_w = hv == 2 || hv == 3, has_l = hv == 1 || hv == 2 || hv == 3;
        int col = 0;
        d.col_w = has_w ? col : -1; col += has_w ? d.H : 0;
        d.col_l = has_l ? col : -1; col += has_l ? d.H : 0;
        d.col_g = col; col += d.H;
        d.OD = col;
    }
    d.Dp = round_up(d.D, 4);
    d.Ds = d.Dp;
    if (d.Ds > 0 && ((d.Ds >> 2) & 1) == 0) d.Ds += 4;       // odd number of float4 per row
    d.N1p = round_up(d.N1, 8);
    d.Cp = round_up(d.C > 0 ? d.C : 1, 4);
    // backward decomposition: lane = column, N1g columns per lane group, 8 rows per lane
    d.N1g = d.N1 >= 32 ? 32 : pow2_ceil(d.N1);
    d.KR = 8 * (32 / d.N1g);
    d.gcc = d.N1 > 32 ? (d.N1 + 31) / 32 : 1;
    d.KT = d.KR > 64 ? d.KR : 64;
    d.ntiles = d.D > 0 ? (d.D + d.KT - 1) / d.KT : 0;
    // register-tiled path: N1/8 column groups must tile the 256-thread CTA
    d.cg = d.N1 / 8;
    d.fast = (d.kind != B2E_PROBLEM_FUNC && d.N1 % 8 == 0 && d.cg >= 4 && d.cg <= 32 &&
              256 % d.cg == 0 && d.B <= 32 && (long long)d.P >= 4096) ? 1 : 0;
    if (d.fast) {
        const int rows_max = 4 * (256 / d.cg);                 // tile rows one backward pass covers
        d.ntiles = (d.D + rows_max - 1) / rows_max;
        d.KT = round_up((d.D + d.ntiles - 1) / d.ntiles, 4);   // e.g. D = 784 -> 7 tiles of 112 rows
    }
    // threads: small problems use small CTAs so that several fit one SM
    const long long work = (long long)d.P;
    h->nthreads = work >= 4096 ? 256 : (work >= 512 ? 128 : 64);
    int nw = h->nthreads / 32;
    // forward decomposition
    d.nsc = (d.B + 31) / 32;
    d.ncc = d.N1p / 8;
    while (d.nsc * d.ncc > nw * MAXI && h->nthreads < 256) { h->nthreads *= 2; nw *= 2; }
    if (d.nsc * d.ncc > nw * MAXI) {
        if (d.kind != B2E_PROBLEM_SOFTMAX)
            return fail(h, "batch_size x layer width too large for the fused kernel "
                           "(need ceil(B/32) * ceil(N1/8) <= 32)");
        d.generic = 1;
    }
    d.nks = 1;
    while (d.nsc * d.ncc * d.nks * 2 <= nw && d.KT / (d.nks * 2) >= 4 && !d.fast) d.nks *= 2;
    d.fitems = d.nsc * d.ncc * d.nks;
    if (d.fast) d.nks = 256 / (8 * d.cg);                      // K slices of the fast forward
    // large problems run as a pipeline of kernels (eval / update / eval / observations)
    h->use_eval_kernel = d.fast && d.nks * d.B * d.N1p <= 2 * round_up(d.KT, 4) * d.N1p;
    if (d.generic) { h->use_eval_kernel = false; d.fast = 0; }
    int thin_kc = 0;                                           // largest chunk <= 128 with KC*C % 4 == 0, dividing D if possible
    for (int k = THIN_KC; k >= 8 && !thin_kc; k -= 4)
        if ((k * d.C) % 4 == 0 && d.D % k == 0) thin_kc = k;
    if (!thin_kc) thin_kc = (d.C % 4 == 0) ? THIN_KC : ((d.C % 2 == 0) ? THIN_KC : THIN_KC);
    h->smem_thin = (size_t)(THIN_STAGES * d.B * (thin_kc + 4) + (THIN_STAGES + 2) * thin_kc * d.C + d.B * THIN_CMAX + d.B + THIN_CMAX + 8) * sizeof(float);
    h->use_thin = !d.generic && !h->use_eval_kernel && d.kind == B2E_PROBLEM_SOFTMAX && !d.hidden &&
                  d.C <= THIN_CMAX && d.B <= 32 && d.P >= 4096 && (thin_kc * d.C) % 4 == 0 && d.D % 4 == 0;
    h->thin_kc = thin_kc;
    d.split = (c.env_kind == B2E_ENV_MULTIOPTIMIZE || h->use_eval_kernel || h->use_thin || d.generic) ? 1 : 0;
    // shared memory carve-up (float offsets, all multiples of 4)
    d.xslack = round_up(d.KR + 8, 4) > 64 ? round_up(d.KR + 8, 4) : 64;
    int off = d.B * d.Ds + d.xslack;
    d.off_T = off; off += round_up(d.KT, 4) * d.N1p;
    d.off_T2 = off; off += d.fast ? round_up(d.KT, 4) * d.N1p : 0;
    d.off_H = off; off += round_up(d.B * d.N1p, 4);
    d.off_dP = off; off += round_up(d.B * d.N1p, 4);
    d.off_tw = off; off += round_up(d.tailP, 4);
    d.off_tg = off; off += round_up(d.tailP, 4);
    d.off_Z = off; off += d.hidden ? round_up(d.B * d.Cp, 4) : 0;
    const int red_floats = 2 * NSTAT * 16;
    const int fred = d.nks > 1 ? d.nks * d.B * d.N1p : 0;
    if (d.fast && fred <= 2 * round_up(d.KT, 4) * d.N1p) {
        d.off_red = d.off_T;            // tiles are idle when the forward partials are reduced ...
        d.off_red2 = off; off += red_floats;                       // ... the statistics scratch is not
    } else {
        d.off_red = off; off += round_up(fred > red_floats ? fred : red_floats, 4);
        d.off_red2 = d.off_red;
    }
    // large problems: compute kernel + streaming observation kernel (see DESIGN.md)
    d.nseg = (d.P + SEG_ROWS - 1) / SEG_ROWS;
    d.stage_stride = round_up(SPAN_CAP * d.OD + 8, 4);
    d.off_stage = off; off += d.split ? 0 : nw * d.stage_stride;
    d.off_rows = off; off += d.split ? 0 : nw * (128 + SPAN_CAP);
    d.off_idx = off; off += round_up(d.B, 4);
    d.off_y = off; off += round_up(d.B * (d.kind == B2E_PROBLEM_LINREG ? d.C : 1), 4);
    d.off_lb = off; off += round_up(d.B, 4);
    d.off_misc = off; off += 8 + 2 * B2E_MAX_HISTORY;
    h->smem_bytes = (size_t)off * sizeof(float);
    if (!d.generic && h->smem_bytes > 227 * 1024 && d.kind == B2E_PROBLEM_SOFTMAX) {
        d.generic = 1; d.fast = 0; d.split = 1;               // does not fit the fused kernel
        h->use_eval_kernel = h->use_thin = false;
    }
    if (d.generic) {
        h->smem_bytes = 0;
        int maxw = 0, o = 0;
        for (int l = 0; l <= d.nlayers; ++l) {
            d.aoff[l] = o; o += round_up(d.B * d.dims[l], 4);
            if (l > 0 && d.dims[l] > maxw) maxw = d.dims[l];
        }
        d.doff0 = o; o += round_up(d.B * maxw, 4);
        d.doff1 = o; o += round_up(d.B * maxw, 4);
        d.ws_stride = o;
    }
    {   // observation kernel variant: B2E_OBS = "<stages><b|s>" (cp.async gathers, e.g. "4b"),
        // "r<rows><b|s>" (register-batched gathers, e.g. "r4b"), "0" = obs_kernel;
        // b = cp.async.bulk row-block stores, s = 16-byte stores
        const char *v = getenv("B2E_OBS");
        h->obs_stages = 0; h->obs_regs = 4; h->obs_bulk = 1;
        if (v && *v) {
            h->obs_bulk = strchr(v, 's') ? 0 : 1;
            if (*v == 'r') { h->obs_regs = atoi(v + 1); h->obs_stages = 0; }
            else { h->obs_stages = atoi(v); h->obs_regs = 0; }
        }
        if (h->obs_stages != 0 && h->obs_stages != 3 && h->obs_stages != 4 && h->obs_stages != 6)
            return fail(h, "B2E_OBS: stages must be 0, 3, 4 or 6");
        if (h->obs_regs != 0 && h->obs_regs != 1 && h->obs_regs != 2 && h->obs_regs != 4)
            return fail(h, "B2E_OBS: rows per lane must be 1, 2 or 4");
        if (d.H != 5 || !d.split || c.env_kind != B2E_ENV_MULTIOPTLRS) h->obs_stages = h->obs_regs = 0;
        if (h->obs_stages || h->obs_regs) {
            // warp items of 32 units; small batches (BASELINE config 3: 8192 such items = 3.5 waves of the 296 resident
            // CTAs) get 8-unit items, so that the last wave is 1/14 instead of 1/4 of the kernel
            const int nblk = (d.P + 31) / 32;
            const long long items32 = (long long)d.E * ((nblk + O2_UNITS - 1) / O2_UNITS);
            d.obs_units = items32 < 8LL * 2 * O2_WARPS * h->num_sms ? 8 : O2_UNITS;
            d.nseg = (nblk + d.obs_units - 1) / d.obs_units;
            const int npl1 = 2 * d.H + 2, stg = 32 * d.OD + 8;
            h->smem_obs2 = (size_t)O2_WARPS * (h->obs_stages * npl1 * 32 + (h->obs_bulk ? 2 : 1) * stg) * sizeof(float);
        }
    }
    h->smem_obs = (size_t)(B2E_MAX_HISTORY + OBS_WARPS * (32 * d.OD + 8)) * sizeof(float);
    d.nsegU = (d.Pp + UPD_SEG - 1) / UPD_SEG;
    {   // eval kernel: X and W1 both streamed through double-buffered tiles
        h->d_eval = d;
        Dev &v = h->d_eval;
        const int kt4 = round_up(d.KT, 4);
        v.ev_XS = ((kt4 >> 2) & 1) ? kt4 : kt4 + 4;              // odd number of float4 per row
        int o = 0;
        v.ev_X0 = o; o += d.B * v.ev_XS;
        v.ev_X1 = o; o += d.B * v.ev_XS;
        v.ev_W0 = o; o += kt4 * d.N1p;
        v.ev_W1 = o; o += kt4 * d.N1p;
        v.off_T = v.ev_W0; v.off_T2 = v.ev_W1;
        v.off_red = v.ev_W0;                                     // forward partials: W tiles are idle then
        v.off_H = o; o += round_up(d.B * d.N1p, 4);
        v.off_dP = o; o += round_up(d.B * d.N1p, 4);
        v.off_tw = o; o += round_up(d.tailP, 4);
        v.off_tg = o; o += round_up(d.tailP, 4);
        v.off_Z = o; o += d.hidden ? round_up(d.B * d.Cp, 4) : 0;
        v.off_red2 = o; o += 2 * NSTAT * 16;
        v.off_idx = o; o += round_up(d.B, 4);
        v.off_y = o; o += round_up(d.B * (d.kind == B2E_PROBLEM_LINREG ? d.C : 1), 4);
        v.off_lb = o; o += round_up(d.B, 4);
        v.off_misc = o; o += 8 + 2 * B2E_MAX_HISTORY;
        h->smem_eval = (size_t)o * sizeof(float);
        v.split = d.split;
    }
    {   // tensor-core eval kernel: operand stage first, then the float regions of the tail
        // opt-in (B2E_TC=1): parity-green, but in the step pipeline it is still slower than the FFMA
        // eval kernel (1.24 vs 1.12 ms at 4096 envs; profiles/r1_notes.md has the analysis)
        const char *tcv = getenv("B2E_TC");
        h->use_tc = h->use_eval_kernel && d.hidden && d.N1 == tc::N1 && d.N1p == tc::N1 && d.B == tc::B &&
                    d.D % tc::KT == 0 && d.kind == B2E_PROBLEM_SOFTMAX && tcv && atoi(tcv) != 0;
        h->d_tc = d;
        Dev &v = h->d_tc;
        // scratch that only lives between the two passes sits inside operand stage 1
        int in1 = tc::STAGE / 4;
        v.off_H = in1; in1 += round_up(d.B * d.N1p, 4);
        v.off_dP = in1; in1 += round_up(d.B * d.N1p, 4);
        v.off_Z = in1; in1 += d.hidden ? round_up(d.B * d.Cp, 4) : 0;
        v.off_lb = in1; in1 += round_up(d.B, 4);
        v.off_red2 = in1; in1 += 2 * NSTAT * 16;
        if (in1 > 2 * tc::STAGE / 4) h->use_tc = false;
        int o = tc::OPERAND_BYTES / 4;
        v.off_tw = o; o += round_up(d.tailP, 4);
        v.off_tg = o; o += round_up(d.tailP, 4);
        v.off_idx = o; o += round_up(d.B, 4);
        v.off_y = o; o += round_up(d.B, 4);
        v.off_misc = o; o += 8 + 2 * B2E_MAX_HISTORY;
        h->smem_tc = (size_t)o * sizeof(float);
    }
    return 0;
}

// base_reset of the envs in `mask` (null = all) through the tcgen05 eval kernel; see reset_list_kernel
int reset_through_pipeline(b2e_handle h, StepArgs a, void *stream) {
    Dev &d = h->d;
    const cudaStream_t cs = (cudaStream_t)stream;
    a.env_list = h->reset_list; a.env_count = h->reset_count; a.loss_out = h->reset_loss;
    a.e_begin = 0; a.e_count = d.E;
    reset_list_kernel<<<1, 1024, 0, cs>>>(a.mask, d.E, h->reset_list, h->reset_count);
    const int wide = d.E < 8 * h->num_sms ? d.E : 8 * h->num_sms;
    reset_prepare_kernel<<<wide, 256, 0, cs>>>(d, a);
    Dev dv = d;
    dv.gnext = d.gprev;                                       // the reset gradient is the newest raw-history entry
    if (b2e_tc2_launch(h->tc2, &dv, &a, 0, cs)) return fail(h, "tc2 launch failed (reset)");
    reset_finish_kernel<<<wide, 256, 0, cs>>>(d, a);
    h->launches += 4;
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

int launch(b2e_handle h, StepArgs args, void *stream) {
    if (args.mode == MODE_RESET && h->reset_pipeline) return reset_through_pipeline(h, args, stream);
    if (h->use_tiny && (args.mode == MODE_STEP || args.mode == MODE_RESET)) {
        if (args.e_count == 0) { args.e_begin = 0; args.e_count = h->d.E; }
        h->launches++;
        if (b2e_tiny_launch(&h->d, &args, stream)) return fail(h, "tiny kernel launch failed");
        return 0;
    }
    if (args.e_count == 0) { args.e_begin = 0; args.e_count = h->d.E; }
    const cudaStream_t cs = (cudaStream_t)stream;
    if (h->d.generic) {
        // MODE_RESET / MODE_EVAL / MODE_EVAL_STEP / MODE_EVAL_FIRST of the generic dense stack
        gen_eval_kernel<<<h->grid, 256, 0, cs>>>(h->d, args);
        h->launches++;
        CUDA_TRY(h, cudaGetLastError());
        return 0;
    }
    if (h->d.fast) {
        if (h->d.H == 5) optenv_kernel<5, true><<<h->grid, h->nthreads, h->smem_bytes, cs>>>(h->d, args);
        else optenv_kernel<0, true><<<h->grid, h->nthreads, h->smem_bytes, cs>>>(h->d, args);
    } else {
        if (h->d.H == 5) optenv_kernel<5, false><<<h->grid, h->nthreads, h->smem_bytes, cs>>>(h->d, args);
        else optenv_kernel<0, false><<<h->grid, h->nthreads, h->smem_bytes, cs>>>(h->d, args);
    }
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

}  // namespace

const void *b2e_dev_view(b2e_handle h, int *ring_ok, int *device) {
    if (!h) return nullptr;
    if (ring_ok) *ring_ok = (h->d.split && h->d.env_kind == B2E_ENV_MULTIOPTLRS && h->d.col_w == 0 && h->ringw && h->ringg) ? 1 : 0;
    if (device) *device = h->cfg.device;
    return &h->d;
}

extern "C" {

int b2e_abi_version(void) { return B2E_ABI_VERSION; }

const char *b2e_last_error(b2e_handle h) { return h ? h->error.c_str() : g_create_error.c_str(); }

int64_t b2e_launch_count(b2e_handle h) { return h ? h->launches : 0; }

int b2e_num_params(b2e_handle h) { return h ? h->d.P : -1; }

int b2e_obs_dim(b2e_handle h) { return h ? h->d.OD : -1; }

int b2e_history_depth(b2e_handle h) { return h ? h->d.H : -1; }

int b2e_create(const b2e_config *cfg, b2e_handle *out) {
    if (!cfg || !out) return fail(nullptr, "b2e_create: null argument");
    if (cfg->struct_size != (int32_t)sizeof(b2e_config))
        return fail(nullptr, "b2e_create: b2e_config.struct_size mismatch (ABI skew)");
    if (cfg->env_kind != B2E_ENV_MULTIOPTLRS && cfg->env_kind != B2E_ENV_MULTIOPTIMIZE)
        return fail(nullptr, "b2e_create: unknown env_kind");
    if (cfg->env_kind == B2E_ENV_MULTIOPTLRS && (cfg->history_version != 3 || cfg->observation_version != 3))
        return fail(nullptr, "b2e_create: MultiOptLRs is history_version 3 / observation_version 3 "
                             "(reference envs/multioptlrs.py:61)");
    // history version 5 exists in utils_env.py:38-42 but MultiOptimize cannot feed it
    // (History.append asserts on the missing 'weights' key, utils_common.py:183)
    if (cfg->env_kind == B2E_ENV_MULTIOPTIMIZE &&
        (cfg->history_version < 0 || cfg->history_version > 4 || cfg->observation_version < 0 ||
         cfg->observation_version > 3 || cfg->action_version > 1))
        return fail(nullptr, "b2e_create: bad history/observation/action version (RuntimeError in the reference)");
    if (cfg->action_version < 0 || cfg->action_version > 3 || cfg->reward_version < 0 ||
        cfg->reward_version > 6)
        return fail(nullptr, "b2e_create: bad action/reward version (RuntimeError in the reference)");
    if (cfg->problem_kind < 0 || cfg->problem_kind > 2) return fail(nullptr, "Not a name of a problem.");
    if (cfg->num_envs < 1 || cfg->max_history < 1 || cfg->max_history > B2E_MAX_HISTORY ||
        cfg->max_batches < 1)
        return fail(nullptr, "b2e_create: num_envs/max_history/max_batches out of range");
    if (cfg->problem_kind != B2E_PROBLEM_FUNC &&
        (cfg->num_features < 1 || cfg->num_outputs < 1 || cfg->num_rows < 1 || cfg->batch_size < 1 ||
         cfg->batch_size > cfg->num_rows || cfg->num_hidden < 0))
        return fail(nullptr, "b2e_create: bad problem shape");
    if (cfg->problem_kind == B2E_PROBLEM_LINREG && cfg->num_hidden != 0)
        return fail(nullptr, "b2e_create: linreg has no hidden layer");
    if (cfg->env_base < 0 || cfg->env_base > 0x7FFFFFFF - cfg->num_envs)
        return fail(nullptr, "b2e_create: env_base must be 0..2^31-1-num_envs");
    if (cfg->auto_reset && cfg->index_mode == B2E_INDEX_EXTERNAL && cfg->problem_kind != B2E_PROBLEM_FUNC)
        return fail(nullptr, "b2e_create: auto_reset needs the internal index stream");
    b2e_handle h = new (std::nothrow) b2e_env();
    if (!h) return fail(nullptr, "b2e_create: out of host memory");
    h->cfg = *cfg;
    h->launches = 0;
    h->nchunks = 1; h->eval_ctas_per_sm = 2; h->eval_c = false; h->eval_bulk = false;
    h->dataset_bound = h->stream_bound = false;
    h->trace = false; h->tr_count = 0;
    for (auto &ev : h->tr) ev = nullptr;
    h->X = h->targets_f = nullptr; h->labels = h->ord = h->perm = h->row_of_param = h->param_of_row = nullptr;
    h->w2 = h->g2 = h->ws = nullptr;
    h->use_tc2 = false; h->tc2 = nullptr; h->tc2_check = false;
    h->w = h->gprev = h->gnext = h->ringw = h->ringg = nullptr; h->sc = nullptr; h->part = nullptr; h->part_u = nullptr; h->part_r = nullptr; h->slot_abs = nullptr; h->reset_list = h->reset_count = nullptr; h->reset_loss = nullptr; h->reset_pipeline = false; h->use_tiny = false; h->use_thin2 = false; h->thin_fused = false;
    h->side = h->hi = nullptr; h->ev_fork = h->ev_join = nullptr;
    for (auto &ev : h->ev_chunk) ev = nullptr;
    auto bail = [&](const std::string &msg) { g_create_error = msg; b2e_destroy(h); return 1; };
    int dev_count = 0;
    if (cudaGetDeviceCount(&dev_count) != cudaSuccess || cfg->device < 0 || cfg->device >= dev_count)
        return bail("b2e_create: no such CUDA device");
    DeviceGuard guard(cfg->device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return bail("cudaGetDeviceProperties failed");
    h->num_sms = prop.multiProcessorCount;                  // configure sizes the observation kernel's work items with it
    if (configure(h)) return bail(h->error);
    if (h->smem_bytes > (size_t)prop.sharedMemPerBlockOptin)
        return bail("b2e_create: problem does not fit the fused kernel's shared memory (" +
                    std::to_string(h->smem_bytes) + " bytes needed)");
    const bool h5 = h->d.H == 5;
    const void *kernel_fn = h->d.fast
        ? (h5 ? (const void *)optenv_kernel<5, true> : (const void *)optenv_kernel<0, true>)
        : (h5 ? (const void *)optenv_kernel<5, false> : (const void *)optenv_kernel<0, false>);
    Dev &d = h->d;
    if (d.generic) {
        // per-CTA workspace of the generic dense stack; at most 4 GB of it
        const size_t ws_bytes = (size_t)d.ws_stride * sizeof(float);
        long long ctas = (long long)(((size_t)4 << 30) / ws_bytes);
        if (ctas < 1) ctas = 1;
        if (ctas > 2LL * h->num_sms) ctas = 2LL * h->num_sms;
        if (ctas > cfg->num_envs) ctas = cfg->num_envs;
        h->grid = (int)ctas;
        if (cudaMalloc((void **)&h->ws, ws_bytes * (size_t)ctas) != cudaSuccess)
            return bail("b2e_create: cudaMalloc of the dense-stack workspace failed (" +
                        std::to_string(ws_bytes * (size_t)ctas) + " bytes)");
    } else {
        if (cudaFuncSetAttribute(kernel_fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_bytes) != cudaSuccess)
            return bail("b2e_create: cudaFuncSetAttribute(smem) failed");
        int occ = 0;
        cudaError_t occ_err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel_fn, h->nthreads,
                                                                            h->smem_bytes);
        if (occ_err != cudaSuccess || occ < 1)
            return bail("b2e_create: kernel does not fit an SM");
        const long long resident = (long long)occ * h->num_sms;
        h->grid = (int)(cfg->num_envs < resident ? cfg->num_envs : resident);
    }
    const size_t EP = (size_t)d.E * d.Pp;
    auto dmalloc = [&](void **p, size_t bytes) { return cudaMalloc(p, bytes ? bytes : 16) == cudaSuccess; };
    if (!dmalloc((void **)&h->w, EP * 4) || !dmalloc((void **)&h->gprev, EP * 4) ||
        !dmalloc((void **)&h->ringw, EP * d.H * 4) || !dmalloc((void **)&h->ringg, EP * d.H * 4) ||
        !dmalloc((void **)&h->sc, (size_t)d.E * sizeof(EnvScalars)))
        return bail("b2e_create: cudaMalloc of env state failed");
    if (cfg->env_kind == B2E_ENV_MULTIOPTIMIZE && cfg->observation_version == 2) {
        if (!dmalloc((void **)&h->w2, EP * 4) || !dmalloc((void **)&h->g2, EP * 4))
            return bail("b2e_create: cudaMalloc of the raw-history planes failed");
        cudaMemset(h->w2, 0, EP * 4); cudaMemset(h->g2, 0, EP * 4);
    }
    if (d.split) {
        if (!dmalloc((void **)&h->gnext, EP * 4) ||
            !dmalloc((void **)&h->part, (size_t)d.E * d.nseg * 4 * sizeof(double)) ||
            !dmalloc((void **)&h->part_u, (size_t)d.E * d.nsegU * 4 * sizeof(double)))
            return bail("b2e_create: cudaMalloc of the split-path buffers failed");
        cudaMemset(h->gnext, 0, EP * 4);
        if (cfg->env_kind == B2E_ENV_MULTIOPTLRS) {          // ring-only steps (obs_out = NULL)
            if (!dmalloc((void **)&h->part_r, (size_t)d.E * d.nsegU * 4 * sizeof(double)) ||
                !dmalloc((void **)&h->slot_abs, (size_t)d.E * d.H * 2 * sizeof(double)))
                return bail("b2e_create: cudaMalloc of the ring-only buffers failed");
            cudaMemset(h->slot_abs, 0, (size_t)d.E * d.H * 2 * sizeof(double));
        }
        if (cudaFuncSetAttribute(mo_obs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_obs) != cudaSuccess)
            return bail("b2e_create: observation kernel does not fit (max_history too large)");
    }
    if (d.split) {
        if (cudaFuncSetAttribute(obs_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_obs) != cudaSuccess ||
            cudaFuncSetAttribute(obs_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_obs) != cudaSuccess)
            return bail("b2e_create: observation kernel does not fit (max_history too large)");
        if ((h->obs_stages || h->obs_regs) &&
            cudaFuncSetAttribute(obs2_fn(h->obs_stages, h->obs_regs, h->obs_bulk), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_obs2) != cudaSuccess)
            return bail("b2e_create: observation kernel (batched gathers) does not fit shared memory");
    }
    if (h->use_thin) {
        if (cudaFuncSetAttribute(thin_eval_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_thin) != cudaSuccess ||
            cudaFuncSetAttribute(thin_eval_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_thin) != cudaSuccess ||
            cudaFuncSetAttribute(thin_eval_kernel<false, 10>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_thin) != cudaSuccess ||
            cudaFuncSetAttribute(thin_eval_kernel<true, 10>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_thin) != cudaSuccess)
            return bail("b2e_create: thin eval kernel does not fit shared memory");
        int occ_ev = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_ev, thin_eval_kernel<true>, 256, h->smem_thin) !=
                cudaSuccess || occ_ev < 1)
            return bail("b2e_create: thin eval kernel does not fit an SM");
        h->eval_grid = occ_ev * h->num_sms;
    }
    if (h->use_tc) {
        if (cudaFuncSetAttribute(tc_eval_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_tc) != cudaSuccess ||
            cudaFuncSetAttribute(tc_eval_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_tc) != cudaSuccess)
            return bail("b2e_create: tensor-core eval kernel does not fit shared memory");
        int occ_tc = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_tc, tc_eval_kernel<true>, 256, h->smem_tc) !=
                cudaSuccess || occ_tc < 1)
            return bail("b2e_create: tensor-core eval kernel does not fit an SM");
        if (occ_tc > 512 / tc::TMEM_COLS) occ_tc = 512 / tc::TMEM_COLS;    // TMEM: 512 columns per SM
        h->tc_grid = occ_tc * h->num_sms;
    }
    {   // tcgen05 eval kernel, warp-specialised (b200tc.cu); its context is made once the state
        // buffers exist (the tensor map holds the address of w)
        // default for the shapes it covers (B2E_TC=0: the FFMA eval kernels, B2E_TC=1: the first,
        // single-role tcgen05 kernel kept for comparison)
        const char *tcv = getenv("B2E_TC");
        h->use_tc2 = h->use_eval_kernel && (!tcv || atoi(tcv) == 2) && b2e_tc2_supported(&h->d);
        if (h->use_tc2) {
            h->tc2_check = getenv("B2E_TC_CHECK") && atoi(getenv("B2E_TC_CHECK")) != 0;
            h->use_tc = false;
        }
    }
    if (h->use_eval_kernel) {
        if (cudaFuncSetAttribute(eval_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_eval) != cudaSuccess ||
            cudaFuncSetAttribute(eval_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_eval) != cudaSuccess ||
            cudaFuncSetAttribute(eval_kernel<false, 64, 112>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_eval) != cudaSuccess ||
            cudaFuncSetAttribute(eval_kernel<true, 64, 112>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)h->smem_eval) != cudaSuccess)
            return bail("b2e_create: eval kernel does not fit shared memory");
        h->eval_c = d.N1 == 64 && d.N1p == 64 && d.KT == 112 && d.B == 32 && d.D % 112 == 0 && d.Dp == d.D &&
                    !getenv("B2E_EVAL_GENERIC");
        h->eval_bulk = h->eval_c && d.kind == B2E_PROBLEM_SOFTMAX &&
                       !(getenv("B2E_EVAL_BULK") && atoi(getenv("B2E_EVAL_BULK")) == 0);
        if (h->eval_bulk &&
            (cudaFuncSetAttribute(eval_bulk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)h->smem_eval) != cudaSuccess ||
             cudaFuncSetAttribute(eval_bulk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)h->smem_eval) != cudaSuccess))
            return bail("b2e_create: bulk eval kernel does not fit shared memory");
        h->fuse_update = h->eval_bulk && !h->use_tc2 && d.env_kind == B2E_ENV_MULTIOPTLRS &&
                         getenv("B2E_FUSE_UPDATE") && atoi(getenv("B2E_FUSE_UPDATE")) != 0 &&
                         cudaFuncSetAttribute(eval_bulk_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              (int)h->smem_eval) == cudaSuccess;
        h->nchunks = getenv("B2E_CHUNKS") ? atoi(getenv("B2E_CHUNKS")) : 1;
        if (h->nchunks > 1) {
            int prio_least = 0, prio_greatest = 0;
            cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
            if (cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, prio_least) != cudaSuccess ||
                cudaStreamCreateWithPriority(&h->hi, cudaStreamNonBlocking, prio_least) != cudaSuccess ||
                cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&h->ev_chunk[0], cudaEventDisableTiming) != cudaSuccess)
                return bail("b2e_create: stream/event creation failed");
        }
        int occ_ev = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_ev, eval_kernel<true>, 256, h->smem_eval) !=
                cudaSuccess || occ_ev < 1)
            return bail("b2e_create: eval kernel does not fit an SM");
        if (h->eval_bulk) {                                  // keep it only at the same residency
            int occ_b = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_b, eval_bulk_kernel<true>, 256, h->smem_eval) !=
                    cudaSuccess || occ_b < occ_ev)
                h->eval_bulk = false;
            if (h->fuse_update &&
                (!h->eval_bulk || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_b, eval_bulk_kernel<false, true>, 256,
                                                                                h->smem_eval) != cudaSuccess || occ_b < occ_ev))
                h->fuse_update = false;
        } else {
            h->fuse_update = false;
        }
        h->eval_grid = occ_ev * h->num_sms;
        h->eval_ctas_per_sm = getenv("B2E_EVAL_CTAS") ? atoi(getenv("B2E_EVAL_CTAS")) : occ_ev;
        h->chunk_envs = 4 * h->num_sms;
        h->obs_grid = 1 << 30;
    }
    cudaMemset(h->w, 0, EP * 4); cudaMemset(h->gprev, 0, EP * 4);
    cudaMemset(h->ringw, 0, EP * d.H * 4); cudaMemset(h->ringg, 0, EP * d.H * 4);
    if (d.kind != B2E_PROBLEM_FUNC) {
        if (!dmalloc((void **)&h->X, (size_t)d.N * d.Dp * 4) ||
            !dmalloc((void **)&h->labels, (size_t)d.N * 4) ||
            !dmalloc((void **)&h->targets_f, (size_t)d.N * d.C * 4))
            return bail("b2e_create: cudaMalloc of the data set failed");
        if (d.index_mode == B2E_INDEX_INTERNAL) {
            if (!dmalloc((void **)&h->ord, (size_t)2 * d.E * d.N * 4) ||
                !dmalloc((void **)&h->perm, (size_t)d.E * d.N * 4))
                return bail("b2e_create: cudaMalloc of the index stream failed");
        }
    }
    if (d.row_lex) {
        int *rows = new (std::nothrow) int[d.Pp];
        if (!rows) return bail("b2e_create: out of host memory");
        for (int i = 0; i < d.Pp; ++i) rows[i] = 0;
        const std::string err = lex_rows(d.P, rows);
        bool ok = err.empty() && dmalloc((void **)&h->row_of_param, (size_t)d.Pp * 4) &&
                  cudaMemcpy(h->row_of_param, rows, (size_t)d.Pp * 4, cudaMemcpyHostToDevice) == cudaSuccess;
        int *params = ok ? new (std::nothrow) int[d.Pp] : nullptr;
        if (params) {
            for (int i = 0; i < d.Pp; ++i) params[i] = 0;
            for (int i = 0; i < d.P; ++i) params[rows[i]] = i;
            ok = dmalloc((void **)&h->param_of_row, (size_t)d.Pp * 4) &&
                 cudaMemcpy(h->param_of_row, params, (size_t)d.Pp * 4, cudaMemcpyHostToDevice) == cudaSuccess;
            delete[] params;
        } else {
            ok = false;
        }
        delete[] rows;
        if (!ok) return bail("b2e_create: row table: " + err);
    }
    d.X = h->X; d.labels = h->labels; d.targets = h->targets_f;
    d.w = h->w; d.gprev = h->gprev; d.gnext = h->gnext; d.part = h->part; d.part_u = h->part_u; d.part_r = h->part_r; d.slot_abs = h->slot_abs;
    d.ringw = h->ringw; d.ringg = h->ringg; d.sc = h->sc; d.w2 = h->w2; d.g2 = h->g2; d.ws = h->ws;
    d.ord = h->ord; d.perm = h->perm; d.perm_stride = d.N; d.row_of_param = h->row_of_param; d.param_of_row = h->param_of_row;
    if (h->use_tc2) {
        std::string err;
        h->tc2 = b2e_tc2_create(&h->d, h->num_sms, &err);
        if (!h->tc2) return bail("b2e_create: " + err);
        // resets run through the same kernel (B2E_RESET_PIPELINE=0: the fused kernel in reset mode, kept for A/B runs)
        if (cfg->env_kind == B2E_ENV_MULTIOPTLRS && !(getenv("B2E_RESET_PIPELINE") && atoi(getenv("B2E_RESET_PIPELINE")) == 0)) {
            if (!dmalloc((void **)&h->reset_list, (size_t)d.E * sizeof(int)) || !dmalloc((void **)&h->reset_count, sizeof(int)) ||
                !dmalloc((void **)&h->reset_loss, (size_t)d.E * sizeof(float)))
                return bail("b2e_create: cudaMalloc of the reset work list failed");
            cudaMemset(h->reset_count, 0, sizeof(int));
            h->reset_pipeline = true;
        }
    }
    h->use_tiny = b2e_tiny_supported(&h->d) && !(getenv("B2E_TINY") && atoi(getenv("B2E_TINY")) == 0);
    h->use_thin2 = h->use_thin && b2e_thin2_supported(&h->d) && !(getenv("B2E_THIN2") && atoi(getenv("B2E_THIN2")) == 0) &&
                   b2e_thin2_prepare(&h->d) == 0;
    h->thin_fused = h->use_thin2 && b2e_thin2_fused_step(&h->d);
    init_scalars_kernel<<<(d.E + 127) / 128, 128>>>(d);
    if (cudaDeviceSynchronize() != cudaSuccess) return bail("b2e_create: device initialisation failed");
    *out = h;
    return 0;
}

void b2e_destroy(b2e_handle h) {
    if (!h) return;
    DeviceGuard guard(h->cfg.device);
    cudaFree(h->X); cudaFree(h->targets_f); cudaFree(h->labels); cudaFree(h->ord); cudaFree(h->perm);
    cudaFree(h->row_of_param); cudaFree(h->param_of_row); cudaFree(h->w); cudaFree(h->gprev); cudaFree(h->ringw);
    cudaFree(h->w2); cudaFree(h->g2); cudaFree(h->ws);
    b2e_tc2_destroy(h->tc2);
    cudaFree(h->ringg); cudaFree(h->sc); cudaFree(h->gnext); cudaFree(h->part); cudaFree(h->part_u); cudaFree(h->part_r); cudaFree(h->slot_abs); cudaFree(h->reset_list); cudaFree(h->reset_count); cudaFree(h->reset_loss);
    if (h->side) cudaStreamDestroy(h->side);
    if (h->hi) cudaStreamDestroy(h->hi);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    for (auto &ev : h->ev_chunk) if (ev) cudaEventDestroy(ev);
    for (auto &ev : h->tr) if (ev) cudaEventDestroy(ev);
    delete h;
}

int b2e_bind_dataset(b2e_handle h, const float *features, const void *targets, void *stream) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    Dev &d = h->d;
    if (d.kind == B2E_PROBLEM_FUNC) return fail(h, "b2e_bind_dataset: the func problem has no data");
    if (!features || !targets) return fail(h, "b2e_bind_dataset: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    pad_rows_kernel<<<1184, 256, 0, s>>>(features, h->X, d.N, d.D, d.Dp);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    if (d.kind == B2E_PROBLEM_SOFTMAX)
        CUDA_TRY(h, cudaMemcpyAsync(h->labels, targets, (size_t)d.N * 4, cudaMemcpyDeviceToDevice, s));
    else
        CUDA_TRY(h, cudaMemcpyAsync(h->targets_f, targets, (size_t)d.N * d.C * 4, cudaMemcpyDeviceToDevice, s));
    h->dataset_bound = true;
    return 0;
}

int b2e_set_index_stream(b2e_handle h, const int32_t *perms, int per_env,
                         const int32_t *init_orders, void *stream) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    Dev &d = h->d;
    if (d.kind == B2E_PROBLEM_FUNC || d.index_mode != B2E_INDEX_INTERNAL)
        return fail(h, "b2e_set_index_stream: handle has no internal index stream");
    if (!perms) return fail(h, "b2e_set_index_stream: null perms");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t bytes = (size_t)(per_env ? d.E : 1) * d.N * 4;
    CUDA_TRY(h, cudaMemcpyAsync(h->perm, perms, bytes, cudaMemcpyDeviceToDevice, s));
    d.perm_stride = per_env ? d.N : 0;
    init_order_kernel<<<1184, 256, 0, s>>>(h->ord, init_orders, d.E, d.N);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    h->stream_bound = true;
    return 0;
}

static int check_ready(b2e_handle h, const int32_t *idx, const int32_t *cnt) {
    const Dev &d = h->d;
    if (d.kind == B2E_PROBLEM_FUNC) return 0;
    if (!h->dataset_bound) return fail(h, "no data set bound (b2e_bind_dataset)");
    if (d.index_mode == B2E_INDEX_INTERNAL) {
        if (!h->stream_bound) return fail(h, "no index stream set (b2e_set_index_stream)");
    } else if (!idx || !cnt) {
        return fail(h, "external index mode: batch_idx / batch_cnt are required");
    }
    return 0;
}

int b2e_reset(b2e_handle h, const uint8_t *env_mask, const float *init_params,
              const int32_t *batch_idx, const int32_t *batch_cnt, float *obs_out, void *stream) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    if (check_ready(h, batch_idx, batch_cnt)) return 1;
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.mode = MODE_RESET; a.mask = env_mask; a.init_params = init_params;
    a.ext_idx = batch_idx; a.ext_cnt = batch_cnt; a.obs = obs_out;
    return launch(h, a, stream);
}

int b2e_step(b2e_handle h, const float *actions, const int32_t *batch_idx,
             const int32_t *batch_cnt, float *obs_out, float *reward_out, uint8_t *done_out,
             double *info_out, void *stream) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    if (!actions || !reward_out || !done_out || !info_out)
        return fail(h, "b2e_step: null pointer");
    // obs_out = NULL: ring-only step, the observation rows are not materialised (b200policy.h reads the rings)
    if (!obs_out && !(h->d.split && h->d.env_kind == B2E_ENV_MULTIOPTLRS && h->slot_abs && !h->fuse_update && h->nchunks <= 1))
        return fail(h, "b2e_step: obs_out = NULL needs a MultiOptLRs env on the large-problem pipeline");
    if (check_ready(h, batch_idx, batch_cnt)) return 1;
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.mode = MODE_STEP; a.actions = actions; a.ext_idx = batch_idx; a.ext_cnt = batch_cnt;
    a.obs = obs_out; a.reward = reward_out; a.done = done_out; a.info = info_out;
    if (!h->d.split) return launch(h, a, stream);
    cudaStream_t main_s = (cudaStream_t)stream;
    Dev &d = h->d;
    if (d.env_kind == B2E_ENV_MULTIOPTIMIZE) {
        // ---- update -> eval(w') + scalars -> observations (envs/multioptimize.py:90-154)
        a.e_begin = 0; a.e_count = d.E;
        mo_update_kernel<<<dim3(d.nsegU, d.E), 256, 0, main_s>>>(d, a);
        h->launches++;
        CUDA_TRY(h, cudaGetLastError());
        if (h->use_eval_kernel) {
            Dev &v = h->use_tc ? h->d_tc : h->d_eval;
            v.gprev = d.gprev; v.gnext = d.gnext; v.perm_stride = d.perm_stride;
            v.X = d.X; v.labels = d.labels; v.targets = d.targets; v.w = d.w; v.sc = d.sc;
            v.ord = d.ord; v.perm = d.perm;
            const int cap = h->use_tc ? h->tc_grid : h->eval_grid;
            const int grid_ev = d.E < cap ? d.E : cap;
            if (h->use_tc2) { if (b2e_tc2_launch(h->tc2, &d, &a, 1, main_s)) return fail(h, "tc2 launch failed"); }
            else if (h->use_tc) tc_eval_kernel<true><<<grid_ev, 256, h->smem_tc, main_s>>>(v, a);
            else if (h->eval_bulk) eval_bulk_kernel<true><<<grid_ev, 256, h->smem_eval, main_s>>>(v, a);
            else if (h->eval_c) eval_kernel<true, 64, 112><<<grid_ev, 256, h->smem_eval, main_s>>>(v, a);
            else eval_kernel<true><<<grid_ev, 256, h->smem_eval, main_s>>>(v, a);
            h->launches++;
            CUDA_TRY(h, cudaGetLastError());
        } else if (h->use_thin) {
            const int grid_ev = d.E < h->eval_grid ? d.E : h->eval_grid;
            if (h->use_thin2) { if (b2e_thin2_launch(&d, &a, 1, h->num_sms, main_s)) return fail(h, "thin2 launch failed"); }
            else { Dev dt = d; dt.KT = h->thin_kc;
          if (d.C == 10) thin_eval_kernel<true, 10><<<grid_ev, 256, h->smem_thin, main_s>>>(dt, a);
          else thin_eval_kernel<true><<<grid_ev, 256, h->smem_thin, main_s>>>(dt, a); }
            h->launches++;
            CUDA_TRY(h, cudaGetLastError());
        } else {
            StepArgs b = a;
            b.mode = MODE_EVAL_STEP;
            if (launch(h, b, main_s)) return 1;
        }
        mo_obs_kernel<<<d.nseg * d.E, OBS_WARPS * 32, h->smem_obs, main_s>>>(d, a);
        info_finalize_kernel<<<(d.E + 127) / 128, 128, 0, main_s>>>(d, a);
        h->launches += 2;
        CUDA_TRY(h, cudaGetLastError());
        if (d.auto_reset) {
            StepArgs r;
            memset(&r, 0, sizeof(r));
            r.mode = MODE_RESET; r.mask = done_out; r.obs = obs_out;
            return launch(h, r, main_s);
        }
        return 0;
    }
    // ---- large problems: eval(w) -> update -> eval(w') -> observations, all on the caller's stream
    Dev &dv = h->use_tc ? h->d_tc : h->d_eval;               // same pointers, eval-kernel smem layout
    dv.gprev = d.gprev; dv.gnext = d.gnext; dv.perm_stride = d.perm_stride;
    dv.X = d.X; dv.labels = d.labels; dv.targets = d.targets; dv.w = d.w; dv.sc = d.sc;
    dv.ord = d.ord; dv.perm = d.perm; dv.part = d.part; dv.part_u = d.part_u;
    dv.ringw = d.ringw; dv.ringg = d.ringg; dv.row_of_param = d.row_of_param; dv.param_of_row = d.param_of_row;
    a.e_begin = 0; a.e_count = d.E;
    const int cap_ev = h->use_tc ? h->tc_grid : h->eval_grid;
    const int grid_ev = d.E < cap_ev ? d.E : cap_ev;
    auto mark = [&](int i) { if (h->trace) cudaEventRecord(h->tr[i], main_s); };
    if (h->nchunks > 1 && h->eval_c && !h->use_tc && (h->obs_stages || h->obs_regs)) {
        // experiment (B2E_CHUNKS=n): env chunks alternate between two internal streams so that the
        // FFMA-bound eval kernels of one chunk can share the SMs with the HBM-bound update /
        // observation kernels of the other
        cudaStream_t st[2] = {h->side, h->hi};
        CUDA_TRY(h, cudaEventRecord(h->ev_fork, main_s));
        CUDA_TRY(h, cudaStreamWaitEvent(st[0], h->ev_fork, 0));
        CUDA_TRY(h, cudaStreamWaitEvent(st[1], h->ev_fork, 0));
        const int chunk = (d.E + h->nchunks - 1) / h->nchunks;
        const void *fn = obs2_fn(h->obs_stages, h->obs_regs, h->obs_bulk);
        for (int c = 0; c < h->nchunks; ++c) {
            StepArgs b = a;
            b.e_begin = c * chunk;
            b.e_count = d.E - b.e_begin < chunk ? d.E - b.e_begin : chunk;
            if (b.e_count <= 0) break;
            cudaStream_t s2 = st[c & 1];
            const int cap = h->eval_ctas_per_sm * h->num_sms;
            const int g = b.e_count < cap ? b.e_count : cap;
            eval_kernel<false, 64, 112><<<g, 256, h->smem_eval, s2>>>(dv, b);
            update_kernel<<<dim3(d.nsegU, b.e_count), 256, 0, s2>>>(d, b);
            eval_kernel<true, 64, 112><<<g, 256, h->smem_eval, s2>>>(dv, b);
            const int grid2 = (d.nseg * b.e_count + O2_WARPS - 1) / O2_WARPS;
            void *params[2] = {(void *)&d, (void *)&b};
            CUDA_TRY(h, cudaLaunchKernel(fn, dim3(grid2), dim3(O2_WARPS * 32), params, h->smem_obs2, s2));
            h->launches += 4;
        }
        CUDA_TRY(h, cudaEventRecord(h->ev_join, st[0]));
        CUDA_TRY(h, cudaStreamWaitEvent(main_s, h->ev_join, 0));
        CUDA_TRY(h, cudaEventRecord(h->ev_chunk[0], st[1]));
        CUDA_TRY(h, cudaStreamWaitEvent(main_s, h->ev_chunk[0], 0));
        h->tr_count = 0;
        CUDA_TRY(h, cudaGetLastError());
        goto after_pipeline;
    }
    mark(0);
    if (h->use_tc2) {
        if (b2e_tc2_launch(h->tc2, &d, &a, 0, main_s)) return fail(h, "tc2 launch failed");
    } else if (h->use_tc) {
        tc_eval_kernel<false><<<grid_ev, 256, h->smem_tc, main_s>>>(dv, a);
    } else if (h->use_eval_kernel) {
        if (h->eval_bulk && h->fuse_update) eval_bulk_kernel<false, true><<<grid_ev, 256, h->smem_eval, main_s>>>(dv, a);
        else if (h->eval_bulk) eval_bulk_kernel<false><<<grid_ev, 256, h->smem_eval, main_s>>>(dv, a);
        else if (h->eval_c) eval_kernel<false, 64, 112><<<grid_ev, 256, h->smem_eval, main_s>>>(dv, a);
        else eval_kernel<false><<<grid_ev, 256, h->smem_eval, main_s>>>(dv, a);
    } else if (h->use_thin) {
        if (h->use_thin2) { if (b2e_thin2_launch(&d, &a, h->thin_fused ? 2 : 0, h->num_sms, main_s)) return fail(h, "thin2 launch failed"); }
        else { Dev dt = d; dt.KT = h->thin_kc;
          if (d.C == 10) thin_eval_kernel<false, 10><<<grid_ev, 256, h->smem_thin, main_s>>>(dt, a);
          else thin_eval_kernel<false><<<grid_ev, 256, h->smem_thin, main_s>>>(dt, a); }
    } else {                                                 // generic dense stack
        StepArgs b = a;
        b.mode = MODE_EVAL_FIRST;
        if (launch(h, b, main_s)) return 1;
        h->launches--;
    }
    mark(1);
    if (h->fuse_update && h->eval_bulk && h->use_eval_kernel && !h->use_tc) h->launches--;   // the first eval did it
    else if (h->thin_fused) h->launches--;                   // thin3_eval_kernel<2> did update and second eval as well
    else update_kernel<<<dim3(d.nsegU, d.E), 256, 0, main_s>>>(d, a);
    mark(2);
    if (h->thin_fused) {
        h->launches--;
    } else if (h->use_tc2) {
        if (b2e_tc2_launch(h->tc2, &d, &a, 1, main_s)) return fail(h, "tc2 launch failed");
    } else if (h->use_tc) {
        tc_eval_kernel<true><<<grid_ev, 256, h->smem_tc, main_s>>>(dv, a);
    } else if (h->use_eval_kernel) {
        if (h->eval_bulk) eval_bulk_kernel<true><<<grid_ev, 256, h->smem_eval, main_s>>>(dv, a);
        else if (h->eval_c) eval_kernel<true, 64, 112><<<grid_ev, 256, h->smem_eval, main_s>>>(dv, a);
        else eval_kernel<true><<<grid_ev, 256, h->smem_eval, main_s>>>(dv, a);
    } else if (h->use_thin) {
        if (h->use_thin2) { if (b2e_thin2_launch(&d, &a, 1, h->num_sms, main_s)) return fail(h, "thin2 launch failed"); }
        else { Dev dt = d; dt.KT = h->thin_kc;
          if (d.C == 10) thin_eval_kernel<true, 10><<<grid_ev, 256, h->smem_thin, main_s>>>(dt, a);
          else thin_eval_kernel<true><<<grid_ev, 256, h->smem_thin, main_s>>>(dt, a); }
    } else {
        StepArgs b = a;
        b.mode = MODE_EVAL_STEP;
        if (launch(h, b, main_s)) return 1;
        h->launches--;
    }
    mark(3);
    if (!obs_out) {
        ring_adjg_kernel<<<dim3(d.nsegU, d.E), 256, 0, main_s>>>(d, a);
    } else {
        const int items = d.nseg * d.E;
        if (h->obs_stages || h->obs_regs) {
            const int grid2 = (items + O2_WARPS - 1) / O2_WARPS;
            const void *fn = obs2_fn(h->obs_stages, h->obs_regs, h->obs_bulk);
            void *params[2] = {(void *)&d, (void *)&a};
            CUDA_TRY(h, cudaLaunchKernel(fn, dim3(grid2), dim3(O2_WARPS * 32), params, h->smem_obs2, main_s));
        }
        else if (d.H == 5) obs_kernel<5><<<items, OBS_WARPS * 32, h->smem_obs, main_s>>>(d, a);
        else obs_kernel<0><<<items, OBS_WARPS * 32, h->smem_obs, main_s>>>(d, a);
    }
    mark(4);
    h->tr_count = h->trace ? 4 : 0;
    h->launches += 4;
    CUDA_TRY(h, cudaGetLastError());
after_pipeline:
    info_finalize_kernel<<<(d.E + 127) / 128, 128, 0, main_s>>>(d, a);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    if (h->use_tc2 && h->tc2_check) {                        // debugging aid: did the kernel's watchdog fire?
        int dbg[4] = {0, 0, 0, 0};
        CUDA_TRY(h, cudaStreamSynchronize(main_s));
        if (b2e_tc2_watchdog(h->tc2, dbg)) return fail(h, "tcgen05 eval kernel: cannot read the watchdog word");
        if (dbg[0] != 0)
            return fail(h, "tcgen05 eval kernel: watchdog fired, wait code " + std::to_string(dbg[0]) + " block " +
                               std::to_string(dbg[1]) + " thread " + std::to_string(dbg[2]) + " parity " + std::to_string(dbg[3]));
    }
    {   // g buffers ping-pong: what was g_t is now the newest raw-history gradient
        float *t = d.gprev; d.gprev = d.gnext; d.gnext = t;
    }
    if (d.auto_reset) {
        StepArgs r;
        memset(&r, 0, sizeof(r));
        r.mode = MODE_RESET; r.mask = done_out; r.obs = obs_out;
        return launch(h, r, main_s);
    }
    return 0;
}

int b2e_eval(b2e_handle h, const int32_t *batch_idx, const int32_t *batch_cnt, float *grad_out,
             float *loss_out, void *stream) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    if (!grad_out || !loss_out) return fail(h, "b2e_eval: null pointer");
    if (check_ready(h, batch_idx, batch_cnt)) return 1;
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.mode = MODE_EVAL; a.ext_idx = batch_idx; a.ext_cnt = batch_cnt;
    a.grad_out = grad_out; a.loss_out = loss_out;
    if (h->use_tc2) {
        // the tensor-core eval kernel writes padded rows into the (idle) g_t buffer; copy them out
        a.e_begin = 0; a.e_count = h->d.E;
        if (b2e_tc2_launch(h->tc2, &h->d, &a, 0, stream)) return fail(h, "tc2 launch failed");
        strided_copy_kernel<<<1184, 256, 0, (cudaStream_t)stream>>>(h->d.gnext, grad_out, h->d.E, h->d.P, h->d.Pp, 1);
        h->launches += 2;
        CUDA_TRY(h, cudaGetLastError());
        return 0;
    }
    return launch(h, a, stream);
}

static int state_io(b2e_handle h, int which, void *user, size_t bytes, void *stream, int to_user) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    if (!user) return fail(h, "b2e_get/set_state: null pointer");
    Dev &d = h->d;
    cudaStream_t s = (cudaStream_t)stream;
    size_t want = 0;
    switch (which) {
        case B2E_STATE_PARAMS: case B2E_STATE_GRAD_PREV: want = (size_t)d.E * d.P * 4; break;
        case B2E_STATE_ADJ_WEIGHTS: case B2E_STATE_ADJ_GRADS: want = (size_t)d.E * d.H * d.P * 4; break;
        case B2E_STATE_ADJ_LOSSES: want = (size_t)d.E * d.H * 4; break;
        case B2E_STATE_RAW_LOSSES: want = (size_t)d.E * RAW_DEPTH * 4; break;
        case B2E_STATE_RAW_GSUMS: want = (size_t)d.E * RAW_DEPTH * 8; break;
        case B2E_STATE_STEP: case B2E_STATE_CURSOR: want = (size_t)d.E * 4; break;
        case B2E_STATE_ORDER: want = (size_t)d.E * d.N * 4; break;
        default: return fail(h, "b2e_get/set_state: unknown selector");
    }
    if (bytes != want)
        return fail(h, "b2e_get/set_state: buffer is " + std::to_string(bytes) + " bytes, expected " +
                           std::to_string(want));
    switch (which) {
        case B2E_STATE_PARAMS: case B2E_STATE_GRAD_PREV:
            strided_copy_kernel<<<1184, 256, 0, s>>>(which == B2E_STATE_PARAMS ? h->w : d.gprev,
                                                     (float *)user, d.E, d.P, d.Pp, to_user);
            break;
        case B2E_STATE_ADJ_WEIGHTS: case B2E_STATE_ADJ_GRADS: case B2E_STATE_ADJ_LOSSES:
            if (!to_user) set_nvalid_kernel<<<(d.E + 127) / 128, 128, 0, s>>>(d, d.H);
            ring_copy_kernel<<<d.E, 256, 0, s>>>(d, which, (float *)user, to_user);
            if (!to_user && d.slot_abs && which != B2E_STATE_ADJ_LOSSES) slot_abs_kernel<<<d.E * d.H, 256, 0, s>>>(d);
            break;
        case B2E_STATE_ORDER:
            if (!h->ord) return fail(h, "b2e_get/set_state: no internal index stream");
            order_copy_kernel<<<d.E, 256, 0, s>>>(d, (int *)user, to_user);
            break;
        default:
            scalars_copy_kernel<<<(d.E + 127) / 128, 128, 0, s>>>(d, which, user, to_user);
    }
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

int b2e_get_state(b2e_handle h, int which, void *dst, size_t bytes, void *stream) {
    return state_io(h, which, dst, bytes, stream, 1);
}

int b2e_set_state(b2e_handle h, int which, const void *src, size_t bytes, void *stream) {
    return state_io(h, which, const_cast<void *>(src), bytes, stream, 0);
}

int b2e_get_batch_indices(b2e_handle h, int32_t *idx_out, int32_t *cnt_out, void *stream) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    if (!idx_out || !cnt_out) return fail(h, "b2e_get_batch_indices: null pointer");
    if (!h->ord || !h->stream_bound) return fail(h, "b2e_get_batch_indices: no internal index stream");
    batch_indices_kernel<<<h->d.E, 64, 0, (cudaStream_t)stream>>>(h->d, idx_out, cnt_out);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

int b2e_set_trace(b2e_handle h, int enabled) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    if (enabled)
        for (auto &ev : h->tr)
            if (!ev && cudaEventCreate(&ev) != cudaSuccess) return fail(h, "b2e_set_trace: cudaEventCreate failed");
    h->trace = enabled != 0;
    h->tr_count = 0;
    return 0;
}

int b2e_get_trace(b2e_handle h, float *ms_out, int capacity) {
    if (!h || !ms_out) return -1;
    DeviceGuard guard(h->cfg.device);
    int n = h->tr_count < capacity ? h->tr_count : capacity;
    for (int i = 0; i < n; ++i) {
        if (cudaEventSynchronize(h->tr[i + 1]) != cudaSuccess ||
            cudaEventElapsedTime(&ms_out[i], h->tr[i], h->tr[i + 1]) != cudaSuccess) return -1;
    }
    return n;
}

int b2e_next_batch(b2e_handle h, const uint8_t *env_mask, void *stream) {
    if (!h) return 1;
    DeviceGuard guard(h->cfg.device);
    if (!h->ord || !h->stream_bound) return fail(h, "b2e_next_batch: no internal index stream");
    next_batch_kernel<<<h->d.E, 256, 0, (cudaStream_t)stream>>>(h->d, env_mask);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

}  // extern "C"
