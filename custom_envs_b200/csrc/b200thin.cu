// Eval kernels of libb200env for softmax regression with a wide input (BASELINE config 3: 784 -> 10,
// P = 7850 agents, minibatch 32, 1024 lock-step envs): loss and batch-SUM gradient of
// logits = X.W + b under softmax cross-entropy (reference problems/optimize_nn.py:35-52, 152-159),
// at w_{t-1} (first launch of a step) and at w_t together with the step's scalars (second launch).
//
// The kernel they replace (thin_eval_kernel, b200env.cu) streams the feature axis in 128-wide chunks
// twice, forward and backward: 65 k warp instructions per env of which a fifth are multiply-adds, at
// 45 % issue utilisation, 0.126 ms per launch.  Here the minibatch is small enough to sit in shared
// memory as a whole, gathered once with 16-byte cp.async (8 threads per row; rows the ragged last
// minibatch does not have are zero filled), the next env's rows requested into L2 meanwhile:
//   thin3_eval_kernel (default, 0.083 / 0.092 ms): a cluster of two CTAs per env, each holding one half of
//       the feature axis of the rows AND of W in shared memory, three CTAs per SM; partial logits meet
//       through distributed shared memory (described at the kernel);
//   thin2_eval_kernel (B2E_THIN2=2, 0.108 ms): one CTA per env with all features of the rows resident, two
//       CTAs per SM, W rows read from L2 inside the forward loop -- which is what it waits for (ncu: 39 %
//       long scoreboard), hence thin3.  Kept for A/B runs:
//   forward  : warp = 8 samples x one half of the feature axis; lane = feature (stride 32); 40 packed
//              FMAs per step on 80 accumulators; one recursive-halving shuffle reduction per warp (155
//              shuffles instead of 400), the two halves meet in shared memory
//   softmax  : thread = sample: cross-entropy, d loss / d logits [32][12] in shared memory
//   backward : thread = features k, k + 256, k + 512 (, k + 768): per sample 3-4 conflict-free feature
//              loads and three broadcast loads of the sample's dZ row for 30-40 FMAs; gradient rows
//              leave as 8-byte stores (a warp writes 1 280 contiguous bytes)
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "b200env_shared.cuh"
#include "b200thin.h"

namespace {
namespace thin2 {

constexpr int THREADS = 256, BMAX = 32, C = 10, CP = 12, KPT = 4;      // classes, dZ row stride, features per backward thread

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
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(gmem_src) : "memory");
}

// One level of the recursive-halving reduction: lanes whose `bit` is clear keep the first N values, the others
// the last N; each adds what its partner (lane ^ bit) held of the half it keeps.
template <int N>
__device__ __forceinline__ void halve(float *v, bool upper, int bit) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const float send = upper ? v[i] : v[N + i];
        const float keep = upper ? v[N + i] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
}

template <bool SECOND>
__global__ void __launch_bounds__(THREADS, 2) thin2_eval_kernel(const __grid_constant__ Dev d, const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    __shared__ float misc[8];
    __shared__ double red[8];
    __shared__ int idx_s[BMAX], ys[BMAX];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int D = d.D;
    float *Xs = sm;                                   // [32][D]
    float *Zp = Xs + BMAX * D;                        // [2 feature halves][32][CP] partial logits
    float *dZ = Zp + 2 * BMAX * CP;                   // [32][CP]
    float *lb = dZ + BMAX * CP;                       // [32] per-sample losses
    const int Dh = ((D / 2 + 31) / 32) * 32;          // first half: a whole number of 32-feature steps
    const int e_end = a.e_begin + a.e_count;
    for (int e = a.e_begin + blockIdx.x; e < e_end; e += gridDim.x) {
        EnvScalars *sc = d.sc + e;
        const float *wE = d.w + (size_t)e * d.Pp;
        float *gout = d.gnext + (size_t)e * d.Pp;
        const int *idx; int cnt;
        current_batch(d, a, e, sc, idx, cnt);
        __syncthreads();                              // the previous env's readers are done with shared memory
        if (tid < BMAX) {
            const int row = (tid < cnt) ? idx[tid] : -1;
            idx_s[tid] = row;
            ys[tid] = row >= 0 ? d.labels[row] : 0;
        } else if (tid < 2 * BMAX && e + (int)gridDim.x < e_end) {
            // the rows of this CTA's NEXT env into L2 while this one computes (one bulk prefetch per row)
            const int en = e + gridDim.x;
            const int *idn; int cn;
            current_batch(d, a, en, d.sc + en, idn, cn);
            if (tid - BMAX < cn)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(d.X + (size_t)idn[tid - BMAX] * d.Dp), "r"(D * 4) : "memory");
        }
        __syncthreads();
        {   // ---- gather: 8 threads per row, 16 bytes each, D / 32 rounds
            const int r = tid >> 3, q0 = tid & 7, nq = D >> 2, row = idx_s[r];
            float *dst = Xs + r * D;
            if (row >= 0) {
                const float *src = d.X + (size_t)row * d.Dp;
                for (int q = q0; q < nq; q += 8) cp_async16(dst + 4 * q, src + 4 * q);
            } else {
                for (int q = q0; q < nq; q += 8) *reinterpret_cast<float4 *>(dst + 4 * q) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        }
        __syncthreads();
        {   // ---- forward: warp = (8 samples, feature half)
            const int sg = warp & 3, kh = warp >> 2;
            const int kbeg = kh * Dh, kend = kh ? D : min(Dh, D);
            f32x2 acc2[8][C / 2];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int c = 0; c < C / 2; ++c) acc2[i][c] = pack2(0.f, 0.f);
            const float *xr = Xs + (8 * sg) * D;
            // the lane's W rows come from L2 (~500 cycles): the row of the NEXT step is requested before this step's FMAs
            f32x2 w2[C / 2], wn[C / 2];
            {
                const int kk = (kbeg + lane < kend) ? kbeg + lane : kbeg;
                const f32x2 *wrow = reinterpret_cast<const f32x2 *>(wE + (size_t)kk * C);   // 40-byte rows: 8-byte aligned
#pragma unroll
                for (int c = 0; c < C / 2; ++c) w2[c] = __ldg(wrow + c);
            }
            for (int k0 = kbeg; k0 < kend; k0 += 32) {
                const int k = k0 + lane;
                const bool live = k < kend;
                const int kk = live ? k : kbeg;
                {
                    const int kn = (k + 32 < kend) ? k + 32 : kbeg;
                    const f32x2 *wrow = reinterpret_cast<const f32x2 *>(wE + (size_t)kn * C);
#pragma unroll
                    for (int c = 0; c < C / 2; ++c) wn[c] = __ldg(wrow + c);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float x = live ? xr[i * D + kk] : 0.f;
                    const f32x2 xx = pack2(x, x);
#pragma unroll
                    for (int c = 0; c < C / 2; ++c) ffma2(acc2[i][c], xx, w2[c]);
                }
#pragma unroll
                for (int c = 0; c < C / 2; ++c) w2[c] = wn[c];
            }
            float v[80];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int c = 0; c < C / 2; ++c) unpack2(acc2[i][c], v[i * C + 2 * c], v[i * C + 2 * c + 1]);
            // 80 partial logits x 32 lanes -> 5 sums per lane pair
            halve<40>(v, (lane & 16) != 0, 16);
            halve<20>(v, (lane & 8) != 0, 8);
            halve<10>(v, (lane & 4) != 0, 4);
            halve<5>(v, (lane & 2) != 0, 2);
#pragma unroll
            for (int i = 0; i < 5; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], 1);
            if ((lane & 1) == 0) {
                const int base = ((lane >> 4) & 1) * 40 + ((lane >> 3) & 1) * 20 + ((lane >> 2) & 1) * 10 + ((lane >> 1) & 1) * 5;
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const int flat = base + i, s = flat / C, c = flat - s * C;
                    Zp[(kh * BMAX + 8 * sg + s) * CP + c] = v[i];
                }
            }
        }
        __syncthreads();
        // ---- softmax cross-entropy per sample, dZ (problems/optimize_nn.py:47-50)
        if (tid < BMAX) {
            const int s = tid;
            float z[C];
            float loss = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) z[c] = (Zp[s * CP + c] + Zp[(BMAX + s) * CP + c]) + wE[d.P1 + c];
            if (s < cnt) {
                const int y = ys[s];
                float m = z[0];
#pragma unroll
                for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
                float sum = 0.f, zy = 0.f;
#pragma unroll
                for (int c = 0; c < C; ++c) { sum += expf(z[c] - m); if (c == y) zy = z[c]; }
                loss = (m + logf(sum)) - zy;
                const float inv = 1.0f / sum;
#pragma unroll
                for (int c = 0; c < C; ++c) z[c] = expf(z[c] - m) * inv - (c == y ? 1.f : 0.f);
            } else {
#pragma unroll
                for (int c = 0; c < C; ++c) z[c] = 0.f;
            }
#pragma unroll
            for (int c = 0; c < C; ++c) dZ[s * CP + c] = z[c];
            dZ[s * CP + 10] = 0.f; dZ[s * CP + 11] = 0.f;
            lb[s] = loss;
        }
        __syncthreads();
        if (tid == 0) {                               // mean loss, the samples in index order
            float l = 0.f;
            for (int s = 0; s < cnt; ++s) l += lb[s];
            misc[0] = l / (float)cnt;
        }
        // ---- backward: thread = features tid + 256 j
        float gsum = 0.f;
        {
            f32x2 g2[KPT][C / 2];
            int kq[KPT];
#pragma unroll
            for (int j = 0; j < KPT; ++j) {
                kq[j] = tid + THREADS * j;
#pragma unroll
                for (int c = 0; c < C / 2; ++c) g2[j][c] = pack2(0.f, 0.f);
            }
            const int nk = (D - tid + THREADS - 1) / THREADS;     // features of this thread (D <= 4 * 256)
#pragma unroll 4
            for (int s = 0; s < cnt; ++s) {
                const float4 z0 = *reinterpret_cast<const float4 *>(dZ + s * CP);
                const float4 z1 = *reinterpret_cast<const float4 *>(dZ + s * CP + 4);
                const float2 z2 = *reinterpret_cast<const float2 *>(dZ + s * CP + 8);
                const f32x2 zz[C / 2] = {pack2(z0.x, z0.y), pack2(z0.z, z0.w), pack2(z1.x, z1.y), pack2(z1.z, z1.w), pack2(z2.x, z2.y)};
                const float *xs = Xs + s * D;
#pragma unroll
                for (int j = 0; j < KPT; ++j) {
                    if (j < nk) {
                        const float x = xs[kq[j]];
                        const f32x2 xx = pack2(x, x);
#pragma unroll
                        for (int c = 0; c < C / 2; ++c) ffma2(g2[j][c], xx, zz[c]);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < KPT; ++j) {
                if (j < nk) {
                    f32x2 *dst = reinterpret_cast<f32x2 *>(gout + (size_t)kq[j] * C);
#pragma unroll
                    for (int c = 0; c < C / 2; ++c) {
                        dst[c] = g2[j][c];
                        float lo, hi;
                        unpack2(g2[j][c], lo, hi);
                        gsum += lo + hi;
                    }
                }
            }
        }
        if (tid < C) {                                // bias gradient: column sums of dZ
            float g = 0.f;
            for (int s = 0; s < cnt; ++s) g += dZ[s * CP + tid];
            gout[d.P1 + tid] = g;
            gsum += g;
        }
        __syncthreads();
        const float loss = misc[0];
        if (!SECOND) {
            if (a.loss_out != nullptr && tid == 0) a.loss_out[e] = loss;
            continue;
        }
        // ---- scalars of the step (multioptlrs.py:89-128)
        const double gtot = block_sum((double)gsum, red);
        if (tid == 0) step_scalars(d, a, sc, e, loss, gtot, misc);
        __syncthreads();
        const bool wrap = misc[4] != 0.f;
        __syncthreads();
        if (wrap) shuffle_order(d, e, sc);
    }
}


// ------------------------------------------------------------------------------------------------
// thin3: a CLUSTER OF TWO CTAs per env, each owning one half of the feature axis -- its half of the
// minibatch rows (50 KB) AND of W (15.7 KB) in shared memory, so three CTAs fit an SM (24 warps to hide the
// gather behind) and the forward pass reads both operands from shared memory (thin2 reads W rows from L2
// inside its inner loop and spends its time waiting for them: profiles/r2_ncu_thin2_v1.txt, 39 % long
// scoreboard).  The partial logits [32][10] of the two halves meet through distributed shared memory, both
// CTAs run the (tiny) softmax, each writes the gradient rows of its half.
//   forward  : warp = 4 samples x the CTA's 392 features; lane = feature (stride 32): 4 feature loads and
//              five 8-byte loads of the lane's W row for 20 packed FMAs; recursive-halving reduction of
//              the 40 partial sums (45 shuffles)
//   backward : thread = features t, t + 256 of the half
namespace cgx = cooperative_groups;

// Loss + gradient at the parameters in HBM (-> Dev::gnext); SECOND: also the step's scalars (second evaluation of a
// pipelined step).
template <bool SECOND>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 3)
thin3_eval_kernel(const __grid_constant__ Dev d, const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) float sm[];
    __shared__ float misc[8];
    __shared__ double red[8];
    __shared__ double gpart;
    __shared__ float bs[C + 2];                       // the bias
    __shared__ int idx_s[BMAX], ys[BMAX];
    cgx::cluster_group cluster = cgx::this_cluster();
    const int rank = (int)cluster.block_rank(), peer = rank ^ 1;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int D = d.D, Dh = D >> 1, kbase = rank * Dh;          // this CTA's features [kbase, kbase + Dh)
    float *Xs = sm;                                   // [32][Dh]
    float *Ws = Xs + BMAX * Dh;                       // [Dh][10]
    float *Zp = Ws + Dh * C;                          // [2 buffers][32][CP] partial logits of this half
    float *dZ = Zp + 2 * BMAX * CP;                   // [32][CP]
    float *lb = dZ + BMAX * CP;                       // [32]
    const int nclusters = gridDim.x >> 1, cid = blockIdx.x >> 1;
    const int e_end = a.e_begin + a.e_count;
    int it = 0;
    for (int e = a.e_begin + cid; e < e_end; e += nclusters) {
        EnvScalars *sc = d.sc + e;
        const float *wE = d.w + (size_t)e * d.Pp;
        float *gout = d.gnext + (size_t)e * d.Pp;
        const int *idx; int cnt;
        current_batch(d, a, e, sc, idx, cnt);
        __syncthreads();
        if (tid < BMAX) {
            const int row = (tid < cnt) ? idx[tid] : -1;
            idx_s[tid] = row;
            ys[tid] = row >= 0 ? d.labels[row] : 0;
        } else if (tid < 2 * BMAX && e + nclusters < e_end) {  // this cluster's next env: its rows into L2
            const int en = e + nclusters;
            const int *idn; int cn;
            current_batch(d, a, en, d.sc + en, idn, cn);
            if (tid - BMAX < cn)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(d.X + (size_t)idn[tid - BMAX] * d.Dp + kbase), "r"(Dh * 4) : "memory");
        } else if (tid >= 2 * BMAX && tid < 2 * BMAX + C) {
            bs[tid - 2 * BMAX] = wE[d.P1 + tid - 2 * BMAX];
        }
        {   // W half: contiguous Dh * 40 bytes
            const float *src = wE + (size_t)kbase * C;
            const int nq = (Dh * C) >> 2;
            for (int q = tid; q < nq; q += THREADS) cp_async16(Ws + 4 * q, src + 4 * q);
        }
        __syncthreads();
        {   // minibatch rows, this half of the features: 8 threads per row
            const int r = tid >> 3, q0 = tid & 7, nq = Dh >> 2, row = idx_s[r];
            float *dst = Xs + r * Dh;
            if (row >= 0) {
                const float *src = d.X + (size_t)row * d.Dp + kbase;
                for (int q = q0; q < nq; q += 8) cp_async16(dst + 4 * q, src + 4 * q);
            } else {
                for (int q = q0; q < nq; q += 8) *reinterpret_cast<float4 *>(dst + 4 * q) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        }
        __syncthreads();
        float gsum = 0.f;
        float *Zmine = Zp + (it++ & 1) * BMAX * CP;     // alternates between envs: the peer may still read the last one
        {   // ---- forward: warp = 4 samples, all Dh features of the half
            f32x2 acc2[4][C / 2];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int c = 0; c < C / 2; ++c) acc2[i][c] = pack2(0.f, 0.f);
            const float *xr = Xs + (4 * warp) * Dh;
            for (int k = lane; k < Dh; k += 32) {
                const f32x2 *wrow = reinterpret_cast<const f32x2 *>(Ws + k * C);
                f32x2 w2[C / 2];
#pragma unroll
                for (int c = 0; c < C / 2; ++c) w2[c] = wrow[c];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float x = xr[i * Dh + k];
                    const f32x2 xx = pack2(x, x);
#pragma unroll
                    for (int c = 0; c < C / 2; ++c) ffma2(acc2[i][c], xx, w2[c]);
                }
            }
            float v[40];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int c = 0; c < C / 2; ++c) unpack2(acc2[i][c], v[i * C + 2 * c], v[i * C + 2 * c + 1]);
            halve<20>(v, (lane & 16) != 0, 16);
            halve<10>(v, (lane & 8) != 0, 8);
            halve<5>(v, (lane & 4) != 0, 4);
#pragma unroll
            for (int i = 0; i < 5; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], 2);
#pragma unroll
            for (int i = 0; i < 5; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], 1);
            if ((lane & 3) == 0) {
                const int base = ((lane >> 4) & 1) * 20 + ((lane >> 3) & 1) * 10 + ((lane >> 2) & 1) * 5;
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const int flat = base + i, s = flat / C, c = flat - s * C;
                    Zmine[(4 * warp + s) * CP + c] = v[i];
                }
            }
        }
        cluster.sync();                           // both halves of the logits are in place
        // ---- softmax cross-entropy per sample (both CTAs, redundantly), dZ (problems/optimize_nn.py:47-50)
        if (tid < BMAX) {
            const int s = tid;
            const float *Zpeer = cluster.map_shared_rank(Zmine, peer);
            const float *Z0 = rank == 0 ? Zmine : Zpeer, *Z1 = rank == 0 ? Zpeer : Zmine;     // feature order: the same sum in both CTAs
            float z[C];
            float ls = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) z[c] = (Z0[s * CP + c] + Z1[s * CP + c]) + bs[c];
            if (s < cnt) {
                const int y = ys[s];
                float m = z[0];
#pragma unroll
                for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
                float sum = 0.f, zy = 0.f;
#pragma unroll
                for (int c = 0; c < C; ++c) { sum += expf(z[c] - m); if (c == y) zy = z[c]; }
                ls = (m + logf(sum)) - zy;
                const float inv = 1.0f / sum;
#pragma unroll
                for (int c = 0; c < C; ++c) z[c] = expf(z[c] - m) * inv - (c == y ? 1.f : 0.f);
            } else {
#pragma unroll
                for (int c = 0; c < C; ++c) z[c] = 0.f;
            }
#pragma unroll
            for (int c = 0; c < C; ++c) dZ[s * CP + c] = z[c];
            dZ[s * CP + 10] = 0.f; dZ[s * CP + 11] = 0.f;
            lb[s] = ls;
        }
        __syncthreads();
        if (tid == 0) {                           // mean loss, the samples in index order
            float l = 0.f;
            for (int s = 0; s < cnt; ++s) l += lb[s];
            misc[0] = l / (float)cnt;
        }
        // ---- backward: thread = features tid, tid + 256 of the half
        constexpr int KH = 2;
        f32x2 g2[KH][C / 2];
#pragma unroll
        for (int j = 0; j < KH; ++j)
#pragma unroll
            for (int c = 0; c < C / 2; ++c) g2[j][c] = pack2(0.f, 0.f);
        const int nk = (Dh - tid + THREADS - 1) / THREADS;     // 0, 1 or 2 features (Dh <= 512)
#pragma unroll 4
        for (int s = 0; s < cnt; ++s) {
            const float4 z0 = *reinterpret_cast<const float4 *>(dZ + s * CP);
            const float4 z1 = *reinterpret_cast<const float4 *>(dZ + s * CP + 4);
            const float2 z2 = *reinterpret_cast<const float2 *>(dZ + s * CP + 8);
            const f32x2 zz[C / 2] = {pack2(z0.x, z0.y), pack2(z0.z, z0.w), pack2(z1.x, z1.y), pack2(z1.z, z1.w), pack2(z2.x, z2.y)};
            const float *xs = Xs + s * Dh;
#pragma unroll
            for (int j = 0; j < KH; ++j) {
                if (j < nk) {
                    const float x = xs[tid + THREADS * j];
                    const f32x2 xx = pack2(x, x);
#pragma unroll
                    for (int c = 0; c < C / 2; ++c) ffma2(g2[j][c], xx, zz[c]);
                }
            }
        }
        float gb = 0.f;                           // bias gradient of class tid: column sum of dZ
        if (tid < C) for (int s = 0; s < cnt; ++s) gb += dZ[s * CP + tid];
#pragma unroll
        for (int j = 0; j < KH; ++j) {
            if (j < nk) {
                f32x2 *dst = reinterpret_cast<f32x2 *>(gout + (size_t)(kbase + tid + THREADS * j) * C);
#pragma unroll
                for (int c = 0; c < C / 2; ++c) {
                    dst[c] = g2[j][c];
                    float lo, hi;
                    unpack2(g2[j][c], lo, hi);
                    gsum += lo + hi;
                }
            }
        }
        if (rank == 0 && tid < C) { gout[d.P1 + tid] = gb; gsum += gb; }
        __syncthreads();
        const float loss = misc[0];
        if (!SECOND) {
            if (rank == 0 && a.loss_out != nullptr && tid == 0) a.loss_out[e] = loss;
            continue;
        }
        // ---- scalars of the step (multioptlrs.py:89-128): CTA 0 adds the other half's gradient sum
        const double gmine = block_sum((double)gsum, red);
        if (tid == 0) gpart = gmine;
        cluster.sync();
        if (rank == 0) {
            if (tid == 0) step_scalars(d, a, sc, e, loss, gmine + *cluster.map_shared_rank(&gpart, peer), misc);
            __syncthreads();
            const bool wrap = misc[4] != 0.f;
            __syncthreads();
            if (wrap) shuffle_order(d, e, sc);
        }
    }
    cluster.sync();                                   // no CTA leaves while its peer may still read its shared memory
}

size_t smem_bytes3(const Dev &d) { return (size_t)(BMAX * (d.D / 2) + (d.D / 2) * C + 2 * BMAX * CP + BMAX * CP + BMAX) * sizeof(float); }

size_t smem_bytes(const Dev &d) { return (size_t)(BMAX * d.D + 2 * BMAX * CP + BMAX * CP + BMAX) * sizeof(float); }

}  // namespace thin2
}  // namespace

bool b2e_thin2_supported(const void *dev) {
    const Dev &d = *static_cast<const Dev *>(dev);
    return d.kind == B2E_PROBLEM_SOFTMAX && !d.hidden && !d.generic && d.C == thin2::C && d.B <= thin2::BMAX &&
           d.D % 4 == 0 && d.D >= 64 && d.D <= thin2::KPT * thin2::THREADS && d.Pp % 4 == 0 &&
           2 * (thin2::smem_bytes(d) + 1024) <= 227 * 1024;
}

// B2E_THIN2=2: the one-CTA-per-env kernel; default: the cluster kernel where the shape allows it
static bool use_cluster_kernel(const Dev &d) {
    const char *v = getenv("B2E_THIN2");
    return !(v && atoi(v) == 2) && d.D % 8 == 0 && d.D / 2 <= 2 * thin2::THREADS &&
           3 * (thin2::smem_bytes3(d) + 1024) <= 227 * 1024;
}

int b2e_thin2_prepare(const void *dev) {
    const Dev &d = *static_cast<const Dev *>(dev);
    const int bytes = (int)thin2::smem_bytes(d), bytes3 = (int)thin2::smem_bytes3(d);
    return (cudaFuncSetAttribute(thin2::thin2_eval_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess &&
            cudaFuncSetAttribute(thin2::thin2_eval_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess &&
            cudaFuncSetAttribute(thin2::thin3_eval_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes3) == cudaSuccess &&
            cudaFuncSetAttribute(thin2::thin3_eval_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes3) == cudaSuccess) ? 0 : 1;
}

int b2e_thin2_launch(const void *dev, const void *args, int second, int num_sms, void *stream) {
    const Dev &d = *static_cast<const Dev *>(dev);
    const StepArgs &a = *static_cast<const StepArgs *>(args);
    const cudaStream_t cs = (cudaStream_t)stream;
    if (use_cluster_kernel(d)) {
        // clusters of two CTAs, three CTAs per SM; every cluster gets the same number of envs (no ragged last round)
        const int max_clusters = (3 * num_sms) / 2;
        const int rounds = (a.e_count + max_clusters - 1) / max_clusters;
        const int clusters = (a.e_count + rounds - 1) / rounds;
        const size_t bytes = thin2::smem_bytes3(d);
        if (second) thin2::thin3_eval_kernel<true><<<2 * clusters, thin2::THREADS, bytes, cs>>>(d, a);
        else thin2::thin3_eval_kernel<false><<<2 * clusters, thin2::THREADS, bytes, cs>>>(d, a);
        return cudaGetLastError() == cudaSuccess ? 0 : 1;
    }
    const int cap = 2 * num_sms;
    const int grid = a.e_count < cap ? a.e_count : cap;
    const size_t bytes = thin2::smem_bytes(d);
    if (second) thin2::thin2_eval_kernel<true><<<grid, thin2::THREADS, bytes, cs>>>(d, a);
    else thin2::thin2_eval_kernel<false><<<grid, thin2::THREADS, bytes, cs>>>(d, a);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}
