// Shared per-agent policy of libb200env (C ABI: include/b200policy.h; SURVEY 8f.2).
//
// What the reference's callers do with the observation matrix of OptVecEnv.step_wait
// (vectorize/optvecenv.py:78-88): stable-baselines' runner evaluates ONE MlpPolicy -- two tanh layers
// of 64 units and a linear head -- on each of the sum(P) agent rows (run_multiagent_exp_single.py:37-49,
// play_optimize.py:79-98).  At BASELINE config 4 that is 2.08e8 rows x (15*64 + 64*64 + 64) MACs =
// 2.1 TFLOP per env step: dense GEMM work, so it runs on the tensor cores:
//
//   tile = 128 agent rows; A1 [128 x 16] bf16 = the observation rows + a column of ones (bias),
//   D1 [128 x 64] = A1 . [W1 | b1]^T         one tcgen05.mma kind::f16 (M 128, N 64, K 16), fp32 in TMEM
//   A2 [128 x 80] bf16 = tanh(D1) + a column of ones + zero padding
//   D2 [128 x 64] = A2 . [W2 | b2 | 0]^T     five MMAs
//   mean = tanh(D2) . w3 + b3                 FFMA on the fp32 accumulators, lane = row
//
// Persistent, one 768-thread CTA per SM, SIX independent groups of four warps; every group runs its own
// tiles start to finish (operand staging, MMA issue by its thread 0, tcgen05.commit -> the group's
// mbarrier, tcgen05.ld epilogues), so while one group waits for its MMA the SM's MUFU units -- the
// bound of this kernel: 128 tanh per row, 16 per clock per SM -- are busy with the other five (four groups
// reach 0.63 of that rate, six 0.75).  TMEM: 64 columns per group, D2 overwrites D1 (read out before).  Operands use the no-swizzle K-major canonical layout: core
// matrices of 8 rows x 16 bytes, contiguous (128 B), LBO = 128 (next core matrix along K), SBO = K/8 * 128
// (next 8 rows).
//
// Two front ends: dense rows (what b2e_step wrote; one 7.5 KB bulk copy per tile, requested a tile ahead) and
// the env's adjusted-history rings (MultiOptLRs; lane = parameter, 2H coalesced 4-byte loads prefetched one
// tile ahead; the 3H observation words per agent never exist in HBM).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <string>
#include <type_traits>

#include "b200env_shared.cuh"
#include "b200env_internal.h"
#include "b200policy.h"

namespace {
namespace pol {

#ifndef B2P_GROUPS
#define B2P_GROUPS 6
#endif
constexpr int TILE = 128, HID = B2P_HIDDEN, K2 = 80;
constexpr int XMAX = 15;                          // the narrow row (K1 = 16): obs_dim <= 15, held in registers
constexpr int SBO2 = (K2 / 8) * 128, A2_BYTES = (TILE / 8) * SBO2, B2_BYTES = (HID / 8) * SBO2;
constexpr int W3_BYTES = (HID + 4) * 4;
constexpr int SMEM_LIMIT = 227 * 1024;

// First-layer K of an observation row (b2p_obs_width): the row and the bias column, rounded up to the MMA's K of 16.
// K1 = 16 is the narrow kernel (obs_dim <= 15); K1 = 32 .. 80 the wide variants.
__host__ __device__ constexpr int obs_width(int obs_dim) { return 16 * ((obs_dim + 16) / 16); }

// policy_kernel's shared memory: per group [dense staging (narrow only) | A1 | A2], then [W1 | b1], [W2 | b2], w3 of the
// action tower; the step kernel (b2p_step*) adds the value tower's operands behind them and runs the two towers one
// after the other in the same TMEM columns and A2 buffer
constexpr int policy_smem(int groups, int g_bytes, int b1_bytes, bool step) {
    const int off_w3 = groups * g_bytes + b1_bytes + B2_BYTES;
    const int off_vw3 = (off_w3 + W3_BYTES + 127) / 128 * 128 + b1_bytes + B2_BYTES;
    return (step ? off_vw3 : off_w3) + W3_BYTES + 128;   // + slack to align the base to 128 bytes
}
// the wide variants: as many groups as the shared memory holds (at most the narrow kernel's six); no staging buffers,
// the front end writes A1 directly
constexpr int wide_groups(int g_bytes, int b1_bytes, bool step) {
    int g = 6;
    while (g > 1 && policy_smem(g, g_bytes, b1_bytes, step) > SMEM_LIMIT - 256) --g;     // 256: the static barriers
    return g;
}
template <int K1, bool STEP>
struct Geo {
    static constexpr bool WIDE = K1 > 16;
    static constexpr int SBO1 = (K1 / 8) * 128, A1_BYTES = (TILE / 8) * SBO1, B1_BYTES = (HID / 8) * SBO1;
    static constexpr int GROUPS = WIDE ? wide_groups(A1_BYTES + A2_BYTES, B1_BYTES, STEP) : B2P_GROUPS;
    static constexpr int THREADS = GROUPS * 128;
    static constexpr int NSTG = WIDE ? 0 : GROUPS <= 4 ? 2 : 1;     // staging buffers of the dense front end per group
    static constexpr int STAGE_BYTES = TILE * XMAX * 4;
    static constexpr int G_BYTES = NSTG * STAGE_BYTES + A1_BYTES + A2_BYTES;
    static constexpr int OFF_B1 = GROUPS * G_BYTES, OFF_B2 = OFF_B1 + B1_BYTES, OFF_W3 = OFF_B2 + B2_BYTES;
    static constexpr int OFF_VB1 = (OFF_W3 + W3_BYTES + 127) / 128 * 128, OFF_VB2 = OFF_VB1 + B1_BYTES, OFF_VW3 = OFF_VB2 + B2_BYTES;
    static constexpr int SMEM_BYTES = policy_smem(GROUPS, G_BYTES, B1_BYTES, STEP);
    static constexpr int TMEM_COLS = GROUPS <= 4 ? 256 : 512;   // 64 columns per group: D2 overwrites D1, which is fully read before the second layer's MMAs are issued
    static_assert(K1 % 16 == 0 && K1 >= 16 && K1 <= K2, "first-layer K");
    static_assert(G_BYTES % 128 == 0 && OFF_B1 % 128 == 0 && OFF_B2 % 128 == 0 && OFF_VB1 % 128 == 0 && OFF_VB2 % 128 == 0,
                  "operand blocks are 128-byte aligned");
    static_assert(SMEM_BYTES <= SMEM_LIMIT, "shared memory");
};
static_assert(Geo<16, true>::GROUPS == 6 && Geo<32, true>::GROUPS == 6 && Geo<80, true>::GROUPS == 4, "group counts");

struct Args {
    const float *w1, *b1, *w2, *b2, *w3, *b3;
    const float *obs;                 // dense front end: [rows, obs_dim]
    float *out;
    long long rows, tiles;
    int units, segs;                  // ring front end: units = envs x segments of an env's tiles
    unsigned long long seed;
    const unsigned long long *seed_counter;   // added to seed when set (b2p_set_seed_counter)
    float noise_std, low, high;
    int obs_dim, bulk_ok;
};

// the rest of stable-baselines' model.step / model.value (b2p_step*): a NULL output is not computed
struct StepArgs {
    const float *w1, *b1, *w2, *b2, *w3, *b3;      // value tower (vf), NULL without values
    float *raw, *values, *neglogp;                  // [rows]; Args::out holds the clipped actions
    uint4 *obs16;                                   // [rows][K1] bf16 = K1 / 8 x uint4 per row
    float nlp_const;                                // 0.5 log(2 pi) + log_std
    int want_pi;                                    // any action output requested
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
                 ::"r"(tmem), "l"(ad), "l"(bd), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void group_bar(int g) { asm volatile("bar.sync %0, 128;" ::"r"(g + 1) : "memory"); }

#define B2P_LD32(taddr, v) \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, " \
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];" \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), \
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), \
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]) \
                 : "r"(taddr))

#define B2P_LD16(taddr, v) \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];" \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) \
                 : "r"(taddr))

__device__ __forceinline__ float tanh_f32(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t tanh_bf16x2(uint32_t x) {
    uint32_t y;
    asm("tanh.approx.bf16x2 %0, %1;" : "=r"(y) : "r"(x));
    return y;
}
// {lo at the lower address, hi above it}, round to nearest even
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ unsigned short bf16_bits(float v) { return (unsigned short)(pack_bf16x2(v, 0.f) & 0xFFFFu); }

// N(0, 1) of an agent row: counter-based (splitmix64 of seed and row), Box-Muller.  The row enters as seed + GOLDEN (row + 1),
// so row_noise(seed, base + row) == row_noise(seed + GOLDEN base, row): b2p_set_row_base's global row offset is folded into
// the seed on the host (row_seed) and the kernels see only local rows.
__device__ __forceinline__ float row_noise(unsigned long long seed, long long row) {
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(row + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    const float u1 = ((float)(unsigned)(z >> 40) + 1.0f) * (1.0f / 16777216.0f);       // (0, 1]
    const float u2 = (float)(unsigned)(z & 0xFFFFFFu) * (1.0f / 16777216.0f);          // [0, 1)
    return sqrtf(-2.0f * __logf(u1)) * cospif(2.0f * u2);
}

// FRONT: 0 = dense observation rows, 1 = rings with max_history 5 (every index a compile-time constant),
// 2 = rings with any max_history <= 5
// STEP: the b2p_step* variant (value tower, raw actions, neglogp, observation store; StepArgs); the b2p_act* instantiations
// ignore `s`
template <int FRONT, int TANH, bool STEP = false, int K1 = 16>
__global__ void __launch_bounds__(Geo<K1, STEP>::THREADS, 1) policy_kernel(const __grid_constant__ Args a, const __grid_constant__ Dev d,
                                                                          const __grid_constant__ StepArgs s) {
    using G = Geo<K1, STEP>;
    constexpr bool WIDE = G::WIDE;
    constexpr int GROUPS = G::GROUPS, THREADS = G::THREADS, NSTG = G::NSTG, STAGE_BYTES = G::STAGE_BYTES, G_BYTES = G::G_BYTES;
    constexpr int SBO1 = G::SBO1, A1_BYTES = G::A1_BYTES, OFF_B1 = G::OFF_B1, OFF_B2 = G::OFF_B2;
    constexpr int OFF_W3 = G::OFF_W3, OFF_VB1 = G::OFF_VB1, OFF_VB2 = G::OFF_VB2, OFF_VW3 = G::OFF_VW3, TMEM_COLS = G::TMEM_COLS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t obs_full[GROUPS][2];
    __shared__ __align__(8) uint64_t mma_bar[GROUPS];
    __shared__ uint32_t tmem_slot;
    constexpr bool RING = FRONT != 0;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int g = warp >> 2, wq = warp & 3, gt = tid & 127;          // group, TMEM lane quarter, row of the tile
    const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
    unsigned char *const sm = smem_raw + (sbase - smem_u32(smem_raw));
    unsigned char *const gsm = sm + g * G_BYTES;
    unsigned char *const A1 = gsm + NSTG * STAGE_BYTES, *const A2 = A1 + A1_BYTES;
    float *const w3s = reinterpret_cast<float *>(sm + OFF_W3);
    const int od = a.obs_dim;

    if (tid == 0) {
        for (int i = 0; i < GROUPS; ++i) { mbar_init(&obs_full[i][0], 1); mbar_init(&obs_full[i][1], 1); mbar_init(&mma_bar[i], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    // the network as bf16 B operands [N = 64 units][K], biases as one more K column (the A operands carry a 1 there)
    for (int i = tid; i < HID * K1; i += THREADS) {
        const int n = i / K1, k = i - n * K1;
        const float v = k < od ? a.w1[n * od + k] : (k == K1 - 1 ? a.b1[n] : 0.f);
        *reinterpret_cast<unsigned short *>(sm + OFF_B1 + (n >> 3) * SBO1 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) = bf16_bits(v);
    }
    for (int i = tid; i < HID * K2; i += THREADS) {
        const int n = i / K2, k = i - n * K2;
        const float v = k < HID ? a.w2[n * HID + k] : (k == HID ? a.b2[n] : 0.f);
        *reinterpret_cast<unsigned short *>(sm + OFF_B2 + (n >> 3) * SBO2 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) = bf16_bits(v);
    }
    if (tid < HID) w3s[tid] = a.w3[tid];
    if (tid == HID) w3s[HID] = a.b3[0];
    if constexpr (STEP) {
        if (s.values) {
            for (int i = tid; i < HID * K1; i += THREADS) {
                const int n = i / K1, k = i - n * K1;
                const float v = k < od ? s.w1[n * od + k] : (k == K1 - 1 ? s.b1[n] : 0.f);
                *reinterpret_cast<unsigned short *>(sm + OFF_VB1 + (n >> 3) * SBO1 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) = bf16_bits(v);
            }
            for (int i = tid; i < HID * K2; i += THREADS) {
                const int n = i / K2, k = i - n * K2;
                const float v = k < HID ? s.w2[n * HID + k] : (k == HID ? s.b2[n] : 0.f);
                *reinterpret_cast<unsigned short *>(sm + OFF_VB2 + (n >> 3) * SBO2 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) = bf16_bits(v);
            }
            float *const vw3s = reinterpret_cast<float *>(sm + OFF_VW3);
            if (tid < HID) vw3s[tid] = s.w3[tid];
            if (tid == HID) vw3s[HID] = s.b3[0];
        }
    }
    {   // constant columns of this thread's A2 row: k = 64 is the bias 1, k = 65..79 are zero
        unsigned char *row = A2 + (gt >> 3) * SBO2 + (gt & 7) * 16;
        *reinterpret_cast<uint4 *>(row + 8 * 128) = make_uint4(0x00003F80u, 0u, 0u, 0u);
        *reinterpret_cast<uint4 *>(row + 9 * 128) = make_uint4(0u, 0u, 0u, 0u);
    }
    fence_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(HID >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);   // f32 += bf16 . bf16, both K-major
    const uint64_t a1d = make_desc(sbase + g * G_BYTES + NSTG * STAGE_BYTES, 128, SBO1);
    const uint64_t a2d = make_desc(sbase + g * G_BYTES + NSTG * STAGE_BYTES + A1_BYTES, 128, SBO2);
    const uint64_t b1d = make_desc(sbase + OFF_B1, 128, SBO1), b2d = make_desc(sbase + OFF_B2, 128, SBO2);
    // the value tower's B descriptors: the action tower's moved by the offset of its operands (start address field,
    // 16-byte units; formed where used, so that they hold no registers across the tile loop)
    constexpr uint64_t VDESC_SHIFT = (uint64_t)((OFF_VB1 - OFF_B1) >> 4);
    static_assert(OFF_VB2 - OFF_B2 == OFF_VB1 - OFF_B1, "both value-tower operands sit at the same offset");
    auto want_pi = [&]() -> bool { return !STEP || s.want_pi; };     // read from the parameter space, never held in a register
    auto want_v = [&]() -> bool { return STEP && s.values; };
    const uint32_t tm1 = tmem + 64 * g, tm2 = tm1;
    // D1 = A1 . [W1 | b1]^T: K1 / 16 MMAs into the same accumulator, in K order (ppo_grad_kernel repeats it)
    auto layer1 = [&](uint64_t b1desc) {
#pragma unroll
        for (int kk = 0; kk < K1 / 16; ++kk)
            mma_bf16(tm1, a1d + (uint64_t)(kk * 16), b1desc + (uint64_t)(kk * 16), idesc, kk ? 1u : 0u);
    };
    const uint32_t tlane = (uint32_t)(wq * 32) << 16;
    const float b3 = w3s[HID];
    const unsigned long long seed = a.seed + (a.seed_counter ? *a.seed_counter : 0ull);

    // ---- front ends
    const int tiles_per_env = RING ? (d.P + TILE - 1) / TILE : 1;
    auto fetch_dense = [&](long long tile, int b) {         // observation rows of `tile` -> stage b, completes on obs_full[g][b]
        const long long row0 = tile * TILE;
        const int nrows = (int)min((long long)TILE, a.rows - row0);
        const unsigned bytes = (unsigned)(nrows * od) * 4u;
        const float *src = a.obs + row0 * od;
        float *dst = reinterpret_cast<float *>(gsm + b * STAGE_BYTES);
        if (a.bulk_ok && (bytes & 15u) == 0u) {
            if (gt == 0) {
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&obs_full[g][b])), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(&obs_full[g][b])) : "memory");
            }
        } else {                                            // ragged last tile / unaligned matrix: plain loads
            for (int i = gt; i < nrows * od; i += 128) dst[i] = src[i];
            group_bar(g);
            if (gt == 0) mbar_arrive(&obs_full[g][b]);
        }
    };
    // Ring front end.  A CTA owns "units" (env, segment of the env's tiles), u = blockIdx.x + k * gridDim.x,
    // and its four groups share a unit's tiles round robin: the env's ring position (head, nvalid) and loss
    // history sit behind a dependent load and are fetched once per unit, not once per tile.  The cursor is
    // always ONE TILE AHEAD of the tile being computed: load_ring issues the 2H loads of that tile into
    // registers (raw values) under the current tile's work, ring_row turns them into the observation row
    // when the tile's turn comes.
    struct Cursor {
        long long tile;               // dense: tile index
        int unit, tp, hi, e, head, nvalid;
        bool valid;
        float lv[XMAX / 3];           // adjusted losses newest first (0 beyond nvalid)
    };
    auto ring_enter = [&](Cursor &c) {                      // first tile of this group in unit c.unit or a later one
        for (; c.unit < a.units; c.unit += (int)gridDim.x) {
            const int e = c.unit / a.segs, sg = c.unit - e * a.segs;
            const int lo = (int)((long long)sg * tiles_per_env / a.segs), hi = (int)((long long)(sg + 1) * tiles_per_env / a.segs);
            if (lo + g >= hi) continue;
            const EnvScalars *sc = d.sc + e;
            c.e = e; c.tp = lo + g; c.hi = hi; c.head = sc->head; c.nvalid = sc->nvalid; c.valid = true;
            if constexpr (!WIDE) {
#pragma unroll
                for (int h = 0; h < XMAX / 3; ++h) {
                    const int H = FRONT == 1 ? 5 : d.H;
                    int slot = c.head - h;
                    slot += slot < 0 ? H : 0;
                    c.lv[h] = (h < H && h < c.nvalid) ? sc->adj_loss[slot] : 0.f;
                }
            }
            return;
        }
        c.valid = false;
    };
    auto advance = [&](Cursor &c) {
        if (RING) {
            c.tp += GROUPS;
            if (c.tp >= c.hi) { c.unit += (int)gridDim.x; ring_enter(c); }
        } else {
            c.tile += (long long)gridDim.x * GROUPS;
            c.valid = c.tile < a.tiles;
        }
    };
    auto load_ring = [&](const Cursor &c, float (&x)[XMAX]) {
        const int p = c.tp * TILE + gt, H = FRONT == 1 ? 5 : d.H;
        const bool ok = p < d.P;
#pragma unroll
        for (int h = 0; h < XMAX / 3; ++h) {
            float wv = 0.f, gv = 0.f;
            if (h < H) {
                int slot = c.head - h;
                slot += slot < 0 ? H : 0;
                const size_t off = ((size_t)c.e * H + slot) * d.Pp + p;
                if (ok && h < c.nvalid) { wv = d.ringw[off]; gv = d.ringg[off]; }
            }
            x[3 * h] = wv; x[3 * h + 1] = c.lv[h]; x[3 * h + 2] = gv;
        }
    };
    // Wide rows (K1 > 16): too many values to hold in registers, so the group's loads of the next tile are L2
    // prefetches issued under this tile's work, and the row is read when the tile's turn comes (wide_row below)
    auto prefetch_next = [&](const Cursor &c) {
        auto prefetch_l2 = [](const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); };
        if (RING) {                                         // 2H slot rows of 128 floats = 8H lines of 128 bytes
            const int H = d.H;
            for (int i = gt; i < 8 * H; i += 128) {
                const int h = i >> 3, p = c.tp * TILE + (i & 3) * 32;
                if (h < c.nvalid && p < d.P) {
                    int slot = c.head - h;
                    slot += slot < 0 ? H : 0;
                    prefetch_l2(((i >> 2) & 1 ? d.ringg : d.ringw) + ((size_t)c.e * H + slot) * d.Pp + p);
                }
            }
        } else {                                            // the tile's rows are contiguous
            const long long row0 = c.tile * TILE, n = min((long long)TILE, a.rows - row0) * od;
            const float *src = a.obs + row0 * od;
            for (long long i = gt * 32; i < n; i += 128 * 32) prefetch_l2(src + i);
        }
    };
    auto ring_row = [&](const float (&raw)[XMAX], float (&x)[XMAX]) {   // [adj_w (H) | adj_L (H) | adj_g (H)], clip, -1
#pragma unroll
        for (int k = 0; k < XMAX; ++k) x[k] = 0.f;
        if (FRONT == 1) {
#pragma unroll
            for (int h = 0; h < 5; ++h) { x[h] = clip_m1(raw[3 * h]); x[5 + h] = clip_m1(raw[3 * h + 1]); x[10 + h] = clip_m1(raw[3 * h + 2]); }
        } else {
            const int H = d.H;                               // rare shapes: the row is assembled with selects
#pragma unroll
            for (int k = 0; k < XMAX; ++k) {
                float v = 0.f;
#pragma unroll
                for (int h = 0; h < XMAX / 3; ++h) {
                    v = (k == h && h < H) ? raw[3 * h] : v;
                    v = (k == H + h && h < H) ? raw[3 * h + 1] : v;
                    v = (k == 2 * H + h && h < H) ? raw[3 * h + 2] : v;
                }
                x[k] = k < 3 * H ? clip_m1(v) : 0.f;
            }
        }
    };

    Cursor c;
    c.tile = (long long)blockIdx.x * GROUPS + g;
    c.unit = (int)blockIdx.x;
    c.valid = c.tile < a.tiles;
    if (RING) ring_enter(c);
    uint32_t mph = 0;
    float nxt[XMAX];
    long long tile = 0;               // the tile being computed: dense index / (env, tile of the env)
    int cur_e = 0, cur_tp = 0;
    bool have = c.valid;
    if (have) {
        if (RING) { if constexpr (!WIDE) load_ring(c, nxt); cur_e = c.e; cur_tp = c.tp; }
        else { if constexpr (!WIDE) fetch_dense(c.tile, 0); tile = c.tile; }
        advance(c);
    }
    for (int n = 0; have; ++n) {
        // ---- row of the output vectors (the next b2e_step gathers the action through the same row table)
        auto out_row = [&](bool &live) -> long long {
            if (RING) {
                const int p = cur_tp * TILE + gt;
                live = p < d.P;
                return (long long)cur_e * d.P + (live ? (d.row_lex ? d.row_of_param[p] : p) : 0);
            }
            live = tile * TILE + gt < a.rows;
            return tile * TILE + gt;
        };
        if constexpr (WIDE) {
            // ---- A1 = [row | 0 | 1] as bf16, 16 columns at a time; the observation store gets the same chunks with
            // the bias column 0.  Ring rows are assembled column by column, [adj_w (H) | adj_L (H) | adj_g (H)] newest
            // first, with the narrow front end's values and rounding, so that they equal the dense rows bit for bit.
            unsigned char *row = A1 + (gt >> 3) * SBO1 + (gt & 7) * 16;
            bool live;
            const long long orow = out_row(live);
            uint4 *const store = (STEP && s.obs16 && live) ? s.obs16 + orow * (K1 / 8) : nullptr;
            const int H = RING ? d.H : 0, p = cur_tp * TILE + gt;
            const EnvScalars *sc = d.sc + cur_e;
            const int head = RING ? sc->head : 0, nvalid = RING ? sc->nvalid : 0;
            const float *src = a.obs + (tile * TILE + gt) * od;
            auto col = [&](int k) -> float {
                if (RING) {
                    if (k >= 3 * H) return 0.f;
                    const int sg = k >= 2 * H ? 2 : (k >= H ? 1 : 0), h = k - sg * H;
                    float v = 0.f;
                    if (h < nvalid) {
                        int slot = head - h;
                        slot += slot < 0 ? H : 0;
                        if (sg == 1) v = sc->adj_loss[slot];
                        else if (p < d.P) v = (sg == 0 ? d.ringw : d.ringg)[((size_t)cur_e * H + slot) * d.Pp + p];
                    }
                    return clip_m1(v);
                }
                return (live && k < od) ? src[k] : 0.f;
            };
#pragma unroll 1
            for (int k0 = 0; k0 < K1; k0 += 16) {
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = col(k0 + i);
                const uint4 c0 = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
                uint4 c1 = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
                if (store) { store[k0 / 8] = c0; store[k0 / 8 + 1] = c1; }
                if (k0 + 16 == K1) c1.w = (c1.w & 0xFFFFu) | 0x3F800000u;      // column K1 - 1 >= obs_dim: the bias 1
                *reinterpret_cast<uint4 *>(row + (k0 / 8) * 128) = c0;
                *reinterpret_cast<uint4 *>(row + (k0 / 8 + 1) * 128) = c1;
            }
        } else {
        float x[XMAX];
        if (RING) {
            ring_row(nxt, x);
        } else {
            const int b = n % NSTG;
            if (NSTG == 2 && c.valid) fetch_dense(c.tile, b ^ 1);
            mbar_wait(&obs_full[g][b], (uint32_t)(n / NSTG) & 1u);
            const float *st = reinterpret_cast<const float *>(gsm + b * STAGE_BYTES) + gt * od;
            const bool live = tile * TILE + gt < a.rows;
#pragma unroll
            for (int k = 0; k < XMAX; ++k) x[k] = (live && k < od) ? st[k] : 0.f;
        }
        // ---- A1 = [x | 0 | 1] as bf16, this thread's row
        {
            unsigned char *row = A1 + (gt >> 3) * SBO1 + (gt & 7) * 16;
            const uint4 lo = make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
            *reinterpret_cast<uint4 *>(row) = lo;
            *reinterpret_cast<uint4 *>(row + 128) = make_uint4(pack_bf16x2(x[8], x[9]), pack_bf16x2(x[10], x[11]),
                                                               pack_bf16x2(x[12], x[13]), pack_bf16x2(x[14], 1.0f));
            if constexpr (STEP) {           // the observation store: the row as the MMA reads it, bias column -> 0
                bool live;
                const long long orow = s.obs16 ? out_row(live) : 0;
                if (s.obs16 && live) {
                    s.obs16[2 * orow] = lo;
                    s.obs16[2 * orow + 1] = make_uint4(pack_bf16x2(x[8], x[9]), pack_bf16x2(x[10], x[11]),
                                                       pack_bf16x2(x[12], x[13]), pack_bf16x2(x[14], 0.f));
                }
            }
        }
        }
        fence_async();
        tc_fence_before();
        group_bar(g);
        if (gt == 0 && (want_pi() || want_v())) {
            tc_fence_after();
            layer1(want_pi() ? b1d : b1d + VDESC_SHIFT);
            mma_commit(&mma_bar[g]);
        }
        if constexpr (!WIDE) {
            if (!RING && NSTG == 1 && c.valid) fetch_dense(c.tile, 0);      // the single staging buffer is free again (barrier above)
        }
        const bool have_next = c.valid;
        const long long next_tile = c.tile;
        const int next_e = c.e, next_tp = c.tp;
        if constexpr (WIDE) {
            if (have_next) prefetch_next(c);
        } else {
            if (RING && have_next) load_ring(c, nxt);             // in flight under this tile's work
        }
        if (have_next) advance(c);
        // ---- the rest of a tower whose first-layer MMA has been issued: -> w3 . tanh(D2) + b3 of this thread's row
        auto finish_tower = [&](uint64_t b2desc, const float *w3p, float bias) -> float {
            mbar_wait(&mma_bar[g], mph);
            mph ^= 1u;
            tc_fence_after();
            // ---- A2 = tanh(D1) as bf16, 16 accumulator columns at a time (register budget of 768 threads)
#pragma unroll
            for (int qt = 0; qt < 4; ++qt) {
                uint32_t v[16];
                B2P_LD16(tm1 + tlane + 16 * qt, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                unsigned char *row = A2 + (gt >> 3) * SBO2 + (gt & 7) * 16 + (2 * qt) * 128;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint32_t pk[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float v0 = __uint_as_float(v[8 * c + 2 * i]), v1 = __uint_as_float(v[8 * c + 2 * i + 1]);
                        pk[i] = TANH >= 1 ? tanh_bf16x2(pack_bf16x2(v0, v1)) : pack_bf16x2(tanh_f32(v0), tanh_f32(v1));
                    }
                    *reinterpret_cast<uint4 *>(row + c * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
            fence_async();
            tc_fence_before();
            group_bar(g);
            if (gt == 0) {
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < K2 / 16; ++kk)              // 16 K elements = two core matrices = 256 bytes per MMA
                    mma_bf16(tm2, a2d + (uint64_t)(kk * 16), b2desc + (uint64_t)(kk * 16), idesc, kk ? 1u : 0u);
                mma_commit(&mma_bar[g]);
            }
            mbar_wait(&mma_bar[g], mph);
            mph ^= 1u;
            tc_fence_after();
            // ---- head: tanh(D2) . w3 + b3
            float acc0 = bias, acc1 = 0.f;
#pragma unroll
            for (int qt = 0; qt < 4; ++qt) {
                uint32_t v[16];
                B2P_LD16(tm2 + tlane + 16 * qt, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 w = *reinterpret_cast<const float4 *>(w3p + 16 * qt + 4 * c);
                    float t0, t1, t2, t3;
                    if (TANH == 2) {
                        const uint32_t p0 = tanh_bf16x2(pack_bf16x2(__uint_as_float(v[4 * c]), __uint_as_float(v[4 * c + 1])));
                        const uint32_t p1 = tanh_bf16x2(pack_bf16x2(__uint_as_float(v[4 * c + 2]), __uint_as_float(v[4 * c + 3])));
                        t0 = __uint_as_float(p0 << 16); t1 = __uint_as_float(p0 & 0xFFFF0000u);
                        t2 = __uint_as_float(p1 << 16); t3 = __uint_as_float(p1 & 0xFFFF0000u);
                    } else {
                        t0 = tanh_f32(__uint_as_float(v[4 * c])); t1 = tanh_f32(__uint_as_float(v[4 * c + 1]));
                        t2 = tanh_f32(__uint_as_float(v[4 * c + 2])); t3 = tanh_f32(__uint_as_float(v[4 * c + 3]));
                    }
                    acc0 = fmaf(t0, w.x, acc0); acc1 = fmaf(t1, w.y, acc1);
                    acc0 = fmaf(t2, w.z, acc0); acc1 = fmaf(t3, w.w, acc1);
                }
            }
            tc_fence_before();
            return acc0 + acc1;
        };
        if constexpr (!STEP) {
            float mean = finish_tower(b2d, w3s, b3);
            bool live;
            const long long orow = out_row(live);
            if (a.noise_std != 0.f) mean = fmaf(a.noise_std, row_noise(seed, orow), mean);
            if (live) a.out[orow] = fminf(fmaxf(mean, a.low), a.high);
        } else {
            // the action outputs are stored before the value tower runs, so that nothing of them stays live across it
            if (want_pi()) {
                const float mean = finish_tower(b2d, w3s, w3s[HID]);
                bool live;
                const long long orow = out_row(live);
                float z = 0.f, raw = mean;
                if (a.noise_std != 0.f) { z = row_noise(seed, orow); raw = fmaf(a.noise_std, z, mean); }
                if (live) {
                    if (a.out) a.out[orow] = fminf(fmaxf(raw, a.low), a.high);
                    if (s.raw) s.raw[orow] = raw;
                    if (s.neglogp) s.neglogp[orow] = fmaf(0.5f * z, z, s.nlp_const);
                }
            }
            if (want_v()) {
                if (want_pi()) {          // the value tower reuses D1/D2 (read out above) and A2 (the last MMA has completed)
                    group_bar(g);
                    if (gt == 0) {
                        tc_fence_after();
                        layer1(b1d + VDESC_SHIFT);
                        mma_commit(&mma_bar[g]);
                    }
                }
                const float *vw3s = reinterpret_cast<const float *>(sm + OFF_VW3);
                const float value = finish_tower(b2d + VDESC_SHIFT, vw3s, vw3s[HID]);
                bool live;
                const long long orow = out_row(live);
                if (live) s.values[orow] = value;
            }
        }
        have = have_next; tile = next_tile; cur_e = next_e; cur_tp = next_tp;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS));
}

// GAE of stable-baselines 2's PPO2 Runner (ppo2.py) over a time-major rollout, one thread per agent row, T sequential:
//   nn = 1 - dones[t+1];  delta = r[t] + gamma * values[t+1] * nn - values[t];  adv[t] = last = delta + gamma * lam * nn * last
//   ret[t] = adv[t] + values[t]
// in the Runner's dtypes: gamma * values[t+1] is a float32 product (a Python float times a float32 array), the rest of
// delta and the recursion are float64 (1.0 - a bool array is float64), adv is stored as float32 and ret = adv + value is
// a float32 sum.  Explicit _rn intrinsics: no FMA contraction the numpy code does not have.  The values of U steps are
// loaded ahead of their recursion; rewards and dones are per env (env = row / P) and shared by its rows through the cache.
constexpr int GAE_THREADS = 256, GAE_U = 8;
__global__ void __launch_bounds__(GAE_THREADS) gae_kernel(const float *__restrict__ values, const float *__restrict__ rewards,
                                                          const uint8_t *__restrict__ dones, int T, long long rows, long long P,
                                                          double gamma, double lam, float *__restrict__ adv, float *__restrict__ ret) {
    const long long row = (long long)blockIdx.x * GAE_THREADS + threadIdx.x;
    if (row >= rows) return;
    const long long E = rows / P, e = row / P;
    const double gl = __dmul_rn(gamma, lam);
    const float g32 = (float)gamma;
    double last = 0.0;
    float nv = __ldcs(values + (size_t)T * rows + row);
    for (int t0 = T - 1; t0 >= 0; t0 -= GAE_U) {
        float v[GAE_U], r[GAE_U];
        uint8_t dn[GAE_U];
#pragma unroll
        for (int i = 0; i < GAE_U; ++i) {
            const int t = t0 - i;
            if (t >= 0) {
                v[i] = __ldcs(values + (size_t)t * rows + row);
                r[i] = __ldg(rewards + (size_t)t * E + e);
                dn[i] = __ldg(dones + (size_t)(t + 1) * E + e);
            }
        }
#pragma unroll
        for (int i = 0; i < GAE_U; ++i) {
            const int t = t0 - i;
            if (t >= 0) {
                const double nn = dn[i] ? 0.0 : 1.0;
                const double delta = __dadd_rn(__dadd_rn((double)r[i], __dmul_rn((double)__fmul_rn(g32, nv), nn)), -(double)v[i]);
                last = __dadd_rn(delta, __dmul_rn(__dmul_rn(gl, nn), last));
                const float a32 = (float)last;
                __stcs(adv + (size_t)t * rows + row, a32);
                __stcs(ret + (size_t)t * rows + row, __fadd_rn(a32, v[i]));
                nv = v[i];
            }
        }
    }
}

// ---------------------------------------------------------------- PPO update (b2p_ppo_*)
// Minibatch order: a keyed Feistel network on 2 x `bits` bits (4^bits >= n), cycle-walked into [0, n): a
// permutation of [0, n) that needs no stored index array.  Position p of the order is perm(p).
constexpr int FEISTEL_ROUNDS = 6;
struct Feistel {
    unsigned long long key[FEISTEL_ROUNDS], mask, n;
    int bits;
};
__host__ __device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ long long feistel_at(const Feistel &f, long long p) {
    unsigned long long v = (unsigned long long)p;
    do {
        unsigned long long L = v >> f.bits, R = v & f.mask;
#pragma unroll
        for (int r = 0; r < FEISTEL_ROUNDS; ++r) {
            const unsigned long long nr = L ^ (mix64(R ^ f.key[r]) & f.mask);
            L = R;
            R = nr;
        }
        v = (L << f.bits) | R;
    } while (v >= f.n);
    return (long long)v;
}

// tanh.approx.bf16x2 of every bf16 input, as the policy kernels evaluate it in the bf16 tanh modes (b2p_tanh_table)
__global__ void tanh_bf16_table_kernel(float *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 65536) out[i] = __uint_as_float(tanh_bf16x2((uint32_t)i) << 16);
}

__global__ void ppo_indices_kernel(const Feistel f, long long begin, long long count, long long *__restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
        out[i] = feistel_at(f, begin + i);
}

// a DeviceRolloutBuffer seen through flat time-major indices j = t * rows + row (values: its first T rows)
struct PpoBatch {
    const uint4 *obs;                                  // K1 / 8 x uint4 per row (b2p_obs_width bf16)
    const float *act, *nlp, *val, *ret;
};

// Advantage statistics of every minibatch of an epoch: block (m, c) sums A - K over its slice of minibatch m's
// positions in fp64, thread-strided then a fixed tree (K = A at the minibatch's first position: a shift that keeps
// the sum of squares well conditioned); ppo_adv_final sums a minibatch's slices in order.
constexpr int ADV_THREADS = 256;
constexpr long long ADV_SLICE = 65536;
__device__ __forceinline__ float adv_of(const PpoBatch &b, long long j) { return __fsub_rn(b.ret[j], b.val[j]); }
__global__ void __launch_bounds__(ADV_THREADS) ppo_adv_partial(const PpoBatch b, const Feistel f, long long mb, int slices,
                                                               double *__restrict__ part) {
    __shared__ double s1[ADV_THREADS], s2[ADV_THREADS];
    const long long m = blockIdx.x / slices;
    const int c = (int)(blockIdx.x - m * slices);
    const long long len = (mb + slices - 1) / slices, lo = m * mb + c * len, hi = min(m * mb + mb, lo + len);
    const double K = (double)adv_of(b, feistel_at(f, m * mb));
    double a1 = 0.0, a2 = 0.0;
    for (long long p = lo + threadIdx.x; p < hi; p += ADV_THREADS) {
        const double d = (double)adv_of(b, feistel_at(f, p)) - K;
        a1 += d;
        a2 = fma(d, d, a2);
    }
    s1[threadIdx.x] = a1; s2[threadIdx.x] = a2;
    __syncthreads();
    for (int w = ADV_THREADS / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) { s1[threadIdx.x] += s1[threadIdx.x + w]; s2[threadIdx.x] += s2[threadIdx.x + w]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { part[2 * blockIdx.x] = s1[0]; part[2 * blockIdx.x + 1] = s2[0]; }
}
// moments[m] = {count, K, sum(A - K), sum((A - K)^2)} of minibatch m: its slices summed in order (b2p_ppo_adv_moments)
__global__ void ppo_adv_moments_kernel(const PpoBatch b, const Feistel f, long long mb, long long nmb, int slices,
                                       const double *__restrict__ part, double *__restrict__ moments) {
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= nmb) return;
    double a1 = 0.0, a2 = 0.0;
    for (int c = 0; c < slices; ++c) { a1 += part[2 * (m * slices + c)]; a2 += part[2 * (m * slices + c) + 1]; }
    moments[4 * m] = (double)mb;
    moments[4 * m + 1] = (double)adv_of(b, feistel_at(f, m * mb));
    moments[4 * m + 2] = a1;
    moments[4 * m + 3] = a2;
}
// the moments of `ranks` shards ([ranks][nmb][4], rank order) -> mean and population std of every union minibatch
// (b2p_ppo_adv_combine).  Rank r's sums are moved to rank 0's shift K_0 (d = K_r - K_0):
//   sum(A - K_0) += S1_r + n_r d,   sum((A - K_0)^2) += S2_r + d (2 S1_r + n_r d)
// One rank is rank 0's sums as they are, so b2p_ppo_adv_stats (moments, then this with one rank) keeps its bits.
__global__ void ppo_adv_combine_kernel(const double *__restrict__ moments, int ranks, long long nmb, double *__restrict__ stats) {
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= nmb) return;
    const double *q = moments + 4 * m;
    double n = q[0], a1 = q[2], a2 = q[3];
    const double K = q[1];
    for (int r = 1; r < ranks; ++r) {
        q = moments + 4 * ((long long)r * nmb + m);
        const double d = q[1] - K;
        a1 += q[2] + q[0] * d;
        a2 += q[3] + d * (2.0 * q[2] + q[0] * d);
        n += q[0];
    }
    const double mean = a1 / n, var = a2 / n - mean * mean;
    stats[2 * m] = K + mean;
    stats[2 * m + 1] = sqrt(var > 0.0 ? var : 0.0);                 // population std
}

// The clipped-surrogate gradient of both towers over one minibatch (b2p_ppo_grad).  Per 128-row tile a group
// gathers its rows by index, runs the forward of each tower exactly as policy_kernel's step variant does (same
// operands, MMAs, tanh and head FMA order, so the values at the rollout's weights are the rollout's bits), forms the
// per-row loss derivative g, and runs the tower's backward on the tensor cores:
//   dPre2 = g w3 (1 - h2^2)             bf16 tile [128 rows x 64], K-major (the thread's row)
//   dH1   = dPre2 . W2                   M 128, N 64, K 64: A = dPre2 (K-major), B = [W2 | b2] operand read MN-major
//   dPre1 = dH1 (1 - h1^2)               h1 = the bf16 operand of the second forward MMA
//   [dW2 | db2] += dPre2^T . [h1 | 1]    M 64, N 80, K 128 rows: both operands read MN-major
//   [dW1 | db1] += dPre1^T . A1          M 64, N K1, K 128 rows
//   dw3 += g h2, db3 += g                FFMA: g h2 staged in shared memory as fp32, column sums in fixed order
// MN-major no-swizzle descriptors for bf16: LBO = stride between 8-row K groups, SBO = stride between 8-element MN
// groups (128 B).  An M = 64 accumulator holds row j in TMEM lane (j % 16) + 32 (j / 16).
// TMEM per group: 64 working columns (D1, D2 / h2, dH1) + 2 x (80 + K1) private accumulators.  That is 256 at K1 = 16,
// so two groups share the 512 columns; the wide variants (K1 = 32 .. 80) need 288 .. 384 and run one group per CTA.
// The accumulators are read out and added into the group's fp32 slot of the workspace every FLUSH tiles (the tensor
// core's adder truncates over long sums); ppo_reduce sums the slots in fp64 in a fixed order.
namespace ppo {
constexpr int FLUSH = 16;
constexpr int SBO_P = (HID / 8) * 128, P_BYTES = (TILE / 8) * SBO_P;      // dPre tiles [128 x 64] bf16
constexpr int S_STRIDE = HID + 1, S_BYTES = (TILE * S_STRIDE * 4 + 127) / 128 * 128;   // g h2 stage, fp32
constexpr int TMEM_COLS = 512;
constexpr int NSTATS = 5;                     // per-slot sums: pg, max(vf losses), (nlp - nlp_old)^2, clipped, dL/dlog_std
constexpr int tmem_per_group(int k1) { return 64 + 2 * (K2 + k1); }
constexpr int groups(int k1) { return tmem_per_group(k1) <= 256 ? 2 : 1; }
template <int K1>
struct Geo {
    static constexpr int GROUPS = groups(K1), THREADS = GROUPS * 128;
    static constexpr int SBO1 = pol::Geo<K1, true>::SBO1, A1_BYTES = pol::Geo<K1, true>::A1_BYTES, B1_BYTES = pol::Geo<K1, true>::B1_BYTES;
    static constexpr int ACC_STRIDE = K2 + K1;                                // accumulator columns of one tower: [dW2 | db2 | 0], [dW1 | db1]
    static constexpr int TMEM_STRIDE = TMEM_COLS / GROUPS;                    // TMEM columns of one group
    static constexpr int G_BYTES = A1_BYTES + A2_BYTES + 2 * P_BYTES + S_BYTES;
    static constexpr int TOWER_OPS = B1_BYTES + B2_BYTES;                     // [W1 | b1] and [W2 | b2] of one tower
    static constexpr int OFF_W = GROUPS * G_BYTES, OFF_W3 = OFF_W + 2 * TOWER_OPS;
    static constexpr int SMEM_BYTES = OFF_W3 + 2 * W3_BYTES + 128;
    static_assert(G_BYTES % 128 == 0 && OFF_W % 128 == 0 && TOWER_OPS % 128 == 0, "operand blocks are 128-byte aligned");
    static_assert(SMEM_BYTES <= SMEM_LIMIT, "shared memory");
    static_assert(tmem_per_group(K1) <= TMEM_STRIDE, "tensor memory");
};
static_assert(Geo<16>::GROUPS == 2 && Geo<16>::TMEM_STRIDE == 256 && Geo<80>::GROUPS == 1, "group counts");
}  // namespace ppo

struct GradArgs {
    const float *w;                   // the handle's weights: action tower, value tower
    PpoBatch b;
    Feistel f;
    long long begin, count, tiles;
    const double *adv_stats;          // mean, std of this minibatch's advantages
    float clip, clip_vf, vf_coef, inv_n, inv_sigma, nlp_const;
    float *ws_grad;                   // [slots][stride]
    double *ws_stats;                 // [slots][NSTATS]
    int od, tf, stride;
};

#define B2P_ST16(taddr, v) \
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" \
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), \
                   "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory")

template <int TANH, int K1 = 16>
__global__ void __launch_bounds__(ppo::Geo<K1>::THREADS, 1) ppo_grad_kernel(const __grid_constant__ GradArgs a) {
    using PG = ppo::Geo<K1>;
    constexpr bool WIDE = K1 > 16;
    constexpr int GROUPS = PG::GROUPS, THREADS = PG::THREADS, FLUSH = ppo::FLUSH, SBO_P = ppo::SBO_P, P_BYTES = ppo::P_BYTES;
    constexpr int S_STRIDE = ppo::S_STRIDE, G_BYTES = PG::G_BYTES, TOWER_OPS = PG::TOWER_OPS, OFF_W = PG::OFF_W;
    constexpr int OFF_W3 = PG::OFF_W3, TMEM_COLS = ppo::TMEM_COLS, NSTATS = ppo::NSTATS;
    constexpr int SBO1 = PG::SBO1, A1_BYTES = PG::A1_BYTES, B1_BYTES = PG::B1_BYTES, ACC = PG::ACC_STRIDE;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t mma_bar[GROUPS];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int g = warp >> 2, wq = warp & 3, gt = tid & 127;
    const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
    unsigned char *const sm = smem_raw + (sbase - smem_u32(smem_raw));
    unsigned char *const A1 = sm + g * G_BYTES, *const H = A1 + A1_BYTES, *const P2 = H + A2_BYTES, *const P1 = P2 + P_BYTES;
    float *const S = reinterpret_cast<float *>(P1 + P_BYTES);
    const uint32_t a1s = sbase + g * G_BYTES, hs = a1s + A1_BYTES, p2s = hs + A2_BYTES, p1s = p2s + P_BYTES;
    const int od = a.od;
    const int slot = blockIdx.x * GROUPS + g;
    float *const wsg = a.ws_grad + (size_t)slot * a.stride;

    if (tid == 0) {
        for (int i = 0; i < GROUPS; ++i) mbar_init(&mma_bar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    for (int tw = 0; tw < 2; ++tw) {      // both towers' operands, in policy_kernel's layouts
        const float *w1 = a.w + tw * a.tf, *b1 = w1 + HID * od, *w2 = b1 + HID, *b2 = w2 + HID * HID, *w3 = b2 + HID;
        unsigned char *ob1 = sm + OFF_W + tw * TOWER_OPS, *ob2 = ob1 + B1_BYTES;
        for (int i = tid; i < HID * K1; i += THREADS) {
            const int n = i / K1, k = i - n * K1;
            const float v = k < od ? w1[n * od + k] : (k == K1 - 1 ? b1[n] : 0.f);
            *reinterpret_cast<unsigned short *>(ob1 + (n >> 3) * SBO1 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) = bf16_bits(v);
        }
        for (int i = tid; i < HID * K2; i += THREADS) {
            const int n = i / K2, k = i - n * K2;
            const float v = k < HID ? w2[n * HID + k] : (k == HID ? b2[n] : 0.f);
            *reinterpret_cast<unsigned short *>(ob2 + (n >> 3) * SBO2 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) = bf16_bits(v);
        }
        float *w3s = reinterpret_cast<float *>(sm + OFF_W3) + tw * (HID + 4);
        if (tid <= HID) w3s[tid] = w3[tid];                 // w3 then b3
    }
    {
        unsigned char *row = H + (gt >> 3) * SBO2 + (gt & 7) * 16;
        *reinterpret_cast<uint4 *>(row + 8 * 128) = make_uint4(0x00003F80u, 0u, 0u, 0u);
        *reinterpret_cast<uint4 *>(row + 9 * 128) = make_uint4(0u, 0u, 0u, 0u);
    }
    for (int i = gt; i < a.stride; i += 128) wsg[i] = 0.f;
    fence_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t twk = tmem + PG::TMEM_STRIDE * g;      // working columns; accumulators of tower tw at + 64 + (80 + K1) tw
    const uint32_t tlane = (uint32_t)(wq * 32) << 16;
    constexpr uint32_t F32_BF16 = (1u << 4) | (1u << 7) | (1u << 10), A_MN = 1u << 15, B_MN = 1u << 16;
    const uint32_t idesc = F32_BF16 | ((uint32_t)(HID >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);
    const uint32_t idesc_dh = idesc | B_MN;
    const uint32_t idesc_w2 = F32_BF16 | A_MN | B_MN | ((uint32_t)(K2 >> 3) << 17) | ((uint32_t)(64 >> 4) << 24);
    const uint32_t idesc_w1 = F32_BF16 | A_MN | B_MN | ((uint32_t)(K1 >> 3) << 17) | ((uint32_t)(64 >> 4) << 24);
    const uint64_t a1d = make_desc(a1s, 128, SBO1), hd = make_desc(hs, 128, SBO2);
    const uint64_t b1d = make_desc(sbase + OFF_W, 128, SBO1), b2d = make_desc(sbase + OFF_W + B1_BYTES, 128, SBO2);
    const uint64_t b2mn = make_desc(sbase + OFF_W + B1_BYTES, SBO2, 128);        // [W2 | b2] read as B[N = in][K = out]
    const uint64_t p2k = make_desc(p2s, 128, SBO_P), p2mn = make_desc(p2s, SBO_P, 128), p1mn = make_desc(p1s, SBO_P, 128);
    const uint64_t hmn = make_desc(hs, SBO2, 128), a1mn = make_desc(a1s, SBO1, 128);
    const float *const w3all = reinterpret_cast<const float *>(sm + OFF_W3);
    const double adv_mean = a.adv_stats[0], adv_inv = 1.0 / (a.adv_stats[1] + 1e-8);

    uint32_t mph = 0;
    auto mma_wait = [&]() { mbar_wait(&mma_bar[g], mph); mph ^= 1u; tc_fence_after(); };
    auto issue_begin = [&]() -> bool {                     // every thread's operand writes are visible to the MMA issuer
        fence_async();
        tc_fence_before();
        group_bar(g);
        if (gt == 0) tc_fence_after();
        return gt == 0;
    };
    // forward of tower tw on the A1 tile: policy_kernel's finish_tower, plus h2 written back over D2 for the backward
    auto forward = [&](int tw) -> float {
        const uint64_t shift = (uint64_t)(tw * (TOWER_OPS >> 4));
        if (issue_begin()) {                                // policy_kernel's layer1: the same MMAs in the same K order
#pragma unroll
            for (int kk = 0; kk < K1 / 16; ++kk)
                mma_bf16(twk, a1d + (uint64_t)(kk * 16), b1d + shift + (uint64_t)(kk * 16), idesc, kk ? 1u : 0u);
            mma_commit(&mma_bar[g]);
        }
        mma_wait();
#pragma unroll
        for (int qt = 0; qt < 4; ++qt) {
            uint32_t v[16];
            B2P_LD16(twk + tlane + 16 * qt, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            unsigned char *row = H + (gt >> 3) * SBO2 + (gt & 7) * 16 + (2 * qt) * 128;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t pk[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float v0 = __uint_as_float(v[8 * c + 2 * i]), v1 = __uint_as_float(v[8 * c + 2 * i + 1]);
                    pk[i] = TANH >= 1 ? tanh_bf16x2(pack_bf16x2(v0, v1)) : pack_bf16x2(tanh_f32(v0), tanh_f32(v1));
                }
                *reinterpret_cast<uint4 *>(row + c * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
        }
        if (issue_begin()) {
#pragma unroll
            for (int kk = 0; kk < K2 / 16; ++kk)
                mma_bf16(twk, hd + (uint64_t)(kk * 16), b2d + shift + (uint64_t)(kk * 16), idesc, kk ? 1u : 0u);
            mma_commit(&mma_bar[g]);
        }
        mma_wait();
        const float *w3p = w3all + tw * (HID + 4);
        float acc0 = w3p[HID], acc1 = 0.f;
#pragma unroll
        for (int qt = 0; qt < 4; ++qt) {
            uint32_t v[16];
            B2P_LD16(twk + tlane + 16 * qt, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float4 w = *reinterpret_cast<const float4 *>(w3p + 16 * qt + 4 * c);
                float t0, t1, t2, t3;
                if (TANH == 2) {
                    const uint32_t q0 = tanh_bf16x2(pack_bf16x2(__uint_as_float(v[4 * c]), __uint_as_float(v[4 * c + 1])));
                    const uint32_t q1 = tanh_bf16x2(pack_bf16x2(__uint_as_float(v[4 * c + 2]), __uint_as_float(v[4 * c + 3])));
                    t0 = __uint_as_float(q0 << 16); t1 = __uint_as_float(q0 & 0xFFFF0000u);
                    t2 = __uint_as_float(q1 << 16); t3 = __uint_as_float(q1 & 0xFFFF0000u);
                } else {
                    t0 = tanh_f32(__uint_as_float(v[4 * c])); t1 = tanh_f32(__uint_as_float(v[4 * c + 1]));
                    t2 = tanh_f32(__uint_as_float(v[4 * c + 2])); t3 = tanh_f32(__uint_as_float(v[4 * c + 3]));
                }
                acc0 = fmaf(t0, w.x, acc0); acc1 = fmaf(t1, w.y, acc1);
                acc0 = fmaf(t2, w.z, acc0); acc1 = fmaf(t3, w.w, acc1);
                v[4 * c] = __float_as_uint(t0); v[4 * c + 1] = __float_as_uint(t1);
                v[4 * c + 2] = __float_as_uint(t2); v[4 * c + 3] = __float_as_uint(t3);
            }
            B2P_ST16(twk + tlane + 16 * qt, v);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        return acc0 + acc1;
    };
    float dw3acc[2] = {0.f, 0.f}, db3acc[2] = {0.f, 0.f};
    bool fresh = true;                                     // the accumulators start from zero at the next tile
    // backward of tower tw for this row's dL/d(output) = gr (0 for rows past the minibatch)
    auto backward = [&](int tw, float gr) {
        const float *w3p = w3all + tw * (HID + 4);
        unsigned char *prow = P2 + (gt >> 3) * SBO_P + (gt & 7) * 16;
        float *srow = S + gt * S_STRIDE;
#pragma unroll
        for (int qt = 0; qt < 4; ++qt) {
            uint32_t v[16];
            B2P_LD16(twk + tlane + 16 * qt, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t pk[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int j0 = 16 * qt + 8 * c + 2 * i;
                    const float h0 = __uint_as_float(v[8 * c + 2 * i]), h1 = __uint_as_float(v[8 * c + 2 * i + 1]);
                    pk[i] = pack_bf16x2(gr * w3p[j0] * fmaf(-h0, h0, 1.f), gr * w3p[j0 + 1] * fmaf(-h1, h1, 1.f));
                    srow[j0] = gr * h0;
                    srow[j0 + 1] = gr * h1;
                }
                *reinterpret_cast<uint4 *>(prow + (2 * qt + c) * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
        }
        const uint32_t acc_w2 = twk + 64 + ACC * tw, acc_w1 = acc_w2 + K2;
        if (issue_begin()) {
            const uint64_t shift = (uint64_t)(tw * (TOWER_OPS >> 4));
#pragma unroll
            for (int kk = 0; kk < HID / 16; ++kk)
                mma_bf16(twk, p2k + (uint64_t)(kk * 16), b2mn + shift + (uint64_t)(kk * (2 * SBO2 >> 4)), idesc_dh, kk ? 1u : 0u);
#pragma unroll
            for (int kk = 0; kk < TILE / 16; ++kk)
                mma_bf16(acc_w2, p2mn + (uint64_t)(kk * (2 * SBO_P >> 4)), hmn + (uint64_t)(kk * (2 * SBO2 >> 4)), idesc_w2,
                         (kk || !fresh) ? 1u : 0u);
            mma_commit(&mma_bar[g]);
        }
        {   // dw3 under the MMAs: column j = gt % 64 over rows 64 (gt / 64) .. + 63
            const float *col = S + (gt >> 6) * 64 * S_STRIDE + (gt & 63);
            float s = 0.f;
#pragma unroll 8
            for (int r = 0; r < 64; ++r) s += col[r * S_STRIDE];
            dw3acc[tw] += s;
            db3acc[tw] += gr;
        }
        mma_wait();
        const unsigned char *hrow = H + (gt >> 3) * SBO2 + (gt & 7) * 16;
        unsigned char *p1row = P1 + (gt >> 3) * SBO_P + (gt & 7) * 16;
#pragma unroll
        for (int qt = 0; qt < 4; ++qt) {
            uint32_t v[16];
            B2P_LD16(twk + tlane + 16 * qt, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const uint4 hv = *reinterpret_cast<const uint4 *>(hrow + (2 * qt + c) * 128);
                const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
                uint32_t pk[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float h0 = __uint_as_float(hw[i] << 16), h1 = __uint_as_float(hw[i] & 0xFFFF0000u);
                    pk[i] = pack_bf16x2(__uint_as_float(v[8 * c + 2 * i]) * fmaf(-h0, h0, 1.f),
                                        __uint_as_float(v[8 * c + 2 * i + 1]) * fmaf(-h1, h1, 1.f));
                }
                *reinterpret_cast<uint4 *>(p1row + (2 * qt + c) * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
        }
        if (issue_begin()) {
#pragma unroll
            for (int kk = 0; kk < TILE / 16; ++kk)
                mma_bf16(acc_w1, p1mn + (uint64_t)(kk * (2 * SBO_P >> 4)), a1mn + (uint64_t)(kk * (2 * SBO1 >> 4)), idesc_w1,
                         (kk || !fresh) ? 1u : 0u);
            mma_commit(&mma_bar[g]);
        }
        mma_wait();
    };
    // accumulators -> the group's workspace slot (fp32 adds, one owner per element)
    auto flush = [&]() {
        const int lane = gt & 31, j = wq * 16 + (lane & 15);
        for (int tw = 0; tw < 2; ++tw) {
            float *base = wsg + tw * a.tf;
            float *dw1 = base, *db1 = dw1 + HID * od, *dw2 = db1 + HID, *db2 = dw2 + HID * HID;
            const uint32_t acc_w2 = twk + 64 + ACC * tw, acc_w1 = acc_w2 + K2;
            for (int q = 0; q < K2 / 16; ++q) {
                uint32_t v[16];
                B2P_LD16(acc_w2 + tlane + 16 * q, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (lane < 16) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const int col = 16 * q + i;
                        if (col < HID) dw2[j * HID + col] += __uint_as_float(v[i]);
                        else if (col == HID) db2[j] += __uint_as_float(v[i]);
                    }
                }
            }
            if constexpr (!WIDE) {
                uint32_t v[16];
                B2P_LD16(acc_w1 + tlane, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (lane < 16) {
#pragma unroll
                    for (int k = 0; k < K1 - 1; ++k)
                        if (k < od) dw1[j * od + k] += __uint_as_float(v[k]);
                    db1[j] += __uint_as_float(v[K1 - 1]);
                }
            } else {
                for (int q = 0; q < K1 / 16; ++q) {
                    uint32_t v[16];
                    B2P_LD16(acc_w1 + tlane + 16 * q, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    if (lane < 16) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int k = 16 * q + i;
                            if (k < od) dw1[j * od + k] += __uint_as_float(v[i]);
                            else if (k == K1 - 1) db1[j] += __uint_as_float(v[i]);
                        }
                    }
                }
            }
            S[gt] = dw3acc[tw];
            S[128 + gt] = db3acc[tw];
            group_bar(g);
            float *dw3 = db2 + HID;
            if (gt < HID) dw3[gt] += S[gt] + S[gt + 64];
            if (gt == 0) {
                float s = 0.f;
                for (int r = 0; r < 128; ++r) s += S[128 + r];
                dw3[HID] += s;
            }
            group_bar(g);
            dw3acc[tw] = db3acc[tw] = 0.f;
        }
        tc_fence_before();
    };

    double st[NSTATS] = {0.0, 0.0, 0.0, 0.0, 0.0};
    struct Row { uint4 o0, o1; float act, nlp, val, ret; bool live; };
    auto fetch = [&](long long tile, Row &r) {
        const long long q = tile * TILE + gt;
        r.live = q < a.count;
        if (r.live) {
            const long long j = feistel_at(a.f, a.begin + q);
            r.o0 = __ldg(a.b.obs + 2 * j); r.o1 = __ldg(a.b.obs + 2 * j + 1);
            r.act = __ldg(a.b.act + j); r.nlp = __ldg(a.b.nlp + j); r.val = __ldg(a.b.val + j); r.ret = __ldg(a.b.ret + j);
        } else {
            r.o0 = r.o1 = make_uint4(0u, 0u, 0u, 0u);
            r.act = r.nlp = r.val = r.ret = 0.f;
        }
    };
    // wide rows (K1 > 16) are not held in registers a tile ahead: the next tile's sample index is, and its row and
    // scalars are prefetched to L2 under this tile's work
    auto locate = [&](long long tile) -> long long {       // -1 past the minibatch
        const long long q = tile * TILE + gt;
        if (q >= a.count) return -1;
        const long long j = feistel_at(a.f, a.begin + q);
        auto prefetch_l2 = [](const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); };
        const unsigned char *o = reinterpret_cast<const unsigned char *>(a.b.obs + j * (K1 / 8));
        prefetch_l2(o);
        prefetch_l2(o + 2 * K1 - 1);
        prefetch_l2(a.b.act + j); prefetch_l2(a.b.nlp + j); prefetch_l2(a.b.val + j); prefetch_l2(a.b.ret + j);
        return j;
    };
    const long long step = (long long)gridDim.x * GROUPS;
    long long tile = (long long)blockIdx.x * GROUPS + g;
    Row nx;
    long long nj = -1;
    if (tile < a.tiles) {
        if constexpr (WIDE) nj = locate(tile);
        else fetch(tile, nx);
    }
    for (int since = 0; tile < a.tiles; tile += step) {
        const Row cur = [&]() -> Row {
            if constexpr (WIDE) {                   // A1 = the stored bf16 row with the bias column K1 - 1 set to 1
                Row r;
                r.live = nj >= 0;
                r.act = r.live ? __ldg(a.b.act + nj) : 0.f; r.nlp = r.live ? __ldg(a.b.nlp + nj) : 0.f;
                r.val = r.live ? __ldg(a.b.val + nj) : 0.f; r.ret = r.live ? __ldg(a.b.ret + nj) : 0.f;
                unsigned char *row = A1 + (gt >> 3) * SBO1 + (gt & 7) * 16;
#pragma unroll
                for (int c = 0; c < K1 / 8; ++c) {
                    uint4 o = r.live ? __ldg(a.b.obs + nj * (K1 / 8) + c) : make_uint4(0u, 0u, 0u, 0u);
                    if (c == K1 / 8 - 1 && r.live) o.w = (o.w & 0xFFFFu) | 0x3F800000u;
                    *reinterpret_cast<uint4 *>(row + c * 128) = o;
                }
                return r;
            } else {
                return nx;
            }
        }();
        if constexpr (!WIDE) {   // A1 = the stored bf16 row with the bias column 15 set to 1
            unsigned char *row = A1 + (gt >> 3) * SBO1 + (gt & 7) * 16;
            uint4 o1 = cur.o1;
            if (cur.live) o1.w = (o1.w & 0xFFFFu) | 0x3F800000u;
            *reinterpret_cast<uint4 *>(row) = cur.o0;
            *reinterpret_cast<uint4 *>(row + 128) = o1;
        }
        if (tile + step < a.tiles) {                        // in flight under this tile's work
            if constexpr (WIDE) nj = locate(tile + step);
            else fetch(tile + step, nx);
        }
        // ---- action tower: dL/dmu of the clipped surrogate (TF gradient rules: max -> first operand on ties,
        // clip passes inside the closed interval)
        const float mu = forward(0);
        float gpi = 0.f;
        if (cur.live) {
            const float adv = (float)(((double)__fsub_rn(cur.ret, cur.val) - adv_mean) * adv_inv);
            const float z = (cur.act - mu) * a.inv_sigma;
            const float nlp = fmaf(0.5f * z, z, a.nlp_const);
            const float ratio = expf(cur.nlp - nlp);
            const float lo = 1.f - a.clip, hi = 1.f + a.clip;
            const float l1 = -adv * ratio, l2 = -adv * fminf(fmaxf(ratio, lo), hi);
            const float dratio = (l1 >= l2 || (ratio >= lo && ratio <= hi)) ? -adv : 0.f;
            const float dnlp = -dratio * ratio * a.inv_n;            // d pg / d nlp of this row
            gpi = -dnlp * z * a.inv_sigma;                           // d nlp / d mu = -(a - mu) / sigma^2
            st[0] += (double)fmaxf(l1, l2);
            st[2] += (double)(nlp - cur.nlp) * (double)(nlp - cur.nlp);
            st[3] += fabsf(ratio - 1.f) > a.clip ? 1.0 : 0.0;
            st[4] += (double)(dnlp * fmaf(-z, z, 1.f));              // d nlp / d log_std = 1 - z^2
        }
        backward(0, gpi);
        // ---- value tower
        const float V = forward(1);
        float gv = 0.f;
        if (cur.live) {
            const float d1 = V - cur.ret, dv = V - cur.val;
            const bool clipv = a.clip_vf >= 0.f;
            const float vc = clipv ? cur.val + fminf(fmaxf(dv, -a.clip_vf), a.clip_vf) : V;
            const float d2 = vc - cur.ret;
            const float l1 = d1 * d1, l2 = d2 * d2;
            const float dl = l1 >= l2 ? 2.f * d1 : ((clipv && fabsf(dv) <= a.clip_vf) ? 2.f * d2 : 0.f);
            gv = 0.5f * a.vf_coef * a.inv_n * dl;
            st[1] += (double)fmaxf(l1, l2);
        }
        backward(1, gv);
        fresh = false;
        if (++since == FLUSH || tile + step >= a.tiles) { flush(); since = 0; fresh = true; }
    }
    {   // the group's statistics, fixed order
        double *sd = reinterpret_cast<double *>(S);
        group_bar(g);
        for (int s = 0; s < NSTATS; ++s) sd[s * 128 + gt] = st[s];
        group_bar(g);
        if (gt < NSTATS) {
            double s = 0.0;
            for (int r = 0; r < 128; ++r) s += sd[gt * 128 + r];
            a.ws_stats[(size_t)slot * NSTATS + gt] = s;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS));
}

// The slots of one b2p_ppo_grad* launch -> one fp64 partial vector (b2p_ppo_grad_partial): [0, stride - 1) the gradient
// sums, then the NSTATS statistic sums, each summed in slot order
__global__ void ppo_partial_kernel(const float *__restrict__ ws_grad, const double *__restrict__ ws_stats, int slots, int stride,
                                   double *__restrict__ partial) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < stride - 1) {
        double s = 0.0;
        for (int k = 0; k < slots; ++k) s += (double)ws_grad[(size_t)k * stride + i];
        partial[i] = s;
    } else if (i == stride - 1) {
        double s[ppo::NSTATS] = {0.0, 0.0, 0.0, 0.0, 0.0};
        for (int k = 0; k < slots; ++k)
            for (int q = 0; q < ppo::NSTATS; ++q) s[q] += ws_stats[(size_t)k * ppo::NSTATS + q];
        for (int q = 0; q < ppo::NSTATS; ++q) partial[stride - 1 + q] = s[q];
    }
}

// `ranks` partial vectors (rank order) -> grad_out (the last entry is d loss / d log_std) and the six statistics, summed in
// fp64 from rank 0's vector on (b2p_ppo_combine); one rank is its partial as it is, so b2p_ppo_grad keeps its bits
__global__ void ppo_combine_kernel(const double *__restrict__ partials, int ranks, int stride, double inv_n, double log_std,
                                   double ent_coef, double vf_coef, float *__restrict__ grad, double *__restrict__ stats) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t len = (size_t)stride - 1 + ppo::NSTATS;
    if (i < stride - 1) {
        double s = partials[i];
        for (int r = 1; r < ranks; ++r) s += partials[r * len + i];
        grad[i] = (float)s;
    } else if (i == stride - 1) {
        double s[ppo::NSTATS];
        for (int q = 0; q < ppo::NSTATS; ++q) s[q] = partials[stride - 1 + q];
        for (int r = 1; r < ranks; ++r)
            for (int q = 0; q < ppo::NSTATS; ++q) s[q] += partials[r * len + stride - 1 + q];
        grad[i] = (float)(s[4] - ent_coef);                       // the entropy term: d ent / d log_std = 1
        const double pg = s[0] * inv_n, vf = 0.5 * s[1] * inv_n, ent = log_std + 1.4189385332046727418;   // 0.5 log(2 pi e)
        stats[0] = pg; stats[1] = vf; stats[2] = ent; stats[3] = 0.5 * s[2] * inv_n; stats[4] = s[3] * inv_n;
        stats[5] = pg - ent_coef * ent + vf_coef * vf;
    }
}

}  // namespace pol
}  // namespace

// ---------------------------------------------------------------- host side (C ABI)
struct b2p_policy {
    int device, obs_dim, tanh_mode, num_sms;
    float *weights;                  // w1 [64, obs_dim] | b1 | w2 [64, 64] | b2 | w3 | b3, then the value tower in the same layout
    const unsigned long long *seed_counter;
    unsigned long long row_base;     // global index of row 0 of every launch's rows (b2p_set_row_base)
    bool have_weights, have_value_weights;
    std::string error;
};

namespace {

std::string g_policy_create_error;

int pfail(b2p_handle h, const std::string &msg) {
    if (h) h->error = msg; else g_policy_create_error = msg;
    return 1;
}

// the seed argument of a launch with the handle's global row base folded in (see row_noise)
unsigned long long row_seed(const b2p_policy *h, uint64_t seed) { return (unsigned long long)seed + 0x9E3779B97F4A7C15ull * h->row_base; }

struct PolicyDeviceGuard {
    int prev;
    bool switched;
    explicit PolicyDeviceGuard(int device) : prev(-1), switched(false) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != device) switched = cudaSetDevice(device) == cudaSuccess;
    }
    ~PolicyDeviceGuard() { if (switched) cudaSetDevice(prev); }
};

// f(std::integral_constant<int, K1>()) with the first-layer K of a validated obs_dim (1 .. B2P_MAX_OBS_DIM): the kernels
// are instantiated per K1, and the handle's obs_dim picks them
template <class F>
auto with_k1(int obs_dim, F &&f) {
    switch (pol::obs_width(obs_dim)) {
        case 32: return f(std::integral_constant<int, 32>());
        case 48: return f(std::integral_constant<int, 48>());
        case 64: return f(std::integral_constant<int, 64>());
        case 80: return f(std::integral_constant<int, 80>());
        default: return f(std::integral_constant<int, 16>());
    }
}

template <int FRONT, bool STEP = false, int K1 = 16>
cudaError_t launch_policy(int tanh_mode, int grid, cudaStream_t cs, const pol::Args &a, const Dev &d,
                          const pol::StepArgs &s = pol::StepArgs()) {
    constexpr int smem = pol::Geo<K1, STEP>::SMEM_BYTES, threads = pol::Geo<K1, STEP>::THREADS;
    switch (tanh_mode) {
        case 2: pol::policy_kernel<FRONT, 2, STEP, K1><<<grid, threads, smem, cs>>>(a, d, s); break;
        case 1: pol::policy_kernel<FRONT, 1, STEP, K1><<<grid, threads, smem, cs>>>(a, d, s); break;
        default: pol::policy_kernel<FRONT, 0, STEP, K1><<<grid, threads, smem, cs>>>(a, d, s); break;
    }
    return cudaGetLastError();
}

// the ring front end: FRONT 1 (max_history 5, constant indices) exists only for the narrow row
template <bool STEP, int K1>
cudaError_t launch_ring(int H, int tanh_mode, int grid, cudaStream_t cs, const pol::Args &a, const Dev &d,
                        const pol::StepArgs &s = pol::StepArgs()) {
    if constexpr (K1 == 16) {
        if (H == 5) return launch_policy<1, STEP>(tanh_mode, grid, cs, a, d, s);
    }
    return launch_policy<2, STEP, K1>(tanh_mode, grid, cs, a, d, s);
}

template <int FRONT, bool STEP, int K1 = 16>
bool set_policy_smem() {
    constexpr int smem = pol::Geo<K1, STEP>::SMEM_BYTES;
    return cudaFuncSetAttribute(pol::policy_kernel<FRONT, 0, STEP, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess &&
           cudaFuncSetAttribute(pol::policy_kernel<FRONT, 1, STEP, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess &&
           cudaFuncSetAttribute(pol::policy_kernel<FRONT, 2, STEP, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess;
}

template <int K1>
bool set_smem_all() {
    bool ok = set_policy_smem<0, false, K1>() && set_policy_smem<2, false, K1>() && set_policy_smem<0, true, K1>() &&
              set_policy_smem<2, true, K1>();
    if constexpr (K1 == 16) ok = ok && set_policy_smem<1, false>() && set_policy_smem<1, true>();
    return ok;
}

template <int K1>
bool set_ppo_smem() {
    constexpr int smem = pol::ppo::Geo<K1>::SMEM_BYTES;
    return cudaFuncSetAttribute(pol::ppo_grad_kernel<0, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess &&
           cudaFuncSetAttribute(pol::ppo_grad_kernel<1, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess &&
           cudaFuncSetAttribute(pol::ppo_grad_kernel<2, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess;
}

// grid of a dense front-end launch: one CTA per GROUPS tiles, at most one per SM
int dense_grid(const b2p_policy *h, long long tiles, int groups) {
    const long long want = (tiles + groups - 1) / groups;
    return (int)(want < h->num_sms ? want : h->num_sms);
}

void fill_weights(const b2p_policy *h, pol::Args &a) {
    const int od = h->obs_dim, hid = pol::HID;
    const float *w = h->weights;
    a.w1 = w; a.b1 = a.w1 + hid * od; a.w2 = a.b1 + hid; a.b2 = a.w2 + hid * hid; a.w3 = a.b2 + hid; a.b3 = a.w3 + hid;
    a.obs_dim = od;
}

size_t tower_floats(int obs_dim) {
    return (size_t)pol::HID * obs_dim + pol::HID + pol::HID * pol::HID + pol::HID + pol::HID + 1;
}

int copy_tower(b2p_handle h, float *w, const float *const (&src)[6], cudaStream_t cs, const char *who) {
    const int od = h->obs_dim, hid = pol::HID;
    const size_t cnt[6] = {(size_t)hid * od, (size_t)hid, (size_t)hid * hid, (size_t)hid, (size_t)hid, 1};
    for (int i = 0; i < 6; ++i) {
        if (!src[i]) return pfail(h, std::string(who) + ": null pointer");
        if (cudaMemcpyAsync(w, src[i], cnt[i] * sizeof(float), cudaMemcpyDeviceToDevice, cs) != cudaSuccess)
            return pfail(h, std::string(who) + ": " + cudaGetErrorString(cudaGetLastError()));
        w += cnt[i];
    }
    return 0;
}

// the ring front end's split of the env's tiles over the CTAs (b2p_act_env, b2p_step_env); NULL + error on a bad env
const Dev *ring_setup(b2p_handle h, b2e_handle env, pol::Args &a, int &grid, int groups, const char *who) {
    int ring_ok = 0, device = -1;
    const Dev *dv = static_cast<const Dev *>(b2e_dev_view(env, &ring_ok, &device));
    const std::string w(who);
    if (!dv || !ring_ok) { pfail(h, w + ": the env has no MultiOptLRs adjusted-history rings (large-problem pipeline only)"); return nullptr; }
    if (device != h->device) { pfail(h, w + ": policy and env live on different devices"); return nullptr; }
    if (3 * dv->H != h->obs_dim) { pfail(h, w + ": obs_dim of the policy is not 3 x max_history of the env"); return nullptr; }
    a.rows = (long long)dv->E * dv->P;
    const int tiles_per_env = (dv->P + pol::TILE - 1) / pol::TILE;
    a.tiles = (long long)dv->E * tiles_per_env;
    // few envs: split every env's tiles into segments so that all SMs have work (>= 4 rounds of tiles per group and segment)
    int segs = (3 * h->num_sms + dv->E - 1) / dv->E;
    const int max_segs = tiles_per_env / (4 * groups);
    segs = segs > max_segs ? max_segs : segs;
    a.segs = segs < 1 ? 1 : segs;
    a.units = dv->E * a.segs;
    grid = a.units < h->num_sms ? a.units : h->num_sms;
    return dv;
}

// Args / StepArgs of a b2p_step* launch; non-zero (error set) on a request the handle cannot serve
int step_setup(b2p_handle h, const b2p_step_out *out, float noise_std, float log_std, uint64_t seed, float low, float high,
               pol::Args &a, pol::StepArgs &s, const char *who) {
    const std::string w(who);
    if (!out) return pfail(h, w + ": null output set");
    if (!out->actions && !out->actions_raw && !out->values && !out->neglogp && !out->obs_bf16)
        return pfail(h, w + ": every output is NULL");
    const bool want_pi = out->actions || out->actions_raw || out->neglogp;
    if (want_pi && !h->have_weights) return pfail(h, w + ": b2p_set_weights has not been called");
    if (out->values && !h->have_value_weights) return pfail(h, w + ": values requested but b2p_set_value_weights has not been called");
    if (reinterpret_cast<uintptr_t>(out->obs_bf16) & 15u) return pfail(h, w + ": obs_bf16 must be 16-byte aligned");
    memset(&a, 0, sizeof(a));
    memset(&s, 0, sizeof(s));
    fill_weights(h, a);
    const float *v = h->weights + tower_floats(h->obs_dim);
    const int od = h->obs_dim, hid = pol::HID;
    s.w1 = v; s.b1 = s.w1 + hid * od; s.w2 = s.b1 + hid; s.b2 = s.w2 + hid * hid; s.w3 = s.b2 + hid; s.b3 = s.w3 + hid;
    a.out = out->actions;
    s.raw = out->actions_raw; s.values = out->values; s.neglogp = out->neglogp;
    s.obs16 = static_cast<uint4 *>(out->obs_bf16);
    s.nlp_const = (float)(0.91893853320467274178 + (double)log_std);      // 0.5 log(2 pi) + log_std
    s.want_pi = want_pi ? 1 : 0;
    a.seed_counter = h->seed_counter;
    a.seed = row_seed(h, seed); a.noise_std = noise_std; a.low = low; a.high = high;
    return 0;
}

pol::Feistel feistel_setup(uint64_t key, int64_t n) {
    pol::Feistel f;
    f.n = (unsigned long long)n;
    f.bits = 1;
    while ((1ull << (2 * f.bits)) < f.n) ++f.bits;
    f.mask = (1ull << f.bits) - 1ull;
    for (int r = 0; r < pol::FEISTEL_ROUNDS; ++r) f.key[r] = pol::mix64(key + 0x9E3779B97F4A7C15ull * (unsigned long long)(r + 1));
    return f;
}

int adv_slices(int64_t mb_size) { return (int)((mb_size + pol::ADV_SLICE - 1) / pol::ADV_SLICE); }

size_t grad_stride(int obs_dim) { return 2 * tower_floats(obs_dim) + 1; }

// a b2p_ppo_batch -> PpoBatch; n = T * rows; non-zero (error set on h, or the global error for h = NULL) if malformed
int check_batch(b2p_handle h, const b2p_ppo_batch *b, pol::PpoBatch &pb, int64_t &n, const char *who) {
    const std::string w(who);
    if (!b || !b->obs_bf16 || !b->actions_raw || !b->neglogp || !b->values || !b->returns)
        return pfail(h, w + ": null batch pointer");
    if (reinterpret_cast<uintptr_t>(b->obs_bf16) & 15u) return pfail(h, w + ": obs_bf16 must be 16-byte aligned");
    if (b->T < 1 || b->rows < 1 || b->rows > B2P_PPO_MAX_SAMPLES / b->T) return pfail(h, w + ": bad T or rows");
    n = (int64_t)b->T * b->rows;
    pb.obs = static_cast<const uint4 *>(b->obs_bf16);
    pb.act = b->actions_raw; pb.nlp = b->neglogp; pb.val = b->values; pb.ret = b->returns;
    return 0;
}


}  // namespace

extern "C" {

const char *b2p_last_error(b2p_handle h) { return h ? h->error.c_str() : g_policy_create_error.c_str(); }

int b2p_obs_width(int obs_dim) { return obs_dim >= 1 && obs_dim <= B2P_MAX_OBS_DIM ? pol::obs_width(obs_dim) : 0; }

int b2p_create(int device, int obs_dim, int tanh_mode, b2p_handle *out) {
    if (!out) return pfail(nullptr, "b2p_create: null output pointer");
    *out = nullptr;
    if (obs_dim < 1 || obs_dim > B2P_MAX_OBS_DIM)
        return pfail(nullptr, "b2p_create: obs_dim must be 1..79 (3 x max_history up to max_history 26)");
    if (tanh_mode < 0 || tanh_mode > 2) return pfail(nullptr, "b2p_create: unknown tanh_mode");
    PolicyDeviceGuard guard(device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return pfail(nullptr, "b2p_create: no such CUDA device");
    if (prop.major != 10) return pfail(nullptr, "b2p_create: the policy kernel needs an sm_100 GPU (tcgen05); there is no fallback");
    if (!with_k1(obs_dim, [](auto k) { return set_smem_all<decltype(k)::value>(); }))
        return pfail(nullptr, "b2p_create: the policy kernel does not fit shared memory");
    if (!with_k1(obs_dim, [](auto k) { return set_ppo_smem<decltype(k)::value>(); }))
        return pfail(nullptr, "b2p_create: the PPO gradient kernel does not fit shared memory");
    b2p_policy *h = new (std::nothrow) b2p_policy();
    if (!h) return pfail(nullptr, "b2p_create: out of host memory");
    h->device = device; h->obs_dim = obs_dim; h->tanh_mode = tanh_mode; h->num_sms = prop.multiProcessorCount;
    h->have_weights = h->have_value_weights = false;
    h->seed_counter = nullptr;
    h->row_base = 0;
    if (cudaMalloc((void **)&h->weights, 2 * tower_floats(obs_dim) * sizeof(float)) != cudaSuccess) {
        delete h;
        return pfail(nullptr, "b2p_create: cudaMalloc failed");
    }
    *out = h;
    return 0;
}

int b2p_set_seed_counter(b2p_handle h, const uint64_t *counter) {
    if (!h) return 1;
    h->seed_counter = reinterpret_cast<const unsigned long long *>(counter);
    return 0;
}

int b2p_set_row_base(b2p_handle h, int64_t row_base) {
    if (!h) return 1;
    if (row_base < 0) return pfail(h, "b2p_set_row_base: row_base must be >= 0");
    h->row_base = (unsigned long long)row_base;
    return 0;
}

void b2p_destroy(b2p_handle h) {
    if (!h) return;
    PolicyDeviceGuard guard(h->device);
    cudaFree(h->weights);
    delete h;
}

int b2p_set_weights(b2p_handle h, const float *w1, const float *b1, const float *w2, const float *b2,
                    const float *w3, const float *b3, void *stream) {
    if (!h) return 1;
    if (!w1 || !b1 || !w2 || !b2 || !w3 || !b3) return pfail(h, "b2p_set_weights: null pointer");
    PolicyDeviceGuard guard(h->device);
    const float *const src[6] = {w1, b1, w2, b2, w3, b3};
    if (copy_tower(h, h->weights, src, (cudaStream_t)stream, "b2p_set_weights")) return 1;
    h->have_weights = true;
    return 0;
}

int b2p_set_value_weights(b2p_handle h, const float *w1, const float *b1, const float *w2, const float *b2,
                          const float *w3, const float *b3, void *stream) {
    if (!h) return 1;
    PolicyDeviceGuard guard(h->device);
    const float *const src[6] = {w1, b1, w2, b2, w3, b3};
    if (copy_tower(h, h->weights + tower_floats(h->obs_dim), src, (cudaStream_t)stream, "b2p_set_value_weights")) return 1;
    h->have_value_weights = true;
    return 0;
}

int b2p_act(b2p_handle h, const float *obs, int64_t rows, float *actions_out, float noise_std,
            uint64_t seed, float low, float high, void *stream) {
    if (!h) return 1;
    if (!obs || !actions_out || rows < 0) return pfail(h, "b2p_act: bad argument");
    if (!h->have_weights) return pfail(h, "b2p_act: b2p_set_weights has not been called");
    if (rows == 0) return 0;
    PolicyDeviceGuard guard(h->device);
    pol::Args a;
    memset(&a, 0, sizeof(a));
    fill_weights(h, a);
    a.obs = obs; a.out = actions_out; a.rows = rows; a.tiles = (rows + pol::TILE - 1) / pol::TILE;
    a.seed_counter = h->seed_counter;
    a.seed = row_seed(h, seed); a.noise_std = noise_std; a.low = low; a.high = high;
    a.bulk_ok = (reinterpret_cast<uintptr_t>(obs) & 15u) == 0 ? 1 : 0;
    Dev d;
    memset(&d, 0, sizeof(d));
    const cudaError_t err = with_k1(h->obs_dim, [&](auto k) {
        constexpr int K1 = decltype(k)::value;
        const int grid = dense_grid(h, a.tiles, pol::Geo<K1, false>::GROUPS);
        return launch_policy<0, false, K1>(h->tanh_mode, grid, (cudaStream_t)stream, a, d);
    });
    if (err != cudaSuccess) return pfail(h, std::string("b2p_act: ") + cudaGetErrorString(err));
    return 0;
}

int b2p_act_env(b2p_handle h, b2e_handle env, float *actions_out, float noise_std, uint64_t seed,
                float low, float high, void *stream) {
    if (!h) return 1;
    if (!env || !actions_out) return pfail(h, "b2p_act_env: null pointer");
    if (!h->have_weights) return pfail(h, "b2p_act_env: b2p_set_weights has not been called");
    pol::Args a;
    memset(&a, 0, sizeof(a));
    int grid = 0;
    const int groups = with_k1(h->obs_dim, [](auto k) { return pol::Geo<decltype(k)::value, false>::GROUPS; });
    const Dev *dv = ring_setup(h, env, a, grid, groups, "b2p_act_env");
    if (!dv) return 1;
    PolicyDeviceGuard guard(h->device);
    fill_weights(h, a);
    a.out = actions_out;
    a.seed_counter = h->seed_counter;
    a.seed = row_seed(h, seed); a.noise_std = noise_std; a.low = low; a.high = high;
    const cudaError_t err = with_k1(h->obs_dim, [&](auto k) {
        return launch_ring<false, decltype(k)::value>(dv->H, h->tanh_mode, grid, (cudaStream_t)stream, a, *dv);
    });
    if (err != cudaSuccess) return pfail(h, std::string("b2p_act_env: ") + cudaGetErrorString(err));
    return 0;
}

int b2p_step(b2p_handle h, const float *obs, int64_t rows, const b2p_step_out *out, float noise_std, float log_std,
             uint64_t seed, float low, float high, void *stream) {
    if (!h) return 1;
    if (!obs || rows < 0) return pfail(h, "b2p_step: bad argument");
    pol::Args a;
    pol::StepArgs s;
    if (step_setup(h, out, noise_std, log_std, seed, low, high, a, s, "b2p_step")) return 1;
    if (rows == 0) return 0;
    PolicyDeviceGuard guard(h->device);
    a.obs = obs; a.rows = rows; a.tiles = (rows + pol::TILE - 1) / pol::TILE;
    a.bulk_ok = (reinterpret_cast<uintptr_t>(obs) & 15u) == 0 ? 1 : 0;
    Dev d;
    memset(&d, 0, sizeof(d));
    const cudaError_t err = with_k1(h->obs_dim, [&](auto k) {
        constexpr int K1 = decltype(k)::value;
        const int grid = dense_grid(h, a.tiles, pol::Geo<K1, true>::GROUPS);
        return launch_policy<0, true, K1>(h->tanh_mode, grid, (cudaStream_t)stream, a, d, s);
    });
    if (err != cudaSuccess) return pfail(h, std::string("b2p_step: ") + cudaGetErrorString(err));
    return 0;
}

int b2p_step_env(b2p_handle h, b2e_handle env, const b2p_step_out *out, float noise_std, float log_std, uint64_t seed,
                 float low, float high, void *stream) {
    if (!h) return 1;
    if (!env) return pfail(h, "b2p_step_env: null pointer");
    pol::Args a;
    pol::StepArgs s;
    if (step_setup(h, out, noise_std, log_std, seed, low, high, a, s, "b2p_step_env")) return 1;
    int grid = 0;
    const int groups = with_k1(h->obs_dim, [](auto k) { return pol::Geo<decltype(k)::value, true>::GROUPS; });
    const Dev *dv = ring_setup(h, env, a, grid, groups, "b2p_step_env");
    if (!dv) return 1;
    PolicyDeviceGuard guard(h->device);
    const cudaError_t err = with_k1(h->obs_dim, [&](auto k) {
        return launch_ring<true, decltype(k)::value>(dv->H, h->tanh_mode, grid, (cudaStream_t)stream, a, *dv, s);
    });
    if (err != cudaSuccess) return pfail(h, std::string("b2p_step_env: ") + cudaGetErrorString(err));
    return 0;
}

int b2p_gae(const float *values, const float *rewards, const uint8_t *dones, int T, int64_t rows, int64_t P, double gamma,
            double lam, float *adv_out, float *ret_out, void *stream) {
    if (!values || !rewards || !dones || !adv_out || !ret_out || T < 0 || rows < 0 || P < 1)
        return pfail(nullptr, "b2p_gae: bad argument");
    if (rows % P) return pfail(nullptr, "b2p_gae: rows is not a multiple of P (rows per env)");
    if (T == 0 || rows == 0) return 0;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, values) != cudaSuccess || attr.type != cudaMemoryTypeDevice)
        return pfail(nullptr, "b2p_gae: values is not device memory");
    PolicyDeviceGuard guard(attr.device);
    const long long blocks = (rows + pol::GAE_THREADS - 1) / pol::GAE_THREADS;
    pol::gae_kernel<<<(unsigned)blocks, pol::GAE_THREADS, 0, (cudaStream_t)stream>>>(values, rewards, dones, T, rows, P, gamma, lam,
                                                                                   adv_out, ret_out);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return pfail(nullptr, std::string("b2p_gae: ") + cudaGetErrorString(err));
    return 0;
}

int b2p_tanh_table(float *out, void *stream) {
    if (!out) return pfail(nullptr, "b2p_tanh_table: null output");
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, out) != cudaSuccess || attr.type != cudaMemoryTypeDevice)
        return pfail(nullptr, "b2p_tanh_table: out is not device memory");
    PolicyDeviceGuard guard(attr.device);
    pol::tanh_bf16_table_kernel<<<256, 256, 0, (cudaStream_t)stream>>>(out);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return pfail(nullptr, std::string("b2p_tanh_table: ") + cudaGetErrorString(err));
    return 0;
}

int b2p_ppo_indices(uint64_t key, int64_t n, int64_t begin, int64_t count, int64_t *out, void *stream) {
    if (n < 1 || n > B2P_PPO_MAX_SAMPLES) return pfail(nullptr, "b2p_ppo_indices: n must be 1..2^62");
    if (count < 1) return pfail(nullptr, "b2p_ppo_indices: count must be >= 1");
    if (begin < 0 || begin > n - count) return pfail(nullptr, "b2p_ppo_indices: range outside [0, n)");
    if (!out) return pfail(nullptr, "b2p_ppo_indices: null output");
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, out) != cudaSuccess || attr.type != cudaMemoryTypeDevice)
        return pfail(nullptr, "b2p_ppo_indices: out is not device memory");
    PolicyDeviceGuard guard(attr.device);
    const pol::Feistel f = feistel_setup(key, n);
    const long long blocks = std::min<long long>((count + 255) / 256, 1 << 16);
    pol::ppo_indices_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(f, begin, count, reinterpret_cast<long long *>(out));
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return pfail(nullptr, std::string("b2p_ppo_indices: ") + cudaGetErrorString(err));
    return 0;
}

size_t b2p_ppo_adv_stats_workspace_size(int64_t n, int64_t mb_size) {
    if (n < 1 || mb_size < 1 || n % mb_size) return 0;
    const size_t nmb = (size_t)(n / mb_size);
    return nmb * (size_t)adv_slices(mb_size) * 2 * sizeof(double) + nmb * 4 * sizeof(double);
}

}  // extern "C"

namespace {

// the slice sums of every minibatch of an epoch -> moments [nmb][4] (b2p_ppo_adv_moments, b2p_ppo_adv_stats); `part` holds
// the slice sums, nmb * slices * 2 doubles
int adv_moments(const b2p_ppo_batch *b, uint64_t key, int64_t mb_size, double *moments, double *part, void *stream,
                int &device, const char *who) {
    pol::PpoBatch pb;
    int64_t n = 0;
    const std::string w(who);
    if (check_batch(nullptr, b, pb, n, who)) return 1;
    if (!moments || !part) return pfail(nullptr, w + ": null output or workspace");
    if (mb_size < 1 || n % mb_size) return pfail(nullptr, w + ": T * rows is not a multiple of the minibatch size");
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, b->returns) != cudaSuccess || attr.type != cudaMemoryTypeDevice)
        return pfail(nullptr, w + ": returns is not device memory");
    device = attr.device;
    PolicyDeviceGuard guard(attr.device);
    const pol::Feistel f = feistel_setup(key, n);
    const long long nmb = n / mb_size;
    const int slices = adv_slices(mb_size);
    if (nmb > 0x7FFFFFFFLL / slices)
        return pfail(nullptr, w + ": too many minibatches for one launch (more than 2^31 - 1 blocks)");
    pol::ppo_adv_partial<<<(unsigned)(nmb * slices), pol::ADV_THREADS, 0, (cudaStream_t)stream>>>(pb, f, mb_size, slices, part);
    pol::ppo_adv_moments_kernel<<<(unsigned)((nmb + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pb, f, mb_size, nmb, slices, part,
                                                                                                 moments);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return pfail(nullptr, w + ": " + cudaGetErrorString(err));
    return 0;
}

int adv_combine(const double *moments, int ranks, int64_t nmb, double *stats_out, void *stream, const char *who) {
    pol::ppo_adv_combine_kernel<<<(unsigned)((nmb + 255) / 256), 256, 0, (cudaStream_t)stream>>>(moments, ranks, nmb, stats_out);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return pfail(nullptr, std::string(who) + ": " + cudaGetErrorString(err));
    return 0;
}

// doubles of one partial vector: the gradient sums before log_std's, then the NSTATS statistic sums
size_t partial_doubles(int obs_dim) { return grad_stride(obs_dim) - 1 + pol::ppo::NSTATS; }

// The gradient workspace (b2p_ppo_workspace_size bytes): from its first 256-byte boundary the fp32 gradient slots
// [slots][stride], from the next 8-byte boundary the fp64 statistic slots [slots][NSTATS], then b2p_ppo_grad's own
// partial vector.  `slots` is that of the largest grid (num_sms x groups), so the layout does not depend on the launch.
struct PpoWorkspace {
    float *grad;
    double *stats, *partial;
};
size_t max_slots(const b2p_policy *h) { return (size_t)h->num_sms * pol::ppo::groups(pol::obs_width(h->obs_dim)); }
size_t ppo_workspace_bytes(const b2p_policy *h) {
    return max_slots(h) * (grad_stride(h->obs_dim) * sizeof(float) + pol::ppo::NSTATS * sizeof(double)) +
           partial_doubles(h->obs_dim) * sizeof(double) + 255 + 7;      // + the two alignments
}
PpoWorkspace ppo_workspace(const b2p_policy *h, void *workspace) {
    const size_t slots = max_slots(h);
    const uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
    PpoWorkspace w;
    w.grad = reinterpret_cast<float *>(base);
    w.stats = reinterpret_cast<double *>(base + ((slots * grad_stride(h->obs_dim) * sizeof(float) + 7) & ~(size_t)7));
    w.partial = w.stats + slots * pol::ppo::NSTATS;
    return w;
}

// the gradient kernel over one shard's minibatch and its slot reduction into `partial` (b2p_ppo_grad, b2p_ppo_grad_partial):
// the per-row scale is 1 / count_total, the size of the union minibatch
int grad_partial(b2p_handle h, const b2p_ppo_batch *b, const b2p_ppo_params *p, int64_t count_total, double *partial,
                 void *workspace, cudaStream_t cs, const char *who) {
    const std::string w(who);
    if (!h->have_weights || !h->have_value_weights)
        return pfail(h, w + ": weights not set (b2p_set_weights and b2p_set_value_weights)");
    pol::PpoBatch pb;
    int64_t n = 0;
    if (check_batch(h, b, pb, n, who)) return 1;
    if (!p || !partial || !workspace || !p->adv_stats) return pfail(h, w + ": null params, adv_stats, output or workspace");
    if (p->count < 1) return pfail(h, w + ": count must be >= 1");
    if (p->begin < 0 || p->begin > n - p->count) return pfail(h, w + ": range outside [0, T * rows)");
    if (count_total < p->count || count_total > B2P_PPO_MAX_SAMPLES)
        return pfail(h, w + ": count_total must be count..2^62 (the size of the union minibatch)");
    if (!(p->cliprange > 0.f)) return pfail(h, w + ": cliprange must be > 0");
    PolicyDeviceGuard guard(h->device);
    pol::GradArgs a;
    memset(&a, 0, sizeof(a));
    a.w = h->weights;
    a.b = pb;
    a.f = feistel_setup(p->key, n);
    a.begin = p->begin; a.count = p->count; a.tiles = (p->count + pol::TILE - 1) / pol::TILE;
    a.adv_stats = p->adv_stats;
    a.clip = p->cliprange; a.clip_vf = p->cliprange_vf; a.vf_coef = p->vf_coef;
    a.inv_n = (float)(1.0 / (double)count_total);
    a.inv_sigma = (float)exp(-(double)p->log_std);
    a.nlp_const = (float)(0.91893853320467274178 + (double)p->log_std);      // as b2p_step: 0.5 log(2 pi) + log_std
    a.od = h->obs_dim; a.tf = (int)tower_floats(h->obs_dim); a.stride = (int)grad_stride(h->obs_dim);
    const int groups = pol::ppo::groups(pol::obs_width(h->obs_dim));
    const int grid = dense_grid(h, a.tiles, groups), slots = grid * groups;
    const PpoWorkspace ws = ppo_workspace(h, workspace);
    a.ws_grad = ws.grad;
    a.ws_stats = ws.stats;
    with_k1(h->obs_dim, [&](auto k) {
        using PG = pol::ppo::Geo<decltype(k)::value>;
        switch (h->tanh_mode) {
            case 2: pol::ppo_grad_kernel<2, decltype(k)::value><<<grid, PG::THREADS, PG::SMEM_BYTES, cs>>>(a); break;
            case 1: pol::ppo_grad_kernel<1, decltype(k)::value><<<grid, PG::THREADS, PG::SMEM_BYTES, cs>>>(a); break;
            default: pol::ppo_grad_kernel<0, decltype(k)::value><<<grid, PG::THREADS, PG::SMEM_BYTES, cs>>>(a); break;
        }
        return 0;
    });
    pol::ppo_partial_kernel<<<(a.stride + 255) / 256, 256, 0, cs>>>(a.ws_grad, a.ws_stats, slots, a.stride, partial);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return pfail(h, w + ": " + cudaGetErrorString(err));
    return 0;
}

int combine(b2p_handle h, const double *partials, int ranks, int64_t count_total, float log_std, float ent_coef, float vf_coef,
            float *grad_out, double *stats_out, cudaStream_t cs, const char *who) {
    PolicyDeviceGuard guard(h->device);
    const int stride = (int)grad_stride(h->obs_dim);
    pol::ppo_combine_kernel<<<(stride + 255) / 256, 256, 0, cs>>>(partials, ranks, stride, 1.0 / (double)count_total,
                                                                  (double)log_std, (double)ent_coef, (double)vf_coef, grad_out,
                                                                  stats_out);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return pfail(h, std::string(who) + ": " + cudaGetErrorString(err));
    return 0;
}

}  // namespace

extern "C" {

int b2p_ppo_adv_moments(const b2p_ppo_batch *b, uint64_t key, int64_t mb_size, double *moments_out, void *workspace,
                        void *stream) {
    int device = -1;
    return adv_moments(b, key, mb_size, moments_out, static_cast<double *>(workspace), stream, device, "b2p_ppo_adv_moments");
}

int b2p_ppo_adv_combine(const double *moments, int ranks, int64_t nmb, double *stats_out, void *stream) {
    if (!moments || !stats_out) return pfail(nullptr, "b2p_ppo_adv_combine: null moments or output");
    if (ranks < 1) return pfail(nullptr, "b2p_ppo_adv_combine: ranks must be >= 1");
    if (nmb < 1 || nmb > 0x7FFFFFFFLL * 256) return pfail(nullptr, "b2p_ppo_adv_combine: nmb must be 1..(2^31 - 1) x 256");
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, moments) != cudaSuccess || attr.type != cudaMemoryTypeDevice)
        return pfail(nullptr, "b2p_ppo_adv_combine: moments is not device memory");
    PolicyDeviceGuard guard(attr.device);
    return adv_combine(moments, ranks, nmb, stats_out, stream, "b2p_ppo_adv_combine");
}

int b2p_ppo_adv_stats(const b2p_ppo_batch *b, uint64_t key, int64_t mb_size, double *stats_out, void *workspace,
                      void *stream) {
    pol::PpoBatch pb;
    int64_t n = 0;
    if (check_batch(nullptr, b, pb, n, "b2p_ppo_adv_stats")) return 1;
    if (!stats_out || !workspace) return pfail(nullptr, "b2p_ppo_adv_stats: null output or workspace");
    if (mb_size < 1 || n % mb_size) return pfail(nullptr, "b2p_ppo_adv_stats: T * rows is not a multiple of the minibatch size");
    const int64_t nmb = n / mb_size;
    double *part = static_cast<double *>(workspace), *moments = part + nmb * adv_slices(mb_size) * 2;   // the slice sums, then the moments
    int device = -1;
    if (adv_moments(b, key, mb_size, moments, part, stream, device, "b2p_ppo_adv_stats")) return 1;
    PolicyDeviceGuard guard(device);
    return adv_combine(moments, 1, nmb, stats_out, stream, "b2p_ppo_adv_stats");
}

size_t b2p_ppo_workspace_size(b2p_handle h) {
    if (!h) return 0;
    return ppo_workspace_bytes(h);
}

size_t b2p_ppo_partial_size(b2p_handle h) { return h ? partial_doubles(h->obs_dim) : 0; }

int b2p_ppo_grad_partial(b2p_handle h, const b2p_ppo_batch *b, const b2p_ppo_params *p, int64_t count_total,
                         double *partial_out, void *workspace, void *stream) {
    if (!h) return 1;
    return grad_partial(h, b, p, count_total, partial_out, workspace, (cudaStream_t)stream, "b2p_ppo_grad_partial");
}

int b2p_ppo_combine(b2p_handle h, const double *partials, int ranks, int64_t count_total, float log_std, float ent_coef,
                    float vf_coef, float *grad_out, double *stats_out, void *stream) {
    if (!h) return 1;
    if (!partials || !grad_out || !stats_out) return pfail(h, "b2p_ppo_combine: null partials or output");
    if (ranks < 1) return pfail(h, "b2p_ppo_combine: ranks must be >= 1");
    if (count_total < 1 || count_total > B2P_PPO_MAX_SAMPLES) return pfail(h, "b2p_ppo_combine: count_total must be 1..2^62");
    return combine(h, partials, ranks, count_total, log_std, ent_coef, vf_coef, grad_out, stats_out, (cudaStream_t)stream,
                   "b2p_ppo_combine");
}

int b2p_ppo_grad(b2p_handle h, const b2p_ppo_batch *b, const b2p_ppo_params *p, float *grad_out, double *stats_out,
                 void *workspace, void *stream) {
    if (!h) return 1;
    // its own partial vector lives in the workspace (a NULL output makes grad_partial report the nulls)
    double *partial = workspace && grad_out && stats_out ? ppo_workspace(h, workspace).partial : nullptr;
    const cudaStream_t cs = (cudaStream_t)stream;
    if (grad_partial(h, b, p, p ? p->count : 0, partial, workspace, cs, "b2p_ppo_grad")) return 1;
    return combine(h, partial, 1, p->count, p->log_std, p->ent_coef, p->vf_coef, grad_out, stats_out, cs, "b2p_ppo_grad");
}

}  // extern "C"
