/* b200policy.h -- C ABI of the shared per-agent policy of libb200env.so (SURVEY 8f.2).
 *
 * The reference's callers evaluate ONE policy network on every agent row of the VecEnv: the
 * stable-baselines runner behind `PPO2/A2C(MlpPolicy, vec_env).learn()` and `.predict(obs)`
 * (run_multiagent_exp_single.py:37-49, play_optimize.py:79-98) calls `model.step(obs)` with the
 * [sum(P), 3H] observation matrix that OptVecEnv.step_wait returned (vectorize/optvecenv.py:78-88).
 * MlpPolicy is two tanh layers of 64 units and a linear head.  At BASELINE config 4 that matrix has
 * 2.08e8 rows; pulling it to the host costs 12.5 GB per step.  These entry points evaluate the
 * action head on the device instead:
 *
 *   action[row] = clip(mean(obs[row]) + noise_std * N(0, 1), low, high)
 *   mean(x)     = w3 . tanh(W2 tanh(W1 x + b1) + b2) + b3
 *
 * with bf16 operands and fp32 accumulation on the tcgen05 tensor cores (a policy is the caller's
 * model, not part of the reference's arithmetic: the parity bar of the env step does not apply;
 * tests/test_gpu_policy.py holds it to a bf16-rounded torch evaluation of the same network).
 *
 * b2p_act reads a dense observation matrix (what b2e_step wrote).  b2p_act_env reads the env's
 * adjusted-history rings directly -- the observation row of agent p of env e is
 * clip(nan_to_num([adj_w[e][newest..oldest][p] | adj_L[e][..] | adj_g[e][..][p]]), +-100) - 1
 * (envs/multioptlrs.py:96-101) -- so that b2e_step may be called with obs_out = NULL and the
 * 3H observation words per agent are never written to or read from HBM.
 *
 * Pointers are DEVICE pointers; `stream` is a cudaStream_t passed as void*; calls are asynchronous
 * on it.  Return 0 on success, non-zero with b2p_last_error() otherwise.
 */
#ifndef B200POLICY_H
#define B200POLICY_H

#include <stddef.h>
#include <stdint.h>

#include "b200env.h"

#ifdef __cplusplus
extern "C" {
#endif

#define B2P_HIDDEN 64            /* units of both hidden layers (stable-baselines MlpPolicy) */
#define B2P_MAX_OBS_DIM 79       /* 3H with H <= 26 (MultiOptLRs; the reference's max_history search space is 5..25) */

/* tanh_mode */
#define B2P_TANH_F32    0        /* tanh.approx.f32 on the fp32 accumulators (default)                      */
#define B2P_TANH_BF16X2 1        /* first layer: tanh.approx.bf16x2 on the packed operand of the second MMA */

typedef struct b2p_policy *b2p_handle;

/* obs_dim 1..B2P_MAX_OBS_DIM; anything else is rejected. */
int b2p_create(int device, int obs_dim, int tanh_mode, b2p_handle *out);

/* W, the bf16 columns of a stored observation row (b2p_step_out.obs_bf16, b2p_ppo_batch.obs_bf16) for obs_dim:
 * 16 * ceil((obs_dim + 1) / 16), i.e. 16 for obs_dim 1..15, 32 for 16..31, 48 for 32..47, 64 for 48..63 and 80 for
 * 64..79.  Columns obs_dim..W-1 are stored as zero; column W-1 is the bias slot the kernels set to 1 when they read
 * the row.  0 outside 1..B2P_MAX_OBS_DIM.  Needs no device. */
int b2p_obs_width(int obs_dim);
void b2p_destroy(b2p_handle h);
const char *b2p_last_error(b2p_handle h);

/* torch.nn.Linear layouts: w1 [64, obs_dim], b1 [64], w2 [64, 64], b2 [64], w3 [64], b3 [1]; float32.
 * The handle keeps its own copy. */
int b2p_set_weights(b2p_handle h, const float *w1, const float *b1, const float *w2,
                    const float *b2, const float *w3, const float *b3, void *stream);

/* Optional: a device counter added to `seed` by every later b2p_act / b2p_act_env launch (NULL = none).  The caller
 * advances it on the stream between launches; a CUDA graph that captured the launches then draws fresh noise on
 * every replay although the seed argument is baked into the graph. */
int b2p_set_seed_counter(b2p_handle h, const uint64_t *counter);

/* obs float32 [rows, obs_dim] dense -> actions_out float32 [rows].  noise_std = exp(log_std) of the
 * diagonal Gaussian (0 = deterministic, `model.predict(deterministic=True)`); the noise of a row is a
 * counter-based hash of (seed, row). */
int b2p_act(b2p_handle h, const float *obs, int64_t rows, float *actions_out, float noise_std,
            uint64_t seed, float low, float high, void *stream);

/* The same for every agent row of `env` (MultiOptLRs layout, large-problem pipeline), read from the env's
 * rings; actions_out float32 [E*P] in VecEnv row order, ready for the next b2e_step. */
int b2p_act_env(b2p_handle h, b2e_handle env, float *actions_out, float noise_std, uint64_t seed,
                float low, float high, void *stream);

/* out float32 [65536]: out[x] = the bf16 tanh of the bf16 with bit pattern x, as the kernels evaluate it in
 * B2P_TANH_BF16X2 and the mode that also uses it for the second layer (tanh.approx.bf16x2).  For references that
 * reproduce those modes exactly.  Errors: b2p_last_error(NULL). */
int b2p_tanh_table(float *out, void *stream);

/* ---- PPO rollouts: the rest of stable-baselines' model.step / model.value, and GAE.
 *
 * MlpPolicy has a second tower of the same shape for the value (net_arch pi = vf = [64, 64]); it is
 * set in the torch.nn.Linear layouts of b2p_set_weights.  The handle keeps its own copy. */
int b2p_set_value_weights(b2p_handle h, const float *w1, const float *b1, const float *w2,
                          const float *b2, const float *w3, const float *b3, void *stream);

/* Outputs of one step launch, each [rows] float32 in the row order of the front end (VecEnv order on
 * the rings), any of them NULL = not computed:
 *   actions      clip(raw, low, high): bit for bit what b2p_act / b2p_act_env write with the same
 *                seed, noise and bounds (the env steps with these)
 *   actions_raw  raw = mean + noise_std * z, z = the row's N(0, 1) draw (PPO stores and scores this)
 *   values       the value tower's output (model.value)
 *   neglogp      0.5 z^2 + 0.5 log(2 pi) + log_std: -log density of raw under the diagonal Gaussian
 *   obs_bf16     [rows][W] bf16, W = b2p_obs_width(obs_dim), 16-byte aligned: the observation row the first
 *                layer read, already rounded to bf16, columns obs_dim..W-1 zero (2W bytes per row)
 * The action tower runs only for actions / actions_raw / neglogp, the value tower only for values
 * (values alone = model.value).  values needs b2p_set_value_weights; an all-NULL set is an error. */
typedef struct b2p_step_out {
    float *actions;
    float *actions_raw;
    float *values;
    float *neglogp;
    void *obs_bf16;
} b2p_step_out;

/* Dense front end: obs float32 [rows, obs_dim], as b2p_act.  `out` is read when the call is made. */
int b2p_step(b2p_handle h, const float *obs, int64_t rows, const b2p_step_out *out, float noise_std,
             float log_std, uint64_t seed, float low, float high, void *stream);

/* Ring front end: every agent row of `env`, as b2p_act_env. */
int b2p_step_env(b2p_handle h, b2e_handle env, const b2p_step_out *out, float noise_std, float log_std,
                 uint64_t seed, float low, float high, void *stream);

/* Generalised advantage estimation of the PPO2 Runner over a time-major rollout of T steps:
 *   values float32 [T+1, rows] (values[T] = the value of the observation after the last step),
 *   rewards float32 [T, E], dones uint8 [T+1, E] (dones[t+1] = done returned by step t; dones[0] is
 *   not read), E = rows / P with P rows per env (env = row / P in both VecEnv row orders)
 *   -> adv_out, ret_out float32 [T, rows]:
 *   nn = 1 - dones[t+1], delta = r[t] + gamma values[t+1] nn - values[t],
 *   adv[t] = last = delta + gamma lam nn last, ret[t] = adv[t] + values[t]
 * with the Runner's precision (float64 recursion, float32 stores).  Runs on the device of `values`;
 * errors are read with b2p_last_error(NULL). */
int b2p_gae(const float *values, const float *rewards, const uint8_t *dones, int T, int64_t rows,
            int64_t P, double gamma, double lam, float *adv_out, float *ret_out, void *stream);

/* ---- PPO updates: the gradient of stable-baselines 2's PPO2 loss over one minibatch of a rollout.
 *
 * A minibatch is a range of positions of a keyed permutation of the T * rows flat sample indices
 * j = t * rows + row (a Feistel bijection, cycle-walked into [0, T * rows); no index array is stored):
 * epoch e of PPO2 uses one key and minibatch m the positions [m * n, (m + 1) * n). */
#define B2P_PPO_MAX_SAMPLES (1LL << 62)

typedef struct b2p_ppo_batch {          /* a DeviceRolloutBuffer, time-major */
    const void *obs_bf16;               /* [T][rows][W] bf16, W = b2p_obs_width(obs_dim), 16-byte aligned (column W-1
                                           is not read: the bias 1) */
    const float *actions_raw, *neglogp, *values, *returns;   /* [T][rows] (values: first T rows of [T+1][rows]) */
    int T;
    int64_t rows;
} b2p_ppo_batch;

typedef struct b2p_ppo_params {
    float cliprange, cliprange_vf;      /* cliprange_vf < 0: no value clipping (the None default is resolved by the caller) */
    float ent_coef, vf_coef, log_std;
    uint64_t key;                       /* permutation key of the epoch */
    int64_t begin, count;               /* the minibatch = positions [begin, begin + count) of the permutation */
    const double *adv_stats;            /* device [2]: mean and population std of this minibatch's returns - values */
} b2p_ppo_params;

/* out int64 [count] = the flat sample indices at positions [begin, begin + count) of the permutation of [0, n)
 * with `key`.  Errors: b2p_last_error(NULL). */
int b2p_ppo_indices(uint64_t key, int64_t n, int64_t begin, int64_t count, int64_t *out, void *stream);

/* Advantage statistics of every minibatch of an epoch: stats_out double [T * rows / mb_size][2] = mean and population
 * std of A = returns - values (float32 difference, fp64 sums in a fixed order) over each minibatch's samples.
 * T * rows must be a multiple of mb_size.  workspace: b2p_ppo_adv_stats_workspace_size(T * rows, mb_size) bytes.
 * Errors: b2p_last_error(NULL). */
size_t b2p_ppo_adv_stats_workspace_size(int64_t n, int64_t mb_size);
int b2p_ppo_adv_stats(const b2p_ppo_batch *b, uint64_t key, int64_t mb_size, double *stats_out, void *workspace,
                      void *stream);

/* The gradient of PPO2's loss over one minibatch, with the weights of the last b2p_set_weights /
 * b2p_set_value_weights and the handle's tanh_mode:
 *   A_n = (A - mean) / (std + 1e-8);  ratio = exp(neglogp_old - neglogp(actions_raw | mu, log_std))
 *   pg = mean(max(-A_n ratio, -A_n clip(ratio, 1 - c, 1 + c)))
 *   vf = 0.5 mean(max((V - R)^2, (V_old + clip(V - V_old, -c_vf, c_vf) - R)^2))   (c_vf < 0: vf = 0.5 mean((V - R)^2))
 *   ent = log_std + 0.5 log(2 pi e);  loss = pg - ent_coef ent + vf_coef vf
 * grad_out float [2 * tower + 1]: d loss / d (action tower, value tower, log_std), the towers in b2p_set_weights layouts
 * (w1, b1, w2, b2, w3, b3); stats_out double [6]: pg, vf, ent, approxkl = 0.5 mean((nlp - nlp_old)^2),
 * clipfrac = mean(|ratio - 1| > c), loss.  Gradients follow TensorFlow's rules (max: the first operand on ties; clip:
 * passes inside the closed interval).  workspace: b2p_ppo_workspace_size(h) bytes.  The result is bit-identical from
 * call to call for the same inputs on the same device.  Nothing is allocated. */
size_t b2p_ppo_workspace_size(b2p_handle h);
int b2p_ppo_grad(b2p_handle h, const b2p_ppo_batch *b, const b2p_ppo_params *p, float *grad_out, double *stats_out,
                 void *workspace, void *stream);

/* ---- Data-parallel PPO: one policy trained on the rollouts of R env shards (one per GPU).
 *
 * Shard r rolls out envs [first_env, first_env + E_r) of the whole batch: b2e_config.env_base = first_env, and
 * b2p_set_row_base(first_env * P) on the policy, so that its trajectories are those envs' rows of one unsharded run bit
 * for bit.  Minibatch m of an epoch is the union over shards of positions [m N_r / n_mb, (m + 1) N_r / n_mb) of each
 * shard's own permutation of its N_r = T * rows_r samples (every N_r a multiple of n_mb); its size is
 * n_m = sum_r N_r / n_mb.  The advantages are normalised with the union's mean and std and the loss is a mean over n_m:
 *   b2p_ppo_adv_moments on every shard, the R moment sets gathered in rank order, b2p_ppo_adv_combine;
 *   per minibatch b2p_ppo_grad_partial on every shard, the R partial vectors gathered in rank order, b2p_ppo_combine.
 * The combines sum in fp64 from rank 0 on, so every rank that combines the same inputs gets the same bits.
 * b2p_ppo_adv_stats and b2p_ppo_grad are these with R = 1.  Nothing here allocates; transport is the caller's. */

/* Global index of row 0 of every later b2p_act* / b2p_step* launch (default 0; >= 0): local row r draws the noise of
 * row row_base + r, and everything that depends on it (actions, actions_raw, neglogp) follows. */
int b2p_set_row_base(b2p_handle h, int64_t row_base);

/* Doubles of one partial vector: the 2 * tower gradient sums before log_std's, then the five loss sums
 * (2 * tower + 5; 0 for NULL). */
size_t b2p_ppo_partial_size(b2p_handle h);

/* This shard's part of the gradient over its rows [p->begin, p->begin + p->count) of the minibatch (permutation p->key):
 * b2p_ppo_grad's kernel with every row scaled by 1 / count_total (count_total = n_m >= p->count), p->adv_stats the
 * union's (mean, std) from b2p_ppo_adv_combine.  partial_out: double [b2p_ppo_partial_size(h)]; workspace:
 * b2p_ppo_workspace_size(h) bytes.  p->ent_coef is not read (b2p_ppo_combine applies it). */
int b2p_ppo_grad_partial(b2p_handle h, const b2p_ppo_batch *b, const b2p_ppo_params *p, int64_t count_total,
                         double *partial_out, void *workspace, void *stream);

/* partials double [ranks][b2p_ppo_partial_size(h)] (rank order, ranks >= 1) -> grad_out and stats_out as b2p_ppo_grad
 * writes them, for the union minibatch of count_total rows. */
int b2p_ppo_combine(b2p_handle h, const double *partials, int ranks, int64_t count_total, float log_std, float ent_coef,
                    float vf_coef, float *grad_out, double *stats_out, void *stream);

/* moments_out double [T * rows / mb_size][4] = count, shift K (A at the minibatch's first position), sum(A - K),
 * sum((A - K)^2) of every minibatch of the permutation `key` of this shard's samples, summed as b2p_ppo_adv_stats does.
 * workspace: b2p_ppo_adv_stats_workspace_size(T * rows, mb_size) bytes.  Errors: b2p_last_error(NULL). */
int b2p_ppo_adv_moments(const b2p_ppo_batch *b, uint64_t key, int64_t mb_size, double *moments_out, void *workspace,
                        void *stream);

/* moments double [ranks][nmb][4] (rank order, ranks >= 1) -> stats_out double [nmb][2]: mean and population std of every
 * union minibatch's advantages.  Shard r's sums are moved to rank 0's shift before they are added.
 * Errors: b2p_last_error(NULL). */
int b2p_ppo_adv_combine(const double *moments, int ranks, int64_t nmb, double *stats_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200POLICY_H */
