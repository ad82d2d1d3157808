/* b200env.h -- C ABI of libb200env.so: the batched step of custom_envs' optimisation
 * environments on one B200 (sm_100a).
 *
 * The reference (adolfogonzalez3/custom_envs) is pure Python and has no FFI on this path;
 * each entry point below replaces the Python call chain named beside it (paths relative
 * to the reference tree).  Every pointer is a plain DEVICE pointer unless the name ends
 * in _host; buffers are borrowed for the duration of the call; all work is enqueued on
 * the caller's stream (a cudaStream_t passed as void*), with no hidden synchronisation,
 * so a step is CUDA-graph capturable.  Return value: 0 on success, non-zero on error
 * with the text available from b2e_last_error().  No exceptions or aborts cross the ABI.
 * One handle is bound to one device and must be used from one host thread at a time.
 */
#ifndef B200ENV_H
#define B200ENV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2E_ABI_VERSION 2

/* env_kind */
#define B2E_ENV_MULTIOPTLRS   0   /* envs/multioptlrs.py:39-129   */
#define B2E_ENV_MULTIOPTIMIZE 1   /* envs/multioptimize.py:40-154 */
/* problem_kind */
#define B2E_PROBLEM_SOFTMAX 0     /* problems/optimize_nn.py:35-52: Dense[+relu Dense] + softmax CE */
#define B2E_PROBLEM_LINREG  1     /* XW+b with utils/utils_math.py:37-48 per-sample loss             */
#define B2E_PROBLEM_FUNC    2     /* problems/optimize_function.py:35-50: Rosenbrock, P = 2          */
/* row_order: which parameter a VecEnv row shows */
#define B2E_ROWS_LEXICOGRAPHIC 0  /* gym Dict key order, vectorize/optvecenv.py:10-14 (reference)    */
#define B2E_ROWS_NATURAL       1  /* row j = parameter j                                             */
/* index_mode */
#define B2E_INDEX_INTERNAL 0      /* device keeps each env's InMemoryDataSet order + cursor          */
#define B2E_INDEX_EXTERNAL 1      /* caller passes [E,B] row indices + [E] counts to every call      */

#define B2E_INFO_STRIDE 16        /* doubles per env in info_out, see b2e_step                       */
#define B2E_MAX_HISTORY 32
#define B2E_MAX_LAYERS 8          /* Dense layers of the classifier, output layer included           */

/* b2e_get_state / b2e_set_state selectors (per-env stride in elements in brackets) */
#define B2E_STATE_PARAMS      0   /* float  [P]   current parameters, natural (flatten_arrays) order */
#define B2E_STATE_GRAD_PREV   1   /* float  [P]   newest raw-history gradient                         */
#define B2E_STATE_ADJ_WEIGHTS 2   /* float  [H,P] adjusted weights history, NEWEST FIRST (H = b2e_history_depth) */
#define B2E_STATE_ADJ_GRADS   3   /* float  [H,P] adjusted gradients history, NEWEST FIRST            */
#define B2E_STATE_ADJ_LOSSES  4   /* float  [H]   adjusted loss history, NEWEST FIRST                 */
#define B2E_STATE_RAW_LOSSES  5   /* float  [5]   raw loss history, NEWEST FIRST                      */
#define B2E_STATE_RAW_GSUMS   6   /* double [5]   per-entry sum of the raw gradient history           */
#define B2E_STATE_STEP        7   /* int32  [1]   BaseEnvironment.current_step                        */
#define B2E_STATE_CURSOR      8   /* int32  [1]   batch number inside the epoch                       */
#define B2E_STATE_ORDER       9   /* int32  [N]   current row order of the env's data set             */

typedef struct b2e_env *b2e_handle;

typedef struct b2e_config {
    int32_t  struct_size;         /* = sizeof(b2e_config) */
    int32_t  device;              /* CUDA ordinal */
    int32_t  env_kind;
    int32_t  problem_kind;
    int32_t  num_features;        /* D */
    int32_t  num_hidden;          /* units of the first relu hidden layer, 0 = none
                                     (utils/utils_tf.py:74-86 create_neural_net) */
    int32_t  num_outputs;         /* C */
    int32_t  num_rows;            /* N rows in the data set */
    int32_t  batch_size;          /* B (load_data default 32, data/load_data.py:47) */
    int32_t  num_envs;            /* E */
    int32_t  max_batches;         /* episode length (multioptlrs.py:39) */
    int32_t  max_history;         /* H (multioptlrs.py:39) */
    int32_t  history_version;     /* utils/utils_env.py:9-47  */
    int32_t  observation_version; /* utils/utils_env.py:126-164 */
    int32_t  action_version;      /* utils/utils_env.py:102-123 / multioptimize.py:95-102 */
    int32_t  reward_version;      /* utils/utils_env.py:71-99 */
    int32_t  row_order;
    int32_t  index_mode;
    int32_t  auto_reset;          /* 1: finished envs are reset inside b2e_step, the row block
                                     of such an env holds the RESET observation
                                     (vectorize/concurrentvecenv.py:32-38) */
    int32_t  env_base;            /* global index of this handle's env 0 (0..2^31-1-num_envs): the on-device
                                     Glorot initialiser draws env e's parameters as those of env env_base + e,
                                     so a shard of envs [env_base, env_base + num_envs) of a larger batch
                                     starts and auto-resets from the weights that batch gives them */
    int32_t  hidden_more[B2E_MAX_LAYERS]; /* widths of the 2nd, 3rd ... hidden layers, 0 terminated
                                     (the reference default is layers=(256, 256)) */
    uint64_t init_seed;           /* seed of the on-device Glorot-uniform initialiser */
} b2e_config;

/* OptVecEnv.__init__ + MultiOptLRs.__init__ / MultiOptimize.__init__ + get_problem
 * (vectorize/optvecenv.py:60-68, envs/multioptlrs.py:39-61, envs/multioptimize.py:40-76,
 * problems/__init__.py:7-16).  Allocates all device state. */
int b2e_create(const b2e_config *cfg, b2e_handle *out);
void b2e_destroy(b2e_handle h);
/* Text of the last error on this handle (or of the last failed b2e_create if h is NULL). */
const char *b2e_last_error(b2e_handle h);
int b2e_abi_version(void);

int b2e_num_params(b2e_handle h);   /* BaseProblem.size, problems/base_problem.py:65-68 */
int b2e_obs_dim(b2e_handle h);      /* observation_space.shape[0], utils/utils_env.py:22-44 */
int b2e_history_depth(b2e_handle h); /* depth of the adjusted History: max_history, or 1 for
                                       MultiOptimize history versions 0 and 2 (utils_env.py:22-31) */

/* load_data / InMemoryDataSet.__init__ (data/load_data.py:47-112, dataset/inmemorydataset.py:11-15).
 * features [N,D] float32 row-major; targets: int32 labels [N] (softmax) or float32 [N,C]
 * (linreg).  The library keeps its own (row padded) copy. */
int b2e_bind_dataset(b2e_handle h, const float *features, const void *targets, void *stream);

/* The permutation each env's epoch-end shuffle applies (utils/utils_math.py:10-22 +
 * utils/utils_common.py:12-23 give every shuffle of one env the same permutation) and the
 * initial row order.  perms: int32 [E,N] (per_env != 0) or [N]; init_orders: int32 [E,N]
 * or NULL for the identity.  B2E_INDEX_INTERNAL only. */
int b2e_set_index_stream(b2e_handle h, const int32_t *perms, int per_env,
                         const int32_t *init_orders, void *stream);

/* OptVecEnv.reset / _worker 'reset' (vectorize/optvecenv.py:90-91, concurrentvecenv.py:39-41,
 * envs/baseenvironment.py:43-49, envs/multioptlrs.py:66-78).  env_mask: uint8 [E] or NULL =
 * all.  init_params: float32 [E,P] or NULL = on-device Glorot-uniform / zero bias
 * (keras Dense defaults).  batch_idx/batch_cnt: EXTERNAL index mode only, else NULL.
 * obs_out: float32 [E*P, obs_dim] in VecEnv row order; only rows of reset envs are written. */
int b2e_reset(b2e_handle h, const uint8_t *env_mask, const float *init_params,
              const int32_t *batch_idx, const int32_t *batch_cnt, float *obs_out,
              void *stream);

/* OptVecEnv.step_async + step_wait (vectorize/optvecenv.py:70-88) = E x
 * MultiOptLRs.base_step / MultiOptimize.base_step.
 *   actions   float32 [E*P]  one action per agent row, VecEnv row order
 *   obs_out   float32 [E*P, obs_dim], or NULL for a RING-ONLY step (MultiOptLRs envs on the large-problem
 *             pipeline): the observation rows are not materialised -- the adjusted-history rings, which a
 *             device policy reads in place (b200policy.h, b2p_act_env), are the observation; state, rewards,
 *             done flags and info are those of the ordinary step
 *   reward_out float32 [E], done_out uint8 [E]   (per env; the VecEnv surface repeats them P times)
 *   info_out  double  [E, B2E_INFO_STRIDE]: the 14 values of envs/multioptlrs.py:111-127 in
 *             that order (loss = NaN unless terminal), then episode r, episode l
 *             (envs/baseenvironment.py:40). */
int b2e_step(b2e_handle h, const float *actions, const int32_t *batch_idx,
             const int32_t *batch_cnt, float *obs_out, float *reward_out,
             uint8_t *done_out, double *info_out, void *stream);

/* BaseProblem.get (problems/optimize_nn.py:152-159): gradient [E,P] and loss [E] of every
 * env's current parameters on its current minibatch.  Does not change env state. */
int b2e_eval(b2e_handle h, const int32_t *batch_idx, const int32_t *batch_cnt,
             float *grad_out, float *loss_out, void *stream);

/* State access for parity tests, checkpoints and BaseProblem.set_parameters
 * (problems/optimize_nn.py:142-150).  Buffers are dense [E, stride] arrays. */
int b2e_get_state(b2e_handle h, int which, void *dst, size_t bytes, void *stream);
int b2e_set_state(b2e_handle h, int which, const void *src, size_t bytes, void *stream);

/* The minibatch every env will use in its next step: idx int32 [E,B], cnt int32 [E]. */
int b2e_get_batch_indices(b2e_handle h, int32_t *idx_out, int32_t *cnt_out, void *stream);

/* BaseProblem.next (problems/optimize_nn.py:102-112) for the envs in env_mask (uint8 [E] or
 * NULL = all): advance to the next minibatch, reshuffling at the end of an epoch. */
int b2e_next_batch(b2e_handle h, const uint8_t *env_mask, void *stream);

/* Per-kernel timing of the large-problem step pipeline (bench bookkeeping, off by default):
 * with tracing enabled b2e_step records a CUDA event between its kernels; b2e_get_trace
 * synchronises on them and returns how many durations (ms) it wrote, in launch order:
 * eval(w_{t-1}), update, eval(w_t), observations.  Returns 0 for the single-kernel path. */
int b2e_set_trace(b2e_handle h, int enabled);
int b2e_get_trace(b2e_handle h, float *ms_out, int capacity);

/* Kernel launches issued on behalf of this handle so far (bench bookkeeping). */
int64_t b2e_launch_count(b2e_handle h);

#ifdef __cplusplus
}
#endif
#endif /* B200ENV_H */
