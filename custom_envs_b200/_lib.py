"""ctypes binding of libb200env.so (C ABI in include/b200env.h).

The shared object is built in-tree by ``__graft_entry__.build()`` /
``custom_envs_b200.build.build_library()``.  There is NO CPU fallback: if the library is
missing or cannot be loaded, the product path raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libb200env.so')

ENV_MULTIOPTLRS, ENV_MULTIOPTIMIZE = 0, 1
PROBLEM_SOFTMAX, PROBLEM_LINREG, PROBLEM_FUNC = 0, 1, 2
ROWS_LEXICOGRAPHIC, ROWS_NATURAL = 0, 1
INDEX_INTERNAL, INDEX_EXTERNAL = 0, 1
INFO_STRIDE = 16
MAX_HISTORY = 32
MAX_LAYERS = 8
(STATE_PARAMS, STATE_GRAD_PREV, STATE_ADJ_WEIGHTS, STATE_ADJ_GRADS, STATE_ADJ_LOSSES,
 STATE_RAW_LOSSES, STATE_RAW_GSUMS, STATE_STEP, STATE_CURSOR, STATE_ORDER) = range(10)

EXPORTS = (
    'b2e_abi_version', 'b2e_create', 'b2e_destroy', 'b2e_last_error', 'b2e_num_params',
    'b2e_obs_dim', 'b2e_history_depth', 'b2e_bind_dataset', 'b2e_set_index_stream', 'b2e_reset', 'b2e_step',
    'b2e_step_adam',
    'b2e_eval', 'b2e_get_state', 'b2e_set_state', 'b2e_get_batch_indices', 'b2e_next_batch',
    'b2e_set_trace', 'b2e_get_trace', 'b2e_launch_count',
    # data front-end (include/b200data.h)
    'b2d_last_error', 'b2d_resize_nearest', 'b2d_minmax_workspace', 'b2d_column_minmax',
    'b2d_normalize', 'b2d_rank_workspace', 'b2d_label_ranks', 'b2d_onehot', 'b2d_shuffle_permutations',
    # shared per-agent policy (include/b200policy.h)
    'b2p_create', 'b2p_destroy', 'b2p_last_error', 'b2p_set_weights', 'b2p_act', 'b2p_act_env', 'b2p_set_seed_counter',
    'b2p_set_value_weights', 'b2p_step', 'b2p_step_env', 'b2p_gae',
    'b2p_obs_width', 'b2p_tanh_table', 'b2p_ppo_indices', 'b2p_ppo_adv_stats_workspace_size', 'b2p_ppo_adv_stats', 'b2p_ppo_workspace_size', 'b2p_ppo_grad',
    'b2p_set_row_base', 'b2p_ppo_partial_size', 'b2p_ppo_grad_partial', 'b2p_ppo_combine', 'b2p_ppo_adv_moments',
    'b2p_ppo_adv_combine')
DTYPE_U8, DTYPE_I32, DTYPE_F32, DTYPE_F64 = range(4)


class Config(ctypes.Structure):
    _fields_ = [(name, ctypes.c_int32) for name in (
        'struct_size', 'device', 'env_kind', 'problem_kind', 'num_features', 'num_hidden',
        'num_outputs', 'num_rows', 'batch_size', 'num_envs', 'max_batches', 'max_history',
        'history_version', 'observation_version', 'action_version', 'reward_version',
        'row_order', 'index_mode', 'auto_reset', 'env_base')] + [
        ('hidden_more', ctypes.c_int32 * MAX_LAYERS), ('init_seed', ctypes.c_uint64)]


class Adam(ctypes.Structure):
    """b2e_adam: the constants of b2e_step_adam (Keras 2.2 Adam)."""
    _fields_ = [(name, ctypes.c_float) for name in ('beta_1', 'beta_2', 'epsilon')]


class StepOut(ctypes.Structure):
    """b2p_step_out: device pointers of the outputs of one b2p_step / b2p_step_env launch (NULL = not computed)."""
    _fields_ = [(name, ctypes.c_void_p) for name in ('actions', 'actions_raw', 'values', 'neglogp', 'obs_bf16')]


class PpoBatch(ctypes.Structure):
    """b2p_ppo_batch: device pointers of a time-major rollout buffer."""
    _fields_ = [(name, ctypes.c_void_p) for name in ('obs_bf16', 'actions_raw', 'neglogp', 'values', 'returns')] + [
        ('T', ctypes.c_int), ('rows', ctypes.c_int64)]


class PpoParams(ctypes.Structure):
    """b2p_ppo_params: loss coefficients and the minibatch of one b2p_ppo_grad call."""
    _fields_ = [(name, ctypes.c_float) for name in ('cliprange', 'cliprange_vf', 'ent_coef', 'vf_coef', 'log_std')] + [
        ('key', ctypes.c_uint64), ('begin', ctypes.c_int64), ('count', ctypes.c_int64), ('adv_stats', ctypes.c_void_p)]


class B200EnvError(RuntimeError):
    pass


_lib = None


def load():
    """Load libb200env.so; raises if it has not been built (no fallback by design)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200EnvError(
            'libb200env.so is not built: run `python -c "import __graft_entry__ as g; g.build()"` '
            '(there is no CPU fallback for the optimise-env step)')
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, usize = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
    lib.b2e_abi_version.restype = i32
    lib.b2e_create.argtypes = [ctypes.POINTER(Config), ctypes.POINTER(vp)]
    lib.b2e_destroy.argtypes = [vp]
    lib.b2e_destroy.restype = None
    lib.b2e_last_error.argtypes = [vp]
    lib.b2e_last_error.restype = ctypes.c_char_p
    lib.b2e_num_params.argtypes = [vp]
    lib.b2e_obs_dim.argtypes = [vp]
    lib.b2e_history_depth.argtypes = [vp]
    lib.b2e_bind_dataset.argtypes = [vp, vp, vp, vp]
    lib.b2e_set_index_stream.argtypes = [vp, vp, i32, vp, vp]
    lib.b2e_reset.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.b2e_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b2e_step_adam.argtypes = [vp, ctypes.POINTER(Adam), vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b2e_eval.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.b2e_get_state.argtypes = [vp, i32, vp, usize, vp]
    lib.b2e_set_state.argtypes = [vp, i32, vp, usize, vp]
    lib.b2e_get_batch_indices.argtypes = [vp, vp, vp, vp]
    lib.b2e_next_batch.argtypes = [vp, vp, vp]
    lib.b2e_set_trace.argtypes = [vp, i32]
    lib.b2e_get_trace.argtypes = [vp, ctypes.POINTER(ctypes.c_float), i32]
    lib.b2e_launch_count.argtypes = [vp]
    lib.b2e_launch_count.restype = ctypes.c_int64
    i64 = ctypes.c_int64
    lib.b2d_last_error.argtypes = []
    lib.b2d_last_error.restype = ctypes.c_char_p
    lib.b2d_resize_nearest.argtypes = [vp, i32, i64, i32, i32, vp, vp, i32, i32, vp, vp]
    lib.b2d_minmax_workspace.argtypes = [i32]
    lib.b2d_minmax_workspace.restype = usize
    lib.b2d_column_minmax.argtypes = [vp, i32, i64, i32, vp, vp, vp, vp]
    lib.b2d_normalize.argtypes = [vp, i32, i64, i32, vp, vp, vp, i32, i64, vp]
    lib.b2d_rank_workspace.argtypes = []
    lib.b2d_rank_workspace.restype = usize
    lib.b2d_label_ranks.argtypes = [vp, i64, vp, ctypes.POINTER(ctypes.c_int32), vp, vp]
    lib.b2d_onehot.argtypes = [vp, i64, i32, vp, i32, vp, vp]
    lib.b2d_shuffle_permutations.argtypes = [vp, i32, i64, i32, vp, vp]
    f32, u64 = ctypes.c_float, ctypes.c_uint64
    lib.b2p_create.argtypes = [i32, i32, i32, ctypes.POINTER(vp)]
    lib.b2p_obs_width.argtypes = [i32]
    lib.b2p_obs_width.restype = i32
    lib.b2p_destroy.argtypes = [vp]
    lib.b2p_destroy.restype = None
    lib.b2p_last_error.argtypes = [vp]
    lib.b2p_last_error.restype = ctypes.c_char_p
    lib.b2p_set_weights.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b2p_set_seed_counter.argtypes = [vp, vp]
    lib.b2p_act.argtypes = [vp, vp, i64, vp, f32, u64, f32, f32, vp]
    lib.b2p_act_env.argtypes = [vp, vp, vp, f32, u64, f32, f32, vp]
    lib.b2p_set_value_weights.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b2p_step.argtypes = [vp, vp, i64, ctypes.POINTER(StepOut), f32, f32, u64, f32, f32, vp]
    lib.b2p_step_env.argtypes = [vp, vp, ctypes.POINTER(StepOut), f32, f32, u64, f32, f32, vp]
    lib.b2p_gae.argtypes = [vp, vp, vp, i32, i64, i64, ctypes.c_double, ctypes.c_double, vp, vp, vp]
    lib.b2p_tanh_table.argtypes = [vp, vp]
    lib.b2p_ppo_indices.argtypes = [u64, i64, i64, i64, vp, vp]
    lib.b2p_ppo_adv_stats_workspace_size.argtypes = [i64, i64]
    lib.b2p_ppo_adv_stats_workspace_size.restype = usize
    lib.b2p_ppo_adv_stats.argtypes = [ctypes.POINTER(PpoBatch), u64, i64, vp, vp, vp]
    lib.b2p_ppo_workspace_size.argtypes = [vp]
    lib.b2p_ppo_workspace_size.restype = usize
    lib.b2p_ppo_grad.argtypes = [vp, ctypes.POINTER(PpoBatch), ctypes.POINTER(PpoParams), vp, vp, vp, vp]
    lib.b2p_set_row_base.argtypes = [vp, i64]
    lib.b2p_ppo_partial_size.argtypes = [vp]
    lib.b2p_ppo_partial_size.restype = usize
    lib.b2p_ppo_grad_partial.argtypes = [vp, ctypes.POINTER(PpoBatch), ctypes.POINTER(PpoParams), i64, vp, vp, vp]
    lib.b2p_ppo_combine.argtypes = [vp, vp, i32, i64, f32, f32, f32, vp, vp, vp]
    lib.b2p_ppo_adv_moments.argtypes = [ctypes.POINTER(PpoBatch), u64, i64, vp, vp, vp]
    lib.b2p_ppo_adv_combine.argtypes = [vp, i32, i64, vp, vp]
    if lib.b2e_abi_version() != 2:
        raise B200EnvError('libb200env.so ABI version mismatch')
    _lib = lib
    return lib
