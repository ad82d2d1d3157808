"""Device-resident batched optimise-env: E lock-step MultiOptLRs / MultiOptimize envs on one GPU.

Host-side mirror of what ``OptVecEnv([...E env fns...])`` is in the reference
(vectorize/optvecenv.py:57-91): same row order, same per-step outputs, but state lives in
HBM and every step is ONE launch of the fused sm_100a kernel in libb200env.so (through
the C ABI of include/b200env.h).  torch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from custom_envs_b200 import _lib

INFO_KEYS = ('loss', 'batch_loss', 'weights_mean', 'weights_sum', 'actions_mean',
             'actions_std', 'states_mean', 'states_sum', 'grads_mean', 'grads_sum',
             'loss_mean', 'adjusted_loss', 'adjusted_grad', 'grad_diff')   # multioptlrs.py:111-127

_PROBLEM_KINDS = {'softmax': _lib.PROBLEM_SOFTMAX, 'nn': _lib.PROBLEM_SOFTMAX,
                  'linreg': _lib.PROBLEM_LINREG, 'func': _lib.PROBLEM_FUNC}
_STATE = {'params': (_lib.STATE_PARAMS, torch.float32), 'grad_prev': (_lib.STATE_GRAD_PREV, torch.float32),
          'adj_weights': (_lib.STATE_ADJ_WEIGHTS, torch.float32),
          'adj_grads': (_lib.STATE_ADJ_GRADS, torch.float32),
          'adj_losses': (_lib.STATE_ADJ_LOSSES, torch.float32),
          'raw_losses': (_lib.STATE_RAW_LOSSES, torch.float32),
          'raw_gsums': (_lib.STATE_RAW_GSUMS, torch.float64),
          'step': (_lib.STATE_STEP, torch.int32), 'cursor': (_lib.STATE_CURSOR, torch.int32),
          'order': (_lib.STATE_ORDER, torch.int32)}


@dataclass(frozen=True)
class ProblemSpec:
    """kind: 'softmax' (Dense[+relu Dense]+softmax CE, reference problems/optimize_nn.py),
    'linreg', or 'func' (Rosenbrock, reference problems/optimize_function.py)."""
    kind: str = 'softmax'
    num_features: int = 4
    hidden: tuple = ()
    num_outputs: int = 3

    @property
    def size(self):
        if self.kind == 'func':
            return 2
        dims = (self.num_features,) + tuple(self.hidden) + (self.num_outputs,)
        return int(sum(a * b + b for a, b in zip(dims[:-1], dims[1:])))


def env_permutations(num_rows, seeds):
    """perm[e] = what ``np.random.shuffle(arange(N))`` yields from RandomState(seed_e); the
    reference's ``use_random_state`` hands every epoch-end shuffle of an env the same
    generator state (utils/utils_math.py:10-22), hence one permutation per env."""
    out = np.empty((len(seeds), num_rows), np.int32)
    for i, seed in enumerate(seeds):
        state = seed if isinstance(seed, np.random.RandomState) else np.random.RandomState(seed)
        if isinstance(seed, np.random.RandomState):
            copy = np.random.RandomState()
            copy.set_state(seed.get_state())
            state = copy
        idx = np.arange(num_rows, dtype=np.int32)
        state.shuffle(idx)
        out[i] = idx
    return out


def _ptr(tensor):
    return ctypes.c_void_p(0 if tensor is None else tensor.data_ptr())


def env_permutations_device(num_rows, seeds, device):
    """``env_permutations`` on the device (``b2d_shuffle_permutations``: numpy's legacy MT19937 stream, seeding and
    Fisher-Yates shuffle restated bit for bit, one thread per generator): int32 [E, N] device tensor.  Integer seeds
    travel as 4 bytes each; RandomState objects (e.g. classic gym's hash-seeded generators) as their 625-word state.
    Host cost of the numpy path: ~1.2 ms per env at 60 000 rows, i.e. 80 s for the 64 K envs of BASELINE config 5."""
    lib = _lib.load()
    dev = torch.device(device)
    seeds = list(seeds)
    plain = all(isinstance(s, (int, np.integer)) and 0 <= int(s) < 2 ** 32 for s in seeds)
    if plain:
        gen = torch.as_tensor(np.asarray(seeds, dtype=np.uint32).view(np.int32)).to(dev)
        mode = 0
    else:
        states = np.empty((len(seeds), 625), np.uint32)
        for i, seed in enumerate(seeds):
            state = (seed if isinstance(seed, np.random.RandomState) else np.random.RandomState(seed)).get_state()
            states[i, :624] = state[1]
            states[i, 624] = state[2]
        gen = torch.as_tensor(states.view(np.int32)).to(dev)
        mode = 1
    out = torch.empty((len(seeds), int(num_rows)), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        code = lib.b2d_shuffle_permutations(_ptr(gen), mode, len(seeds), int(num_rows), _ptr(out),
                                            ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    if code:
        raise _lib.B200EnvError(lib.b2d_last_error().decode())
    torch.cuda.current_stream(dev).synchronize()              # `gen` may be freed by the caller's scope
    return out


class BatchedOptEnv:
    def __init__(self, problem: ProblemSpec, features=None, targets=None, num_envs=1,
                 batch_size=32, max_batches=400, max_history=5, env_kind='optlrs',
                 history_version=3, observation_version=3, action_version=0, reward_version=6,
                 row_order='lexicographic', index_mode='internal', auto_reset=True,
                 seeds=None, perms=None, init_orders=None, device='cuda:0', init_seed=0,
                 materialize_obs=True, env_base=0):
        """``materialize_obs=False``: no [E*P, obs_dim] observation matrix is allocated (12.5 GB at
        BASELINE config 4); every step is then ring-only and the consumer reads the adjusted-history
        rings in place (``custom_envs_b200.vectorize.device_policy.DevicePolicy.act_env``).

        ``env_base``: the global index of this batch's env 0, when it is the shard
        ``[env_base, env_base + num_envs)`` of a larger batch (``sharding.shard_bases``).  The on-device Glorot
        initialiser and the default ``seeds`` then follow the global index, so the shard's envs start and
        auto-reset exactly as they do inside the whole batch; pass that batch's ``init_seed`` and the shard's
        slice of its ``seeds``."""
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.B200EnvError('BatchedOptEnv needs a CUDA device (no CPU fallback)')
        self.device = torch.device(device)
        self.problem = problem
        if len(problem.hidden) > _lib.MAX_LAYERS - 1:
            raise _lib.B200EnvError('at most %d hidden layers' % (_lib.MAX_LAYERS - 1))
        self.num_envs = int(num_envs)
        self.index_mode = index_mode
        cfg = _lib.Config()
        cfg.struct_size = ctypes.sizeof(_lib.Config)
        cfg.device = self.device.index or 0
        cfg.env_kind = _lib.ENV_MULTIOPTLRS if env_kind == 'optlrs' else _lib.ENV_MULTIOPTIMIZE
        self.env_kind_name = 'optlrs' if env_kind == 'optlrs' else 'optimize'
        cfg.problem_kind = _PROBLEM_KINDS[problem.kind]
        func = problem.kind == 'func'
        if not func:
            features = torch.as_tensor(np.asarray(features, np.float32) if not torch.is_tensor(features)
                                       else features).to(self.device, torch.float32).contiguous()
            num_rows = features.shape[0]
            batch_size = num_rows if batch_size is None else int(batch_size)
            cfg.num_features, cfg.num_outputs = problem.num_features, problem.num_outputs
            cfg.num_hidden = problem.hidden[0] if problem.hidden else 0
            for i, width in enumerate(problem.hidden[1:]):
                cfg.hidden_more[i] = int(width)
            cfg.num_rows, cfg.batch_size = num_rows, batch_size
            assert features.shape[1] == problem.num_features
        self.batch_size = 1 if func else batch_size
        cfg.num_envs = self.num_envs
        cfg.max_batches, cfg.max_history = int(max_batches), int(max_history)
        cfg.history_version, cfg.observation_version = history_version, observation_version
        cfg.action_version, cfg.reward_version = action_version, reward_version
        cfg.row_order = _lib.ROWS_LEXICOGRAPHIC if row_order == 'lexicographic' else _lib.ROWS_NATURAL
        cfg.index_mode = _lib.INDEX_INTERNAL if index_mode == 'internal' else _lib.INDEX_EXTERNAL
        cfg.auto_reset = int(bool(auto_reset))
        cfg.init_seed = int(init_seed)
        self.env_base = cfg.env_base = int(env_base)
        self.max_batches, self.max_history = int(max_batches), int(max_history)
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            if self.lib.b2e_create(ctypes.byref(cfg), ctypes.byref(handle)):
                raise _lib.B200EnvError(self.lib.b2e_last_error(None).decode())
        self.handle = handle
        self.num_params = self.lib.b2e_num_params(handle)
        self.obs_dim = self.lib.b2e_obs_dim(handle)
        self.history_depth = self.lib.b2e_history_depth(handle)
        self.num_rows = self.num_envs * self.num_params
        dev = self.device
        self.obs = (torch.empty((self.num_rows, self.obs_dim), dtype=torch.float32, device=dev)
                    if materialize_obs else None)
        self._fixed_ptrs = None
        self._device_index = dev.index if dev.index is not None else torch.cuda.current_device()
        self.reward = torch.zeros(self.num_envs, dtype=torch.float32, device=dev)
        self.done = torch.zeros(self.num_envs, dtype=torch.uint8, device=dev)
        self.info = torch.zeros((self.num_envs, _lib.INFO_STRIDE), dtype=torch.float64, device=dev)
        if not func:
            if problem.kind == 'linreg':
                targets = torch.as_tensor(np.asarray(targets, np.float32) if not torch.is_tensor(targets)
                                          else targets).to(dev, torch.float32).contiguous()
                targets = targets.reshape(num_rows, problem.num_outputs)
            else:
                targets = torch.as_tensor(np.asarray(targets) if not torch.is_tensor(targets)
                                          else targets).to(dev, torch.int32).contiguous()
            self._check(self.lib.b2e_bind_dataset(handle, _ptr(features), _ptr(targets), self._stream()))
            if index_mode == 'internal':
                if perms is None:                    # the epoch permutation of every env, generated on the device
                    seeds = range(self.env_base, self.env_base + self.num_envs) if seeds is None else seeds
                    perms = env_permutations_device(num_rows, list(seeds), dev)
                if torch.is_tensor(perms):
                    perms = perms.to(dev, torch.int32).contiguous()
                else:
                    perms = torch.as_tensor(np.ascontiguousarray(perms, np.int32)).to(dev)
                if perms.ndim == 2 and perms.shape[0] == 1:
                    perms = perms[0]
                per_env = int(perms.ndim == 2)       # [N] = one permutation shared by all envs
                assert perms.shape[-1] == num_rows and (not per_env or perms.shape[0] == self.num_envs)
                if init_orders is not None:
                    if torch.is_tensor(init_orders):        # e.g. built on the device for very many envs
                        init_orders = init_orders.to(dev, torch.int32).contiguous()
                    else:
                        init_orders = torch.as_tensor(np.ascontiguousarray(init_orders, np.int32)).to(dev)
                    assert tuple(init_orders.shape) == (self.num_envs, num_rows)
                self._check(self.lib.b2e_set_index_stream(handle, _ptr(perms), per_env,
                                                          _ptr(init_orders), self._stream()))
            torch.cuda.synchronize(dev)       # library copied what it needs

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, code):
        if code:
            raise _lib.B200EnvError(self.lib.b2e_last_error(self.handle).decode())

    def close(self):
        if getattr(self, 'handle', None):
            torch.cuda.synchronize(self.device)
            self.lib.b2e_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:      # noqa: BLE001 (interpreter shutdown)
            pass

    @property
    def launch_count(self):
        return int(self.lib.b2e_launch_count(self.handle))

    def _idx(self, batch_idx, batch_cnt):
        if batch_idx is None:
            return None, None
        idx = torch.as_tensor(batch_idx).to(self.device, torch.int32).contiguous()
        cnt = torch.as_tensor(batch_cnt).to(self.device, torch.int32).contiguous()
        assert idx.shape == (self.num_envs, self.batch_size) and cnt.shape == (self.num_envs,)
        return idx, cnt

    # --------------------------------------------------------------- env surface
    def reset(self, env_mask=None, init_params=None, batch_idx=None, batch_cnt=None):
        """-> obs [E*P, obs_dim] float32 device tensor (rows of envs outside the mask keep
        their previous content)."""
        mask = None
        if env_mask is not None:
            mask = torch.as_tensor(env_mask).to(self.device, torch.uint8).contiguous()
        params = None
        if init_params is not None:
            params = torch.as_tensor(init_params).to(self.device, torch.float32).contiguous()
            assert params.shape == (self.num_envs, self.num_params)
        idx, cnt = self._idx(batch_idx, batch_cnt)
        self._check(self.lib.b2e_reset(self.handle, _ptr(mask), _ptr(params), _ptr(idx), _ptr(cnt),
                                       _ptr(self.obs), self._stream()))
        return self.obs

    def step(self, actions, batch_idx=None, batch_cnt=None, obs_out=None, ring_only=False):
        """actions: [E*P] (or [E*P,1]) float32 device tensor in VecEnv row order.
        -> (obs [E*P,obs_dim], reward [E] f32, done [E] u8, info [E,16] f64): views of
        buffers that the next step overwrites.  ``obs_out``: write the observation rows there
        instead (any device-accessible float32 buffer of that shape, e.g. pinned host memory:
        the rows then cross PCIe straight from the observation kernel).  ``ring_only``: do not
        write observation rows at all (obs is None in the result): the adjusted-history rings are
        the observation, read in place by a device policy (MultiOptLRs, large problems)."""
        if (batch_idx is None and obs_out is None and not ring_only and self.obs is not None
                and actions.dtype == torch.float32 and actions.device == self.device
                and actions.is_contiguous() and actions.numel() == self.num_rows):
            # the usual call: nothing to convert or check, raw stream handle, pointers of the fixed buffers cached
            # (the tiny problems are bound by this host path: 14 -> 9 us per call)
            if self._fixed_ptrs is None:
                self._fixed_ptrs = (self.reward.data_ptr(), self.done.data_ptr(), self.info.data_ptr())
            fixed = self._fixed_ptrs
            if self.lib.b2e_step(self.handle, actions.data_ptr(), None, None, self.obs.data_ptr(), fixed[0], fixed[1], fixed[2],
                                 torch._C._cuda_getCurrentRawStream(self._device_index)):
                self._check(1)
            return self.obs, self.reward, self.done, self.info
        actions = actions.reshape(-1)
        if actions.dtype != torch.float32 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(self.device, torch.float32).contiguous()
        assert actions.numel() == self.num_rows
        idx, cnt = self._idx(batch_idx, batch_cnt)
        obs = self.obs if obs_out is None else obs_out
        if ring_only or obs is None:
            obs = None
        else:
            assert obs.dtype == torch.float32 and obs.is_contiguous() and obs.numel() == self.num_rows * self.obs_dim
        self._check(self.lib.b2e_step(self.handle, _ptr(actions), _ptr(idx), _ptr(cnt), _ptr(obs),
                                      _ptr(self.reward), _ptr(self.done), _ptr(self.info),
                                      self._stream()))
        return obs, self.reward, self.done, self.info

    def capture_step_graph(self, actions, steps=None):
        """Record the batched step into a CUDA graph (``b2e_step`` enqueues kernels on the caller's
        stream and nothing else: no allocation, no synchronisation, no host read-back).

        ``actions`` is the static device buffer the replays read; refill it in place between
        replays.  The kernel pipeline of the large problems alternates between two gradient
        buffers, so one replay covers TWO consecutive steps there (``steps`` defaults to that
        period; the small fused problems replay one step).  Returns ``(graph, steps)``;
        ``graph.replay()`` leaves the outputs of the last step in ``self.obs / reward / done / info``.
        Host-supplied minibatch indices (index_mode='external') cannot be captured."""
        if self.index_mode != 'internal' and self.problem.kind != 'func':
            raise _lib.B200EnvError('capture_step_graph needs the on-device minibatch stream')
        actions = actions.reshape(-1)
        assert actions.dtype == torch.float32 and actions.device == self.device and actions.is_contiguous()
        period = 2 if self.num_params >= 4096 or self.env_kind_name == 'optimize' else 1
        steps = period if steps is None else int(steps)
        if steps % period:
            raise _lib.B200EnvError('this problem replays in multiples of %d steps' % period)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            self.step(actions)                       # warm-up outside the capture (lazy module loading)
            if period == 2:
                self.step(actions)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        with torch.cuda.graph(graph):
            for _ in range(steps):
                self.step(actions)
        return graph, steps

    def evaluate(self, batch_idx=None, batch_cnt=None):
        """BaseProblem.get for every env: (grad [E,P], loss [E]) on the current minibatch."""
        grad = torch.empty((self.num_envs, self.num_params), dtype=torch.float32, device=self.device)
        loss = torch.empty(self.num_envs, dtype=torch.float32, device=self.device)
        idx, cnt = self._idx(batch_idx, batch_cnt)
        self._check(self.lib.b2e_eval(self.handle, _ptr(idx), _ptr(cnt), _ptr(grad), _ptr(loss),
                                      self._stream()))
        return grad, loss

    def _state_shape(self, name):
        e, p, h = self.num_envs, self.num_params, self.history_depth
        return {'params': (e, p), 'grad_prev': (e, p), 'adj_weights': (e, h, p),
                'adj_grads': (e, h, p), 'adj_losses': (e, h), 'raw_losses': (e, 5),
                'raw_gsums': (e, 5), 'step': (e,), 'cursor': (e,),
                'order': (e, getattr(self, '_num_data_rows', 0))}[name]

    def get_state(self, name):
        which, dtype = _STATE[name]
        shape = self._state_shape(name) if name != 'order' else None
        if name == 'order':
            raise NotImplementedError('use batch_indices()')
        out = torch.empty(shape, dtype=dtype, device=self.device)
        self._check(self.lib.b2e_get_state(self.handle, which, _ptr(out),
                                           out.numel() * out.element_size(), self._stream()))
        return out

    def set_state(self, name, value):
        which, dtype = _STATE[name]
        value = torch.as_tensor(value).to(self.device, dtype).contiguous()
        assert tuple(value.shape) == self._state_shape(name), (value.shape, self._state_shape(name))
        self._check(self.lib.b2e_set_state(self.handle, which, _ptr(value),
                                           value.numel() * value.element_size(), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def batch_indices(self):
        idx = torch.empty((self.num_envs, self.batch_size), dtype=torch.int32, device=self.device)
        cnt = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        self._check(self.lib.b2e_get_batch_indices(self.handle, _ptr(idx), _ptr(cnt), self._stream()))
        return idx, cnt

    def next_batch(self, env_mask=None):
        """BaseProblem.next for the masked envs."""
        mask = None
        if env_mask is not None:
            mask = torch.as_tensor(env_mask).to(self.device, torch.uint8).contiguous()
        self._check(self.lib.b2e_next_batch(self.handle, _ptr(mask), self._stream()))

    PIPELINE_KERNELS = ('eval_kernel<w_prev>', 'update_kernel', 'eval_kernel<w_new>', 'obs_kernel')

    def set_trace(self, enabled=True):
        self._check(self.lib.b2e_set_trace(self.handle, int(enabled)))

    def last_step_kernel_ms(self):
        """Per-kernel durations of the last traced step ({} for the single-kernel path)."""
        buf = (ctypes.c_float * 8)()
        n = self.lib.b2e_get_trace(self.handle, buf, 8)
        return {name: float(buf[i]) for i, name in enumerate(self.PIPELINE_KERNELS[:max(n, 0)])}

    def info_dict(self, info=None):
        """info [E,16] -> {key: np.ndarray[E]} with the reference's key names."""
        arr = (self.info if info is None else info).cpu().numpy()
        out = {key: arr[:, i] for i, key in enumerate(INFO_KEYS)}
        out['episode_r'], out['episode_l'] = arr[:, 14], arr[:, 15].astype(np.int64)
        return out
