"""Shared per-agent policy on the device (C ABI: include/b200policy.h; kernel: csrc/b200policy.cu).

The reference's runner evaluates one stable-baselines ``MlpPolicy`` (two tanh layers of 64, linear
head) on every agent row of the observation matrix that ``OptVecEnv.step_wait`` returned
(run_multiagent_exp_single.py:37-49, vectorize/optvecenv.py:78-88).  ``DevicePolicy`` evaluates the
action head of such a network -- taken from a ``SharedMlpPolicy`` / any ``torch.nn.Sequential`` of
that shape -- with bf16 tcgen05 MMAs, either on a dense observation matrix (``act``) or straight on
the env's adjusted-history rings (``act_env``), in which case the env can step ring-only and the
[sum(P), 3H] matrix never exists.  There is no fallback: without the library / an sm_100 GPU the
constructor raises (``SharedMlpPolicy.act`` is the torch path, and it is the caller's choice).

For PPO, ``step`` / ``value`` are the rest of stable-baselines' ``model.step`` / ``model.value`` (value
tower, unclipped action, neglogp, bf16 observation store), ``DeviceRolloutBuffer`` and
``device_ppo_rollout`` collect a whole rollout with its GAE advantages on the device, and ``ppo_grad`` /
``device_ppo_update`` run PPO2's minibatch updates over it with a fused clipped-surrogate gradient kernel.

Data-parallel PPO over several GPUs: every rank steps its env shard (``BatchedOptEnv(env_base=...)`` and
``DevicePolicy.set_row_base``, ``sharding.shard_bases``), so its rollout holds exactly the rows of those envs in one
unsharded run, and ``device_ppo_update(..., group=...)`` combines the ranks' fp64 partial sums in rank order, so every
rank takes the same optimizer step bit for bit."""
import ctypes
import math

import torch

from custom_envs_b200 import _lib

TANH_F32, TANH_BF16X2, TANH_BF16X2_BOTH = 0, 1, 2


def _ptr(tensor):
    return ctypes.c_void_p(tensor.data_ptr())


class DevicePolicy:
    def __init__(self, obs_dim, device='cuda:0', tanh_mode=TANH_F32, log_std=None, low=-4.0, high=6.0):
        """``low`` / ``high``: the action Box of MultiOptLRs agents (utils_env.get_action_space_optlrs);
        ``log_std``: log of the diagonal Gaussian's standard deviation, None = deterministic."""
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.B200EnvError('DevicePolicy needs a CUDA device (no CPU fallback)')
        self.device = torch.device(device)
        self.obs_dim = int(obs_dim)
        self.low, self.high = float(low), float(high)
        self.set_log_std(log_std)
        self.calls = 0
        self.row_base = 0
        self.seed_counter = None
        self.has_value = False
        handle = ctypes.c_void_p()
        if self.lib.b2p_create(self.device.index or 0, self.obs_dim, int(tanh_mode), ctypes.byref(handle)):
            raise _lib.B200EnvError(self.lib.b2p_last_error(None).decode())
        self.handle = handle
        self.obs_width = obs_width(self.obs_dim)

    @classmethod
    def from_torch(cls, tower, obs_dim=None, **kwargs):
        """``tower``: Linear(obs_dim, 64), Tanh, Linear(64, 64), Tanh, Linear(64, 1) -- e.g.
        ``SharedMlpPolicy.pi`` -- or a module with such a ``.pi`` (its ``log_std`` is taken along, and
        its ``.vf`` tower of the same shape, if any, becomes the value tower of ``step`` / ``value``)."""
        vf = None
        if hasattr(tower, 'pi'):
            if 'log_std' not in kwargs and hasattr(tower, 'log_std'):
                kwargs['log_std'] = tower.log_std.detach()
            vf = getattr(tower, 'vf', None)
            tower = tower.pi
        linears = _tower_linears(tower)
        device = linears[0].weight.device
        policy = cls(obs_dim or linears[0].in_features, device=device, **kwargs)
        policy.set_weights(*[t for lin in linears for t in (lin.weight, lin.bias)])
        if vf is not None:
            policy.set_value_weights(*[t for lin in _tower_linears(vf) for t in (lin.weight, lin.bias)])
        return policy

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, code):
        if code:
            raise _lib.B200EnvError(self.lib.b2p_last_error(self.handle).decode())

    def set_weights(self, w1, b1, w2, b2, w3, b3):
        """torch.nn.Linear layouts ([out, in]); the library copies them (fp32), the kernel rounds to bf16."""
        tensors = [t.detach().to(self.device, torch.float32).contiguous() for t in (w1, b1, w2, b2, w3, b3)]
        assert tensors[0].shape == (64, self.obs_dim) and tensors[2].shape == (64, 64) and tensors[4].numel() == 64
        self._check(self.lib.b2p_set_weights(self.handle, *[_ptr(t) for t in tensors], self._stream()))
        torch.cuda.current_stream(self.device).synchronize()      # the sources may be temporaries

    def set_value_weights(self, w1, b1, w2, b2, w3, b3):
        """The value tower (``SharedMlpPolicy.vf``), in the layouts of ``set_weights``."""
        tensors = [t.detach().to(self.device, torch.float32).contiguous() for t in (w1, b1, w2, b2, w3, b3)]
        assert tensors[0].shape == (64, self.obs_dim) and tensors[2].shape == (64, 64) and tensors[4].numel() == 64
        self._check(self.lib.b2p_set_value_weights(self.handle, *[_ptr(t) for t in tensors], self._stream()))
        torch.cuda.current_stream(self.device).synchronize()
        self.has_value = True

    def set_log_std(self, log_std):
        """Log of the Gaussian's standard deviation (None = deterministic): the noise of later launches and the
        neglogp of ``step``.  PPO trains it (``SharedMlpPolicy.log_std``): hand it over with the tower weights after
        every update."""
        self.log_std = None if log_std is None else float(torch.as_tensor(log_std))
        self.noise_std = 0.0 if log_std is None else math.exp(self.log_std)

    def use_seed_counter(self, enabled=True):
        """Draw the noise seed from a device counter (``self.seed_counter``, int64 [1]) added to the seed argument:
        launches captured in a CUDA graph then see fresh noise on every replay if the graph also advances it."""
        if enabled and self.seed_counter is None:
            self.seed_counter = torch.zeros(1, dtype=torch.int64, device=self.device)
        ptr = ctypes.c_void_p(self.seed_counter.data_ptr() if enabled else 0)
        self._check(self.lib.b2p_set_seed_counter(self.handle, ptr))
        if not enabled:
            self.seed_counter = None

    def set_row_base(self, row_base):
        """Global index of row 0 of every later launch (default 0): local row r draws the exploration noise of global
        row ``row_base + r`` (b2p_set_row_base).  For the shard of envs starting at ``first_env`` with P rows per env
        it is ``first_env * P`` in both VecEnv row orders (``sharding.shard_bases``); the shard's actions, neglogp and
        stored rows then equal those rows of one unsharded batch."""
        self._check(self.lib.b2p_set_row_base(self.handle, int(row_base)))
        self.row_base = int(row_base)

    def _seed(self, seed):
        self.calls += 1
        return ctypes.c_uint64((self.calls if seed is None else int(seed)) & (2 ** 64 - 1))

    def act(self, obs, out=None, seed=None):
        """obs [rows, obs_dim] float32 (dense, e.g. ``BatchedOptEnv.obs``) -> actions [rows]."""
        assert obs.dtype == torch.float32 and obs.is_contiguous() and obs.shape[-1] == self.obs_dim
        rows = obs.numel() // self.obs_dim
        if out is None:
            out = torch.empty(rows, dtype=torch.float32, device=self.device)
        assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == rows
        self._check(self.lib.b2p_act(self.handle, _ptr(obs), rows, _ptr(out), self.noise_std, self._seed(seed),
                                     self.low, self.high, self._stream()))
        return out

    def act_env(self, env, out=None, seed=None):
        """Actions of every agent row of ``env`` (a ``BatchedOptEnv``), read from its rings; VecEnv row order."""
        if out is None:
            out = torch.empty(env.num_rows, dtype=torch.float32, device=self.device)
        assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == env.num_rows
        self._check(self.lib.b2p_act_env(self.handle, env.handle, _ptr(out), self.noise_std, self._seed(seed),
                                         self.low, self.high, self._stream()))
        return out

    def _launch(self, source, seed, actions=None, actions_raw=None, values=None, neglogp=None, obs_bf16=None):
        """One b2p_step (``source`` = dense obs [rows, obs_dim] float32) or b2p_step_env (``source`` = a
        ``BatchedOptEnv``, read from its rings) launch; None outputs are not computed."""
        dense = torch.is_tensor(source)
        if dense:
            assert source.dtype == torch.float32 and source.is_contiguous() and source.shape[-1] == self.obs_dim
            rows = source.numel() // self.obs_dim
        else:
            rows = source.num_rows
        for t in (actions, actions_raw, values, neglogp):
            assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == rows
                                 and t.device == self.device)
        if obs_bf16 is not None:
            assert obs_bf16.dtype == torch.bfloat16 and obs_bf16.is_contiguous() and obs_bf16.numel() == rows * self.obs_width
        if neglogp is not None and self.log_std is None:
            raise ValueError('neglogp needs a stochastic policy (log_std)')
        out = _lib.StepOut(*[t.data_ptr() if t is not None else None
                             for t in (actions, actions_raw, values, neglogp, obs_bf16)])
        log_std = 0.0 if self.log_std is None else self.log_std
        if dense:
            code = self.lib.b2p_step(self.handle, _ptr(source), rows, ctypes.byref(out), self.noise_std, log_std, seed,
                                     self.low, self.high, self._stream())
        else:
            code = self.lib.b2p_step_env(self.handle, source.handle, ctypes.byref(out), self.noise_std, log_std, seed,
                                         self.low, self.high, self._stream())
        self._check(code)

    def _rows(self, source):
        return source.numel() // self.obs_dim if torch.is_tensor(source) else source.num_rows

    def step(self, source, seed=None, obs_bf16=None):
        """stable-baselines' ``model.step`` on every row of ``source`` (dense obs [rows, obs_dim] float32, or a
        ``BatchedOptEnv`` whose rings are read, VecEnv row order) -> (actions, actions_raw, values, neglogp,
        obs_bf16), each [rows] float32: the clipped action the env steps with (bit for bit ``act`` /
        ``act_env`` with the same seed), the unclipped one PPO stores, the value tower's output (None
        without one) and -log p(actions_raw).  ``obs_bf16``: a bf16 [rows, obs_width] tensor to receive the
        observation rows as the network read them (columns obs_dim..obs_width-1 zero), or None."""
        if self.log_std is None:
            raise ValueError('step samples from the Gaussian policy: construct it with a log_std')
        new = lambda: torch.empty(self._rows(source), dtype=torch.float32, device=self.device)   # noqa: E731
        actions, actions_raw, neglogp = new(), new(), new()
        values = new() if self.has_value else None
        self._launch(source, self._seed(seed), actions, actions_raw, values, neglogp, obs_bf16)
        return actions, actions_raw, values, neglogp, obs_bf16

    def value(self, source, out=None):
        """``model.value``: the value tower alone on every row of ``source`` (as in ``step``) -> [rows] float32."""
        if out is None:
            out = torch.empty(self._rows(source), dtype=torch.float32, device=self.device)
        self._launch(source, ctypes.c_uint64(0), values=out)
        return out

    def ppo_grad(self, buffer, key, begin, count, adv_stats, cliprange=0.2, cliprange_vf=None, ent_coef=0.01,
                 vf_coef=0.5, grad=None, stats=None):
        """Gradient of PPO2's loss over the minibatch at positions [begin, begin + count) of the permutation ``key`` of
        ``buffer``'s T * rows samples, at this policy's weights and ``log_std`` (b2p_ppo_grad).  ``adv_stats``: device
        float64 [2] (mean, std of the minibatch's returns - values, e.g. a row of ``ppo_adv_stats``);
        ``cliprange_vf`` None = ``cliprange`` (stable-baselines' default), negative = no value clipping.  Returns
        (grad float32 [2 * tower + 1]: action tower, value tower in ``set_weights`` layouts, then log_std; stats float64
        [6]: pg_loss, vf_loss, entropy, approxkl, clipfrac, loss), both on the device, not synchronised."""
        if self.log_std is None:
            raise ValueError('ppo_grad needs a stochastic policy (log_std)')
        tower = 64 * self.obs_dim + 64 + 64 * 64 + 64 + 64 + 1
        if grad is None:
            grad = torch.empty(2 * tower + 1, dtype=torch.float32, device=self.device)
        if stats is None:
            stats = torch.empty(6, dtype=torch.float64, device=self.device)
        assert grad.dtype == torch.float32 and grad.numel() == 2 * tower + 1 and grad.is_contiguous()
        assert stats.dtype == torch.float64 and stats.numel() == 6
        args = self._ppo_args(buffer, key, begin, count, adv_stats, cliprange, cliprange_vf, ent_coef, vf_coef)
        self._check(self.lib.b2p_ppo_grad(self.handle, *args[:2], _ptr(grad), _ptr(stats), *args[2:]))
        return grad, stats

    def _ppo_args(self, buffer, key, begin, count, adv_stats, cliprange, cliprange_vf, ent_coef, vf_coef):
        """(batch, params, workspace, stream) of a b2p_ppo_grad / b2p_ppo_grad_partial call."""
        assert adv_stats.dtype == torch.float64
        assert buffer.obs_bf16.shape[-1] == self.obs_width, 'the buffer\'s rows are not this policy\'s obs_width wide'
        if getattr(self, '_ppo_ws', None) is None:
            self._ppo_ws = torch.empty(self.lib.b2p_ppo_workspace_size(self.handle), dtype=torch.uint8, device=self.device)
        params = _lib.PpoParams(float(cliprange), float(cliprange if cliprange_vf is None else cliprange_vf),
                                float(ent_coef), float(vf_coef), float(self.log_std), int(key) & (2 ** 64 - 1),
                                int(begin), int(count), adv_stats.data_ptr())
        self._ppo_keep = (_ppo_batch(buffer), params)
        return (ctypes.byref(self._ppo_keep[0]), ctypes.byref(params), _ptr(self._ppo_ws), self._stream())

    @property
    def ppo_partial_size(self):
        """Length of the float64 partial vector of ``ppo_grad_partial``: the 2 * tower + 1 - 1 gradient sums before
        log_std's, then the five loss sums."""
        return int(self.lib.b2p_ppo_partial_size(self.handle))

    def ppo_grad_partial(self, buffer, key, begin, count, count_total, adv_stats, cliprange=0.2, cliprange_vf=None,
                         ent_coef=0.01, vf_coef=0.5, partial=None):
        """This shard's part of PPO2's gradient over a minibatch split across shards (b2p_ppo_grad_partial): the rows
        at positions [begin, begin + count) of the permutation ``key`` of ``buffer``, each scaled by 1 / ``count_total``
        (the size of the union minibatch) rather than 1 / count, normalised with the union's ``adv_stats``
        (``ppo_adv_combine``).  Returns float64 [``ppo_partial_size``] on the device, not synchronised; ``ppo_combine``
        sums the shards' vectors in rank order.  With count_total = count, ``ppo_combine`` of this one vector is
        ``ppo_grad`` bit for bit."""
        if self.log_std is None:
            raise ValueError('ppo_grad_partial needs a stochastic policy (log_std)')
        size = self.ppo_partial_size
        if partial is None:
            partial = torch.empty(size, dtype=torch.float64, device=self.device)
        if partial.dtype != torch.float64 or not partial.is_contiguous() or partial.numel() < size:
            raise ValueError('the partial buffer must be a contiguous float64 tensor of at least %d elements' % size)
        args = self._ppo_args(buffer, key, begin, count, adv_stats, cliprange, cliprange_vf, ent_coef, vf_coef)
        self._check(self.lib.b2p_ppo_grad_partial(self.handle, *args[:2], int(count_total), _ptr(partial), *args[2:]))
        return partial

    def ppo_combine(self, partials, count_total, ent_coef=0.01, vf_coef=0.5, grad=None, stats=None):
        """``partials`` float64 [ranks, ``ppo_partial_size``], the shards' ``ppo_grad_partial`` vectors in rank order ->
        (grad, stats) as ``ppo_grad`` returns them for the union minibatch of ``count_total`` rows, at this policy's
        ``log_std`` (b2p_ppo_combine: fp64 sums from rank 0 on, so every rank that combines the same vectors gets the
        same bits)."""
        size = self.ppo_partial_size
        if partials.dtype != torch.float64 or not partials.is_contiguous() or partials.ndim != 2 or partials.shape[1] != size:
            raise ValueError('partials must be a contiguous float64 [ranks, %d] tensor' % size)
        if grad is None:
            grad = torch.empty(size - 4, dtype=torch.float32, device=self.device)
        if stats is None:
            stats = torch.empty(6, dtype=torch.float64, device=self.device)
        assert grad.dtype == torch.float32 and grad.numel() == size - 4 and grad.is_contiguous()
        assert stats.dtype == torch.float64 and stats.numel() == 6
        self._check(self.lib.b2p_ppo_combine(self.handle, _ptr(partials), int(partials.shape[0]), int(count_total),
                                             float(self.log_std), float(ent_coef), float(vf_coef), _ptr(grad), _ptr(stats),
                                             self._stream()))
        return grad, stats

    def close(self):
        if getattr(self, 'handle', None):
            torch.cuda.synchronize(self.device)
            self.lib.b2p_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:      # noqa: BLE001 (interpreter shutdown)
            pass


def obs_width(obs_dim):
    """W, the bf16 columns of a stored observation row for ``obs_dim`` (b2p_obs_width): 16 up to obs_dim 15, then 32,
    48, 64 and 80 (obs_dim 64..79).  Columns obs_dim..W-1 are zero; the last is the bias slot.  Raises outside the
    supported 1..79."""
    width = _lib.load().b2p_obs_width(int(obs_dim))
    if not width:
        raise _lib.B200EnvError('obs_dim %d is outside the policy kernels\' 1..79' % obs_dim)
    return width


def _tower_linears(tower):
    linears = [m for m in tower.modules() if isinstance(m, torch.nn.Linear)]
    if len(linears) != 3 or linears[0].out_features != 64 or linears[1].out_features != 64 \
            or linears[2].out_features != 1:
        raise ValueError('DevicePolicy needs an obs_dim -> 64 -> 64 -> 1 tanh tower')
    return linears


def reference_values(tower, obs, bf16=True):
    """The value tower (``SharedMlpPolicy.vf``) as the kernel evaluates it: ``reference_actions`` without the clip."""
    return reference_actions(tower, obs, low=-math.inf, high=math.inf, bf16=bf16)


def reference_actions(tower, obs, low=-4.0, high=6.0, bf16=True):
    """The same action head in torch, rounding to bf16 where the kernel does (operands of the two
    matmuls; fp32 accumulation, fp32 head): what the parity test holds the kernel to."""
    linears = [m for m in tower.modules() if isinstance(m, torch.nn.Linear)]
    rnd = (lambda t: t.to(torch.bfloat16).to(torch.float32)) if bf16 else (lambda t: t)
    x = rnd(obs.to(torch.float32))
    h1 = torch.tanh(x @ rnd(linears[0].weight.float()).t() + rnd(linears[0].bias.float()))
    h2 = torch.tanh(rnd(h1) @ rnd(linears[1].weight.float()).t() + rnd(linears[1].bias.float()))
    mean = h2 @ linears[2].weight.float().t() + linears[2].bias.float()
    return mean.squeeze(-1).clamp(low, high)


@torch.no_grad()
def device_policy_rollout(env, policy, steps, ring_only=True, on_step=None, use_graph=False):
    """``steps`` lock-step env steps driven by a ``DevicePolicy``; with ``ring_only`` the env never
    writes observation rows and the policy reads the rings (nothing but E rewards / flags / info rows
    and the action vector exists per step).  Returns (per-env reward sums [E], finished episodes).

    ``use_graph``: capture policy -> step -> bookkeeping for two steps (the pipeline's gradient buffers
    alternate) into one CUDA graph and replay it: no per-step Python or launch gaps.  Needs an even
    ``steps``, ``ring_only`` and no ``on_step``; the policy's noise seed then advances on the device."""
    actions = torch.empty(env.num_rows, dtype=torch.float32, device=env.device)
    returns = torch.zeros(env.num_envs, dtype=torch.float64, device=env.device)
    finished = torch.zeros((), dtype=torch.int64, device=env.device)
    obs = env.obs

    def one_step():
        if ring_only:
            policy.act_env(env, actions, seed=0 if use_graph else None)
        else:
            policy.act(obs, actions, seed=0 if use_graph else None)
        out = env.step(actions, ring_only=ring_only)
        returns.add_(out[1])
        finished.add_(out[2].sum())
        return out

    if use_graph:
        if steps % 2 or not ring_only or on_step is not None:
            raise ValueError('use_graph needs an even number of ring-only steps and no on_step hook')
        policy.use_seed_counter(True)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=env.device)
        side.wait_stream(torch.cuda.current_stream(env.device))
        with torch.cuda.stream(side):                      # steps 1 and 2 eagerly (lazy module loading outside the capture)
            for _ in range(2):
                one_step()
                policy.seed_counter.add_(1)
        torch.cuda.current_stream(env.device).wait_stream(side)
        torch.cuda.synchronize(env.device)
        with torch.cuda.graph(graph):
            for _ in range(2):
                one_step()
                policy.seed_counter.add_(1)
        for _ in range(steps // 2 - 1):
            graph.replay()
        torch.cuda.synchronize(env.device)
        policy.use_seed_counter(False)
        return returns, int(finished.item())
    for t in range(steps):
        obs, reward, done, info = one_step()
        if on_step is not None:
            on_step(t, obs, reward, done, info)
    return returns, int(finished.item())


def gae(values, rewards, dones, rows_per_env, gamma=0.99, lam=0.95, advantages=None, returns=None):
    """The PPO2 Runner's GAE on the device (b2p_gae): values [T+1, rows], rewards [T, E] float32, dones [T+1, E]
    uint8 (dones[t+1] = done of step t) -> (advantages, returns) [T, rows] float32; float64 recursion."""
    lib = _lib.load()
    T, rows = values.shape[0] - 1, values.shape[1]
    assert values.dtype == torch.float32 and rewards.dtype == torch.float32 and dones.dtype == torch.uint8
    assert all(t.is_contiguous() for t in (values, rewards, dones))
    assert rewards.shape == (T, rows // rows_per_env) and dones.shape == (T + 1, rows // rows_per_env)
    if advantages is None:
        advantages = torch.empty((T, rows), dtype=torch.float32, device=values.device)
    if returns is None:
        returns = torch.empty((T, rows), dtype=torch.float32, device=values.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(values.device).cuda_stream)
    if lib.b2p_gae(_ptr(values), _ptr(rewards), _ptr(dones), T, rows, int(rows_per_env), float(gamma), float(lam),
                   _ptr(advantages), _ptr(returns), stream):
        raise _lib.B200EnvError(lib.b2p_last_error(None).decode())
    return advantages, returns


class DeviceRolloutBuffer:
    """PPO rollout storage of ``n_steps`` steps of every agent row of ``env``, on its device, allocated once.

    Time-major: ``obs_bf16`` [T, rows, W] bf16 (the observation rows as the policy read them, W = ``obs_width(obs_dim)``,
    columns obs_dim..W-1 zero), ``actions_raw`` / ``neglogp`` / ``advantages`` / ``returns`` [T, rows] float32,
    ``values`` [T+1, rows] float32 (``values[T]`` = value of the observation after the last step),
    ``rewards`` [T, E] float32 and ``dones`` [T+1, E] uint8 (per env; env = row // P; ``dones[0]`` = the
    flags at the rollout's first observation, ``dones[t+1]`` = done of step t).  stable-baselines'
    ``swap_and_flatten`` order is ``.transpose(0, 1)`` of these arrays; PPO samples random minibatches of
    flat indices, so no copy is needed.

    ``actions`` [rows] float32 holds the clipped actions of the current step (what the env steps with).

    Memory: 2W + 20 bytes per agent row and step (the observation row + 5 x 4), plus 8 bytes per agent row (the
    last value slot and ``actions``).  That is 52 B at W = 16, e.g. 10.8 GB per step for the 2.08e8 rows of 4096
    envs of MLP 784-64-10 (88 GB for n_steps = 8), and 180 B at max_history 25 (W = 80: 37.5 GB per step, so
    n_steps = 2 fits a 180 GB card beside the env's rings and 8 does not); the constructor checks it against the
    device's free memory."""

    def __init__(self, env, n_steps):
        self.n_steps = T = int(n_steps)
        if T < 1:
            raise ValueError('n_steps must be >= 1')
        rows, E, dev = env.num_rows, env.num_envs, env.device
        self.rows_per_env = env.num_params
        self.obs_width = W = obs_width(env.obs_dim)
        self.bytes_per_row_step = 2 * W + 5 * 4
        need = rows * (self.bytes_per_row_step * T + 8) + E * (5 * T + 1)
        free, _ = torch.cuda.mem_get_info(dev)
        if need > free:
            raise MemoryError('DeviceRolloutBuffer: n_steps = %d needs %.2f GB (%d rows x %d B per step) but %s has '
                              '%.2f GB free; use fewer steps per rollout' % (T, need / 1e9, rows, self.bytes_per_row_step,
                                                                            dev, free / 1e9))
        f32 = dict(dtype=torch.float32, device=dev)
        self.obs_bf16 = torch.empty((T, rows, W), dtype=torch.bfloat16, device=dev)
        self.actions_raw = torch.empty((T, rows), **f32)
        self.values = torch.empty((T + 1, rows), **f32)
        self.neglogp = torch.empty((T, rows), **f32)
        self.advantages = torch.empty((T, rows), **f32)
        self.returns = torch.empty((T, rows), **f32)
        self.rewards = torch.zeros((T, E), **f32)
        self.dones = torch.zeros((T + 1, E), dtype=torch.uint8, device=dev)
        self.actions = torch.empty(rows, **f32)

    def reset(self):
        """Forget the carried done flags (call after ``env.reset()``): the next rollout starts with dones[0] = 0."""
        self.dones.zero_()


@torch.no_grad()
def device_ppo_rollout(env, policy, buffer, gamma=0.99, lam=0.95, ring_only=True, on_step=None, seed=None):
    """One PPO2 ``Runner.run`` on the device: ``buffer.n_steps`` times ``model.step`` (``policy.step`` into the
    buffer) then the env step with the clipped actions, then ``model.value`` of the last observation and GAE.
    ``ring_only``: the policy reads the env's rings and the env writes no observation rows (MultiOptLRs, large
    problems); otherwise the policy reads ``env.obs``, which must hold the current observation (the only path
    of the small problems).  ``on_step(t, obs, reward, done, info)`` as in ``device_rollout``.  The done flags
    of the last step become ``dones[0]`` of the next rollout; after ``env.reset()`` call ``buffer.reset()`` so that
    they are zero, as the Runner starts.  ``seed``: None draws the exploration noise of launch t from the policy's
    call counter; otherwise launch t draws noise seed ``splitmix64(seed, t)``, so a rollout's noise depends on the
    seed alone.  Returns (buffer, finished episodes)."""
    T = buffer.n_steps
    assert buffer.actions.numel() == env.num_rows and buffer.rewards.shape[1] == env.num_envs
    if not policy.has_value:
        raise ValueError('device_ppo_rollout needs a policy with a value tower (set_value_weights)')
    finished = torch.zeros((), dtype=torch.int64, device=env.device)
    buffer.dones[0].copy_(buffer.dones[T])
    for t in range(T):
        source = env if ring_only else env.obs
        noise_seed = None if seed is None else splitmix64(seed, t)
        policy._launch(source, policy._seed(noise_seed), buffer.actions, buffer.actions_raw[t], buffer.values[t],
                       buffer.neglogp[t], buffer.obs_bf16[t])
        obs, reward, done, info = env.step(buffer.actions, ring_only=ring_only)
        buffer.rewards[t].copy_(reward)
        buffer.dones[t + 1].copy_(done)
        finished.add_(done.sum())
        if on_step is not None:
            on_step(t, obs, reward, done, info)
    policy.value(env if ring_only else env.obs, out=buffer.values[T])
    gae(buffer.values, buffer.rewards, buffer.dones, buffer.rows_per_env, gamma, lam, buffer.advantages, buffer.returns)
    return buffer, int(finished.item())


# ------------------------------------------------------------------ PPO updates
def _ppo_batch(buffer):
    T, rows = buffer.actions_raw.shape
    return _lib.PpoBatch(buffer.obs_bf16.data_ptr(), buffer.actions_raw.data_ptr(), buffer.neglogp.data_ptr(),
                         buffer.values.data_ptr(), buffer.returns.data_ptr(), T, rows)


def _check_global(code):
    if code:
        raise _lib.B200EnvError(_lib.load().b2p_last_error(None).decode())


def tanh_bf16_table(device='cuda'):
    """float32 [65536]: the bf16 tanh the kernels evaluate in the bf16 tanh modes, indexed by the input's bf16 bit
    pattern (b2p_tanh_table) -- for references that reproduce those modes exactly."""
    lib = _lib.load()
    out = torch.empty(65536, dtype=torch.float32, device=device)
    _check_global(lib.b2p_tanh_table(_ptr(out), ctypes.c_void_p(torch.cuda.current_stream(out.device).cuda_stream)))
    return out


def ppo_minibatch_indices(n, key, begin, count, out=None, device='cuda'):
    """The flat sample indices (t * rows + row) at positions [begin, begin + count) of the keyed permutation of
    [0, n) that ``ppo_grad`` reads (b2p_ppo_indices) -> int64 [count] on the device."""
    lib = _lib.load()
    if out is None:
        out = torch.empty(int(count), dtype=torch.int64, device=device)
    assert out.dtype == torch.int64 and out.is_contiguous() and out.numel() == count
    stream = ctypes.c_void_p(torch.cuda.current_stream(out.device).cuda_stream)
    _check_global(lib.b2p_ppo_indices(int(key) & (2 ** 64 - 1), int(n), int(begin), int(count), _ptr(out), stream))
    return out


def ppo_adv_stats(buffer, key, mb_size):
    """Mean and population std (float64 sums) of returns - values over every minibatch of one epoch's permutation
    ``key`` -> float64 [T * rows / mb_size, 2] on the device (b2p_ppo_adv_stats)."""
    lib = _lib.load()
    T, rows = buffer.actions_raw.shape
    n = T * rows
    if mb_size < 1 or n % mb_size:
        raise ValueError('the %d samples of the buffer do not split into minibatches of %d' % (n, mb_size))
    dev = buffer.returns.device
    stats = torch.empty((n // mb_size, 2), dtype=torch.float64, device=dev)
    ws = torch.empty(max(1, lib.b2p_ppo_adv_stats_workspace_size(n, mb_size)), dtype=torch.uint8, device=dev)
    batch = _ppo_batch(buffer)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _check_global(lib.b2p_ppo_adv_stats(ctypes.byref(batch), int(key) & (2 ** 64 - 1), int(mb_size), _ptr(stats),
                                        _ptr(ws), stream))
    return stats


def ppo_adv_moments(buffer, key, mb_size):
    """This shard's advantage moments of every minibatch of one epoch's permutation ``key`` (b2p_ppo_adv_moments) ->
    float64 [T * rows / mb_size, 4] on the device: count, shift K (the advantage at the minibatch's first position),
    sum(A - K) and sum((A - K)^2), fp64 sums in the order of ``ppo_adv_stats``."""
    lib = _lib.load()
    T, rows = buffer.actions_raw.shape
    n = T * rows
    if mb_size < 1 or n % mb_size:
        raise ValueError('the %d samples of the buffer do not split into minibatches of %d' % (n, mb_size))
    dev = buffer.returns.device
    moments = torch.empty((n // mb_size, 4), dtype=torch.float64, device=dev)
    ws = torch.empty(max(1, lib.b2p_ppo_adv_stats_workspace_size(n, mb_size)), dtype=torch.uint8, device=dev)
    batch = _ppo_batch(buffer)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _check_global(lib.b2p_ppo_adv_moments(ctypes.byref(batch), int(key) & (2 ** 64 - 1), int(mb_size), _ptr(moments),
                                          _ptr(ws), stream))
    return moments


def ppo_adv_combine(moments):
    """``moments`` float64 [ranks, nmb, 4], the shards' ``ppo_adv_moments`` in rank order -> float64 [nmb, 2]: mean and
    population std of the advantages of every union minibatch (b2p_ppo_adv_combine; one rank = ``ppo_adv_stats``)."""
    lib = _lib.load()
    if moments.dtype != torch.float64 or not moments.is_contiguous() or moments.ndim != 3 or moments.shape[2] != 4:
        raise ValueError('moments must be a contiguous float64 [ranks, nmb, 4] tensor')
    stats = torch.empty((moments.shape[1], 2), dtype=torch.float64, device=moments.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(moments.device).cuda_stream)
    _check_global(lib.b2p_ppo_adv_combine(_ptr(moments), int(moments.shape[0]), int(moments.shape[1]), _ptr(stats), stream))
    return stats


def _mix64(z):
    z &= 2 ** 64 - 1
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2 ** 64 - 1)
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2 ** 64 - 1)
    return z ^ (z >> 31)


def rank_epoch_key(seed, epoch, rank):
    """The permutation key of rank ``rank``'s shard in epoch ``epoch`` of a data-parallel update seeded ``seed``:
    ``epoch_key(seed, epoch)`` on rank 0, so that a one-rank update is the single-GPU one, and on rank r > 0 the
    splitmix64 finaliser of that key + r * 0x9E3779B97F4A7C15."""
    key = epoch_key(seed, epoch)
    return key if int(rank) == 0 else _mix64(key + int(rank) * 0x9E3779B97F4A7C15)


def splitmix64(seed, index):
    """The splitmix64 finaliser of seed * 0x9E3779B97F4A7C15 + index + 1 (mod 2^64): the ``index``-th value derived
    from ``seed``."""
    return _mix64(int(seed) * 0x9E3779B97F4A7C15 + int(index) + 1)


def epoch_key(seed, epoch):
    """The permutation key of epoch ``epoch`` of an update seeded ``seed`` (``splitmix64(seed, epoch)``)."""
    return splitmix64(seed, epoch)


def _model_params(model):
    """The parameters in the order of ``ppo_grad``'s flat gradient: pi (w1, b1, w2, b2, w3, b3), vf (...), log_std."""
    params = []
    for tower in (model.pi, model.vf):
        for lin in _tower_linears(tower):
            params += [lin.weight, lin.bias]
    return params + [model.log_std]


def load_model(policy, model):
    """Hand ``model``'s (a ``SharedMlpPolicy``) towers and ``log_std`` to ``policy``."""
    policy.set_weights(*[t for lin in _tower_linears(model.pi) for t in (lin.weight, lin.bias)])
    policy.set_value_weights(*[t for lin in _tower_linears(model.vf) for t in (lin.weight, lin.bias)])
    policy.set_log_std(model.log_std.detach())


def device_ppo_update(model, policy, buffer, optimizer, n_epochs=4, n_minibatches=4, cliprange=0.2, cliprange_vf=None,
                      ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5, seed=None, group=None):
    """stable-baselines 2 ``PPO2.learn``'s inner loop over a filled ``DeviceRolloutBuffer``: ``n_epochs`` passes, each
    over a fresh permutation of the T * rows samples cut into ``n_minibatches`` minibatches.  Per minibatch: ``model``'s
    towers and ``log_std`` go to ``policy``, ``policy.ppo_grad`` computes the gradient of PPO2's loss, it is copied into
    the parameters' ``.grad``, then ``clip_grad_norm_(max_grad_norm)`` (skipped for None, as in PPO2) and
    ``optimizer.step()``.  ``model`` (a ``SharedMlpPolicy``) stays the fp32 master copy; the optimizer is the
    caller's -- PPO2's is Adam with eps = 1e-5, i.e. ``torch.optim.Adam(model.parameters(), lr, eps=1e-5)`` (torch places eps outside the square root like TF's
    Adam but without TF's bias-corrected epsilon, so parity with TF is not pinned).  ``seed`` picks the permutations
    (None: drawn from torch's generator).  On return ``policy`` holds the trained weights and ``log_std``.  Returns
    the statistics averaged over minibatches (pg_loss, vf_loss, entropy, approxkl, clipfrac, loss) as float64 numpy
    [6], with one host synchronisation.

    ``group``: a ``torch.distributed`` process group whose every rank holds the rollout of its own env shard (one GPU
    per rank, e.g. under ``torchrun``); None = this GPU alone.  The ranks then train one policy on the union of their
    samples, as PPO2 on the whole env batch with minibatches stratified by rank:

    - rank 0's ``seed`` is used on every rank; rank r permutes its own N_r = T * rows_r samples with
      ``rank_epoch_key(seed, epoch, r)``, and minibatch m is positions [m N_r / n_minibatches, (m + 1) N_r / n_minibatches)
      of every rank, so its size n_m is the sum of the ranks' shares (every N_r must be a multiple of n_minibatches);
    - the advantages are normalised with the mean and std of the union minibatch (``ppo_adv_moments``, all-gather,
      ``ppo_adv_combine``), and gradient and statistics are means over n_m (``ppo_grad_partial``, all-gather,
      ``ppo_combine``);
    - the combine sums the ranks' fp64 vectors in rank order, so every rank applies the same gradient, clip and
      optimizer step bit for bit and the models stay identical without a weight broadcast.

    One all-gather first checks that the ranks agree on T, the observation width, obs_dim, n_epochs and n_minibatches;
    on a mismatch every rank raises the same ValueError.  Per minibatch the exchange is one float64 vector of
    ``policy.ppo_partial_size`` per rank (84 KB at obs_dim 15).  Returns the statistics of the union minibatches,
    the same on every rank."""
    if group is not None:
        return _device_ppo_update_dist(model, policy, buffer, optimizer, n_epochs, n_minibatches, cliprange, cliprange_vf,
                                       ent_coef, vf_coef, max_grad_norm, seed, group)
    T, rows = buffer.actions_raw.shape
    n = T * rows
    if n % n_minibatches:
        raise ValueError('T * rows = %d is not a multiple of n_minibatches = %d' % (n, n_minibatches))
    mb = n // n_minibatches
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    params = _model_params(model)
    total = torch.zeros(6, dtype=torch.float64, device=policy.device)
    grad = stats = None
    for epoch in range(n_epochs):
        key = epoch_key(seed, epoch)
        adv = ppo_adv_stats(buffer, key, mb)
        for m in range(n_minibatches):
            load_model(policy, model)
            grad, stats = policy.ppo_grad(buffer, key, m * mb, mb, adv[m], cliprange, cliprange_vf, ent_coef, vf_coef,
                                          grad, stats)
            _set_grads(params, grad)
            if max_grad_norm is not None:
                torch.nn.utils.clip_grad_norm_(params, max_grad_norm)
            optimizer.step()
            total += stats
    load_model(policy, model)
    return (total / (n_epochs * n_minibatches)).cpu().numpy()


def _set_grads(params, grad):
    offset = 0
    for p in params:
        g = grad[offset:offset + p.numel()].view_as(p)
        if p.grad is None:
            p.grad = g.clone()
        else:
            p.grad.copy_(g)
        offset += p.numel()


def _check_rank_table(table, n_minibatches):
    """The all-gathered [T, buffer width, obs_width, obs_dim, T * rows, n_epochs, n_minibatches, seed] of every rank ->
    (rank 0's seed, n_m = the size of a union minibatch).  Every rank runs it on the same table, so all raise the same
    ValueError or none does."""
    for col, what in ((0, 'T (n_steps)'), (2, 'the observation width'), (3, 'obs_dim'), (5, 'n_epochs'),
                      (6, 'n_minibatches')):
        values = [row[col] for row in table]
        if len(set(values)) > 1:
            raise ValueError('data-parallel PPO: the ranks disagree on %s: %s' % (what, values))
    bad = [r for r, row in enumerate(table) if row[1] != row[2]]
    if bad:
        raise ValueError('data-parallel PPO: the rollout rows of rank(s) %s are not the policy\'s obs_width wide' % bad)
    bad = [r for r, row in enumerate(table) if n_minibatches < 1 or row[4] % n_minibatches]
    if bad:
        raise ValueError('data-parallel PPO: T * rows = %s of rank(s) %s is not a multiple of n_minibatches = %d'
                         % ([table[r][4] for r in bad], bad, n_minibatches))
    return table[0][7] & (2 ** 64 - 1), sum(row[4] // n_minibatches for row in table)


def _device_ppo_update_dist(model, policy, buffer, optimizer, n_epochs, n_minibatches, cliprange, cliprange_vf, ent_coef,
                            vf_coef, max_grad_norm, seed, group):
    """``device_ppo_update`` over the ranks of ``group`` (see there)."""
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = policy.device
    T, rows = buffer.actions_raw.shape
    n = T * rows
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    seed = int(seed) & (2 ** 64 - 1)
    mine = torch.tensor([T, buffer.obs_bf16.shape[-1], policy.obs_width, policy.obs_dim, n, n_epochs, n_minibatches,
                         seed - 2 ** 64 if seed >= 2 ** 63 else seed], dtype=torch.int64, device=dev)
    table = torch.empty((world, mine.numel()), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(table, mine, group=group)
    seed, count_total = _check_rank_table(table.cpu().tolist(), n_minibatches)
    mb = n // n_minibatches
    params = _model_params(model)
    f64 = dict(dtype=torch.float64, device=dev)
    partial = torch.empty(policy.ppo_partial_size, **f64)
    partials = torch.empty((world, partial.numel()), **f64)
    moments_all = torch.empty((world, n_minibatches, 4), **f64)
    total = torch.zeros(6, **f64)
    grad = stats = None
    for epoch in range(n_epochs):
        key = rank_epoch_key(seed, epoch, rank)
        dist.all_gather_into_tensor(moments_all, ppo_adv_moments(buffer, key, mb), group=group)
        adv = ppo_adv_combine(moments_all)
        for m in range(n_minibatches):
            load_model(policy, model)
            policy.ppo_grad_partial(buffer, key, m * mb, mb, count_total, adv[m], cliprange, cliprange_vf, ent_coef,
                                    vf_coef, partial)
            dist.all_gather_into_tensor(partials, partial, group=group)
            grad, stats = policy.ppo_combine(partials, count_total, ent_coef, vf_coef, grad, stats)
            _set_grads(params, grad)
            if max_grad_norm is not None:
                torch.nn.utils.clip_grad_norm_(params, max_grad_norm)
            optimizer.step()
            total += stats
    load_model(policy, model)
    return (total / (n_epochs * n_minibatches)).cpu().numpy()
