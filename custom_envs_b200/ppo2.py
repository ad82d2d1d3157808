"""stable-baselines' ``PPO2`` on the device: ``from custom_envs_b200.ppo2 import PPO2, MlpPolicy`` replaces
``from stable_baselines import PPO2`` and ``from stable_baselines.common.policies import MlpPolicy`` in the reference's
scripts (run_multiagent_exp_single.py, search_optimize_hyperparam.py, play_optimize.py, eval_multiexp.py).

The surface follows stable-baselines 2.10 (constructor, ``learn`` with its timestep accounting, schedules and callbacks,
``predict``, ``get_parameters`` / ``load_parameters``, ``save`` / ``load``).  Every update is one ``device_ppo_rollout``
and one ``device_ppo_update`` over the fused env batch, so the [sum(P), obs_dim] observation matrix never goes to the
host; one float64 [E, 18] array per step does (rewards, done flags and infos, 0.5 MB at 4096 envs), which feeds the
Monitors of an ``OptVecEnv`` and the callbacks.

The parameter names, their order and layouts, the initialisation, TF's Adam and the zip layout of ``save`` are restated
from the stable-baselines 2.10 source; they are not checked against it (stable-baselines is not a dependency)."""
import io
import json
import math
import time
import zipfile
from collections import OrderedDict, deque

import numpy as np
import torch

from custom_envs_b200._lib import B200EnvError
from custom_envs_b200.batched_env import BatchedOptEnv
from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer, _tower_linears,
                                                      device_ppo_rollout, device_ppo_update, load_model, splitmix64)
from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy
from custom_envs_b200.vectorize.optvecenv import LazyInfos, OptVecEnv

HIDDEN = 64
LOSS_NAMES = ('policy_loss', 'value_loss', 'policy_entropy', 'approxkl', 'clipfrac', 'loss')


class MlpPolicy:
    """Marker for stable-baselines' ``MlpPolicy``: two tanh layers of 64 for the action mean and two for the value
    (``net_arch=[dict(pi=[64, 64], vf=[64, 64])]``), a state-independent ``log_std``.  The only policy ``PPO2`` takes."""


# ------------------------------------------------------------------ stable-baselines' parameter names
# MlpPolicy's TF variables in creation order: mlp_extractor builds pi_fc{i} and vf_fc{i} layer by layer, then the
# value head 'vf', then DiagGaussianProbabilityDistributionType builds 'pi', 'pi/logstd' and the unused 'q' head.
# Entries: (name, torch tower, index of the Linear in the tower, 'w' [in, out] / 'b' [out]).
PARAMETER_MAP = (
    ('model/pi_fc0/w:0', 'pi', 0, 'w'), ('model/pi_fc0/b:0', 'pi', 0, 'b'),
    ('model/vf_fc0/w:0', 'vf', 0, 'w'), ('model/vf_fc0/b:0', 'vf', 0, 'b'),
    ('model/pi_fc1/w:0', 'pi', 1, 'w'), ('model/pi_fc1/b:0', 'pi', 1, 'b'),
    ('model/vf_fc1/w:0', 'vf', 1, 'w'), ('model/vf_fc1/b:0', 'vf', 1, 'b'),
    ('model/vf/w:0', 'vf', 2, 'w'), ('model/vf/b:0', 'vf', 2, 'b'),
    ('model/pi/w:0', 'pi', 2, 'w'), ('model/pi/b:0', 'pi', 2, 'b'),
    ('model/pi/logstd:0', 'log_std', None, None),
    ('model/q/w:0', 'q', None, 'w'), ('model/q/b:0', 'q', None, 'b'),
)


def sb_parameters(model):
    """``SharedMlpPolicy`` -> OrderedDict of float32 numpy arrays in stable-baselines' names and TF layouts; the 'q'
    head, which PPO does not use, is zeros."""
    out = OrderedDict()
    for name, tower, layer, kind in PARAMETER_MAP:
        if tower == 'log_std':
            value = model.log_std.detach().reshape(1, 1)
        elif tower == 'q':
            value = torch.zeros((HIDDEN, 1) if kind == 'w' else (1,))
        else:
            lin = _tower_linears(getattr(model, tower))[layer]
            value = lin.weight.detach().t() if kind == 'w' else lin.bias.detach()
        out[name] = np.ascontiguousarray(value.float().cpu().numpy())
    return out


@torch.no_grad()
def load_sb_parameters(model, params, exact_match=True):
    """Copy ``params`` (stable-baselines' names -> arrays, as ``sb_parameters`` gives them) into ``model``.
    ``exact_match``: the names must be exactly those of ``PARAMETER_MAP``; otherwise unknown names are ignored and
    missing ones keep their values.  Raises ValueError on a missing name or a wrong shape."""
    names = [entry[0] for entry in PARAMETER_MAP]
    if exact_match and set(params) != set(names):
        raise ValueError('parameters do not match MlpPolicy\'s: missing %s, unexpected %s'
                         % (sorted(set(names) - set(params)), sorted(set(params) - set(names))))
    want = sb_parameters(model)
    for name, tower, layer, kind in PARAMETER_MAP:
        if name not in params:
            continue
        value = np.asarray(params[name], dtype=np.float32)
        if value.shape != want[name].shape:
            raise ValueError('%s has shape %s, MlpPolicy\'s is %s' % (name, value.shape, want[name].shape))
        if tower == 'q':
            continue
        if tower == 'log_std':
            model.log_std.copy_(torch.as_tensor(value.reshape(())))
            continue
        lin = _tower_linears(getattr(model, tower))[layer]
        target = lin.weight if kind == 'w' else lin.bias
        source = torch.as_tensor(value)
        target.copy_(source.t() if kind == 'w' else source)


@torch.no_grad()
def init_like_stable_baselines(model, generator):
    """stable-baselines' MlpPolicy initialisation, drawn from the CPU ``generator``: orthogonal weights with gain
    sqrt(2) for the hidden layers, 0.01 for 'pi' and 1 for 'vf', zero biases, log_std = 0.  The distribution is
    TF's ortho_init; TF's random stream is not reproduced."""
    for tower, head_gain in ((model.pi, 0.01), (model.vf, 1.0)):
        linears = _tower_linears(tower)
        for i, lin in enumerate(linears):
            weight = torch.empty(lin.weight.shape)
            torch.nn.init.orthogonal_(weight, gain=head_gain if i == len(linears) - 1 else math.sqrt(2),
                                      generator=generator)
            lin.weight.copy_(weight)
            lin.bias.zero_()
    model.log_std.zero_()


# ------------------------------------------------------------------ PPO2's arithmetic
def tf_adam(params, lr, eps=1e-5):
    """``torch.optim.Adam(eps=1e-5)`` stepping as TF's AdamOptimizer: TF computes lr * sqrt(1 - b2^t) / (1 - b1^t) *
    m / (sqrt(v) + eps), which is torch's update with eps / sqrt(1 - b2^t) in place of eps.  A step pre-hook sets that
    eps before step t (equal in exact arithmetic; rounding may differ)."""
    optimizer = torch.optim.Adam(params, lr=lr, eps=eps)

    def set_eps(opt, args, kwargs):
        for group in opt.param_groups:
            state = opt.state.get(group['params'][0], {})
            t = int(state['step']) + 1 if 'step' in state else 1
            group['eps'] = eps / math.sqrt(1.0 - group['betas'][1] ** t)

    optimizer.register_step_pre_hook(set_eps)
    return optimizer


def schedule(value):
    """stable-baselines' ``get_schedule_fn``: a callable of ``frac`` stays, a number becomes a constant."""
    return value if callable(value) else (lambda frac: value)


def update_plan(total_timesteps, n_steps, n_envs, nminibatches):
    """(n_batch, n_updates) of ``PPO2.learn``, with its check that ``nminibatches`` divides n_batch."""
    n_batch = int(n_steps) * int(n_envs)
    assert n_batch % nminibatches == 0, (
        'The number of minibatches (`nminibatches`) is not a factor of the total number of samples collected per '
        'rollout (`n_batch`), some samples won\'t be used.')
    return n_batch, int(total_timesteps) // n_batch


def frac_of(update, n_updates):
    """``frac = 1 - (update - 1) / n_updates`` of update 1..n_updates: the argument of the schedules."""
    return 1.0 - (update - 1.0) / n_updates


def update_seeds(seed, update):
    """(rollout noise seed, minibatch permutation seed) of the ``update``-th update (counted from 1 over the model's
    life) of a model seeded ``seed``."""
    return splitmix64(seed, 2 * update), splitmix64(seed, 2 * update + 1)


@torch.no_grad()
def explained_variance(values, returns, chunk=1 << 24):
    """``1 - var(returns - values) / var(returns)`` over [T, rows] buffers in float64, chunk by chunk (nan if
    var(returns) is 0, as stable-baselines' ``explained_variance``)."""
    sums = torch.zeros(4, dtype=torch.float64, device=returns.device)
    flat_r, flat_v = returns.reshape(-1), values.reshape(-1)
    for lo in range(0, flat_r.numel(), chunk):
        r = flat_r[lo:lo + chunk].double()
        d = r - flat_v[lo:lo + chunk].double()
        sums += torch.stack([r.sum(), (r * r).sum(), d.sum(), (d * d).sum()])
    n = flat_r.numel()
    s_r, ss_r, s_d, ss_d = sums.tolist()
    var_r = ss_r / n - (s_r / n) ** 2
    var_d = ss_d / n - (s_d / n) ** 2
    return float('nan') if var_r == 0 else 1.0 - var_d / var_r


class _StopTraining(Exception):
    def __init__(self, step):
        super().__init__(step)
        self.step = step


class _Callbacks:
    """stable-baselines 2.10's callback protocol: None, a legacy function ``callback(locals_, globals_)`` called after
    every env step, an object with the ``on_*`` hooks, or a list of either."""

    def __init__(self, callback, model):
        items = callback if isinstance(callback, (list, tuple)) else ([] if callback is None else [callback])
        self.items = items
        self.locals = {}
        self.globals = {}
        for item in items:
            if hasattr(item, 'init_callback'):
                item.init_callback(model)

    def _hooks(self, name):
        return [getattr(item, name) for item in self.items if hasattr(item, name)]

    def on_training_start(self, locals_, globals_):
        self.locals, self.globals = locals_, globals_
        for hook in self._hooks('on_training_start'):
            hook(locals_, globals_)

    def on_rollout_start(self):
        for hook in self._hooks('on_rollout_start'):
            hook()

    def on_step(self, step_locals):
        """False if any callback asks to stop."""
        self.locals.update(step_locals)
        keep = True
        for item in self.items:
            if hasattr(item, 'on_step'):
                if hasattr(item, 'update_locals'):
                    item.update_locals(step_locals)
                keep = item.on_step() is not False and keep
            elif callable(item):
                keep = item(self.locals, self.globals) is not False and keep
        return keep

    def on_rollout_end(self):
        for hook in self._hooks('on_rollout_end'):
            hook()

    def on_training_end(self):
        for hook in self._hooks('on_training_end'):
            hook()


# ------------------------------------------------------------------ PPO2
_HYPERPARAMETERS = ('gamma', 'n_steps', 'ent_coef', 'learning_rate', 'vf_coef', 'max_grad_norm', 'lam', 'nminibatches',
                    'noptepochs', 'cliprange', 'cliprange_vf', 'verbose', 'seed', 'policy_kwargs')


def _check_policy(policy, policy_kwargs):
    if policy is not MlpPolicy and policy != 'MlpPolicy':
        raise ValueError('PPO2 on the device supports MlpPolicy only, not %r' % (policy,))
    for key, value in (policy_kwargs or {}).items():
        default = value == [dict(pi=[HIDDEN, HIDDEN], vf=[HIDDEN, HIDDEN])] or value == [dict(vf=[HIDDEN, HIDDEN],
                                                                                               pi=[HIDDEN, HIDDEN])]
        if key != 'net_arch' or not default:
            raise ValueError('unsupported policy_kwargs item %r=%r: only the default net_arch [dict(pi=[64, 64], '
                             'vf=[64, 64])] is supported' % (key, value))


class PPO2:
    """stable-baselines 2.10's ``PPO2(policy, env, ...)`` over the fused env batch on the device.

    ``policy``: ``MlpPolicy`` or ``'MlpPolicy'``; ``policy_kwargs`` may only restate its default ``net_arch``.
    ``env``: an ``OptVecEnv`` on its device-backed (fused) path, or a ``BatchedOptEnv`` (e.g. a rank's shard under
    ``torchrun``, with ``group``).  ``tensorboard_log``, ``tb_log_name``, ``full_tensorboard_log`` and
    ``n_cpu_tf_sess`` are accepted and ignored.

    The fp32 master copy of the weights is ``self.model`` (a ``SharedMlpPolicy``, initialised as stable-baselines
    initialises MlpPolicy from a ``torch.Generator`` seeded with ``seed``), the kernels run ``self.device_policy`` (a
    ``DevicePolicy`` built from it), the rollout lives in ``self.buffer`` (a ``DeviceRolloutBuffer``; an ``n_steps``
    beyond free memory raises its MemoryError) and the optimizer is ``tf_adam``.

    ``group``: a ``torch.distributed`` process group whose every rank holds its ``BatchedOptEnv`` shard.  Rank 0's seed
    is used on every rank (so the initial model is the same everywhere), ``num_envs`` counts the rows of all ranks,
    the shard draws the noise of its global rows and ``device_ppo_update`` trains on the union of the ranks' samples.
    ``save`` writes on rank 0 only."""

    def __init__(self, policy, env, gamma=0.99, n_steps=128, ent_coef=0.01, learning_rate=2.5e-4, vf_coef=0.5,
                 max_grad_norm=0.5, lam=0.95, nminibatches=4, noptepochs=4, cliprange=0.2, cliprange_vf=None,
                 verbose=0, tensorboard_log=None, _init_setup_model=True, policy_kwargs=None,
                 full_tensorboard_log=False, seed=None, n_cpu_tf_sess=None, group=None):
        _check_policy(policy, policy_kwargs)
        self.policy = MlpPolicy
        self.policy_kwargs = dict(policy_kwargs or {})
        self.gamma, self.n_steps, self.ent_coef, self.learning_rate = gamma, int(n_steps), ent_coef, learning_rate
        self.vf_coef, self.max_grad_norm, self.lam = vf_coef, max_grad_norm, lam
        self.nminibatches, self.noptepochs = int(nminibatches), int(noptepochs)
        self.cliprange, self.cliprange_vf = cliprange, cliprange_vf
        self.verbose, self.seed, self.group = verbose, seed, group
        self.tensorboard_log, self.full_tensorboard_log, self.n_cpu_tf_sess = tensorboard_log, full_tensorboard_log, \
            n_cpu_tf_sess
        self.num_timesteps = 0
        self.ep_info_buf = deque(maxlen=100)
        self.env = self.batch = None
        self.model = self.device_policy = self.optimizer = self.buffer = None
        self.obs_dim, self.n_envs = None, None
        self.device = torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else None
        self.action_low, self.action_high, self.action_shape = -1e3, 1e4, (1,)   # MultiOptLRs: get_action_space_optlrs(2)
        self._updates_done = 0
        self._started = False
        self._ring_only = None
        if env is not None:
            self.set_env(env)
        if _init_setup_model:
            if env is None:
                raise ValueError('PPO2 needs an env to set up its model (or _init_setup_model=False)')
            self.setup_model()

    # -------------------------------------------------------------- env and model
    def set_env(self, env):
        """Attach ``env`` (see the class docstring); the next ``learn`` resets it."""
        if isinstance(env, OptVecEnv):
            if not env.is_device_backed:
                raise ValueError('PPO2 on the device needs an OptVecEnv whose envs are fused into one device batch; '
                                 'this one runs on the host fallback, which has no device batch to drive')
            batch = env._impl.env
            space = env.action_space
            self.action_low, self.action_high = float(np.min(space.low)), float(np.max(space.high))
            self.action_shape = tuple(space.shape)
        elif isinstance(env, BatchedOptEnv):
            batch = env
        else:
            raise ValueError('PPO2 on the device takes a device-backed OptVecEnv or a BatchedOptEnv, not %s'
                             % type(env).__name__)
        if self.obs_dim is not None and self.obs_dim != batch.obs_dim:
            raise ValueError('the env\'s obs_dim %d is not the model\'s %d' % (batch.obs_dim, self.obs_dim))
        if self.group is not None and not isinstance(env, BatchedOptEnv):
            raise ValueError('PPO2 with a process group takes each rank\'s BatchedOptEnv shard')
        self.env, self.batch = env, batch
        self.obs_dim, self.device = batch.obs_dim, batch.device
        self.n_envs = batch.num_rows
        self._started = False
        if self.group is not None:
            import torch.distributed as dist
            rows = torch.tensor([batch.num_rows], dtype=torch.int64, device=self.device)
            dist.all_reduce(rows, group=self.group)
            self.n_envs = int(rows.item())
        if self.device_policy is not None:
            self._attach_policy()
        self.buffer = None if self.model is None else DeviceRolloutBuffer(batch, self.n_steps)

    def _base_seed(self):
        """The seed everything is drawn from: ``seed``, or one draw of torch's generator; rank 0's under a group."""
        seed = self.seed if self.seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
        seed = int(seed) & (2 ** 63 - 1)
        if self.group is not None:
            import torch.distributed as dist
            value = torch.tensor([seed], dtype=torch.int64, device=self.device)
            dist.broadcast(value, src=dist.get_global_rank(self.group, 0), group=self.group)
            seed = int(value.item())
        return seed

    def setup_model(self):
        if self.obs_dim is None:
            raise ValueError('PPO2.setup_model needs an env or a known obs_dim')
        self._seed_base = self._base_seed()
        model = SharedMlpPolicy(self.obs_dim)
        init_like_stable_baselines(model, torch.Generator().manual_seed(self._seed_base))
        self.model = model.to(self.device)
        self.device_policy = DevicePolicy.from_torch(self.model, low=self.action_low, high=self.action_high)
        self.optimizer = tf_adam(self.model.parameters(), schedule(self.learning_rate)(1.0))
        if self.batch is not None:
            self._attach_policy()
            self.buffer = DeviceRolloutBuffer(self.batch, self.n_steps)

    def _attach_policy(self):
        if self.group is not None:
            self.device_policy.set_row_base(self.batch.env_base * self.batch.num_params)

    def get_env(self):
        return self.env

    @property
    def n_batch(self):
        return self.n_steps * self.n_envs

    def _start(self):
        """What stable-baselines' Runner does when it is created: reset the env, start with zero done flags.  Also
        picks the rollout's source: the env's adjusted-history rings where it keeps them (MultiOptLRs on the
        large-problem pipeline; ``b2p_step_env`` refuses other envs before it launches anything), else its dense rows."""
        self.env.reset()
        self.buffer.reset()
        if self.batch.obs is None:
            self._ring_only = True
        else:
            try:
                self.device_policy.value(self.batch)
                self._ring_only = True
            except B200EnvError as err:
                if 'rings' not in str(err):
                    raise
                self._ring_only = False
        self._started = True

    # -------------------------------------------------------------- learn
    def learn(self, total_timesteps, callback=None, log_interval=1, tb_log_name='PPO2', reset_num_timesteps=True):
        """stable-baselines 2.10's ``PPO2.learn``: ``total_timesteps // n_batch`` updates (n_batch = n_steps x num_envs
        agent rows), each one ``device_ppo_rollout`` and one ``device_ppo_update`` with the learning rate and clip
        ranges of ``frac = 1 - (update - 1) / n_updates``.

        ``callback``: a function ``callback(locals_, globals_)`` called after every env step (``locals_['self']`` is
        this model; ``'infos'``, ``'rewards'`` [E], ``'dones'`` [E] are the step's), an object with
        ``on_training_start`` / ``on_rollout_start`` / ``on_step`` / ``on_rollout_end`` / ``on_training_end``, or a
        list of them.  When an OptVecEnv's Monitors wrap its envs, their state of the step is recorded before the
        callback runs.  A False return stops training: the rollout is abandoned, its update skipped, and the done
        flags of that step start the next rollout.

        The first ``learn`` resets the env; later ones continue where the last stopped.  Ring-only steps write no
        observation rows, so after ``learn`` the env's last dense observation is stale: reset the env before stepping
        it directly."""
        if self.env is None:
            raise ValueError('PPO2.learn needs an env (set_env)')
        if reset_num_timesteps:
            self.num_timesteps = 0
        n_batch, n_updates = update_plan(total_timesteps, self.n_steps, self.n_envs, self.nminibatches)
        callbacks = _Callbacks(callback, self)
        if not self._started:
            self._start()
        lr_fn, clip_fn = schedule(self.learning_rate), schedule(self.cliprange)
        clip_vf_fn = None if self.cliprange_vf is None else schedule(self.cliprange_vf)
        t_first_start = time.time()
        callbacks.on_training_start(locals(), globals())
        for update in range(1, n_updates + 1):
            t_start = time.time()
            frac = frac_of(update, n_updates)
            lr_now, clip_now = lr_fn(frac), clip_fn(frac)
            clip_vf_now = clip_now if clip_vf_fn is None else clip_vf_fn(frac)
            rollout_seed, permutation_seed = update_seeds(self._seed_base, self._updates_done + 1)
            callbacks.on_rollout_start()
            step_infos = []
            try:
                device_ppo_rollout(self.batch, self.device_policy, self.buffer, self.gamma, self.lam,
                                   ring_only=self._ring_only, seed=rollout_seed,
                                   on_step=self._step_hook(callbacks, step_infos))
            except _StopTraining as stop:
                self.buffer.dones[self.n_steps].copy_(self.buffer.dones[stop.step + 1])
                callbacks.on_rollout_end()
                break
            callbacks.on_rollout_end()
            for infos in step_infos:           # Runner.run: every row's info['episode'] (the buffer keeps the last 100)
                self.ep_info_buf.extend(info['episode'] for info in infos[max(0, len(infos) - 100):]
                                        if info.get('episode') is not None)
            for group in self.optimizer.param_groups:
                group['lr'] = lr_now
            loss_vals = device_ppo_update(self.model, self.device_policy, self.buffer, self.optimizer,
                                          n_epochs=self.noptepochs, n_minibatches=self.nminibatches,
                                          cliprange=clip_now, cliprange_vf=clip_vf_now, ent_coef=self.ent_coef,
                                          vf_coef=self.vf_coef, max_grad_norm=self.max_grad_norm,
                                          seed=permutation_seed, group=self.group)
            self._updates_done += 1
            fps = int(n_batch / max(time.time() - t_start, 1e-9))
            if self.verbose >= 1 and (update % log_interval == 0 or update == 1):
                self._log(update, fps, loss_vals, t_start - t_first_start)
        callbacks.on_training_end()
        return self

    def _step_hook(self, callbacks, step_infos):
        """``on_step`` of ``device_ppo_rollout``: one device-to-host copy of the step's rewards, done flags and infos,
        the Monitor replay, the timestep count and the callbacks."""
        E = self.batch.num_envs
        packed = torch.empty((E, 18), dtype=torch.float64, device=self.device)
        host = torch.empty((E, 18), dtype=torch.float64, pin_memory=True)
        stream = torch.cuda.current_stream(self.device)

        def on_step(t, obs, reward, done, info):
            packed[:, :16].copy_(info)
            packed[:, 16].copy_(reward)
            packed[:, 17].copy_(done)
            host.copy_(packed, non_blocking=True)
            stream.synchronize()
            array = host.numpy()
            info_array = array[:, :16].copy()
            rewards, dones = array[:, 16].astype(np.float32), array[:, 17] != 0
            if isinstance(self.env, OptVecEnv):
                infos = self.env.replay_env_step(rewards, dones, info_array)
            else:
                infos = LazyInfos(info_array, self.batch.num_params)
            step_infos.append(infos)
            self.num_timesteps += self.n_envs
            if not callbacks.on_step({'self': self, 'infos': infos, 'rewards': rewards, 'dones': dones, 'n': t}):
                raise _StopTraining(t)

        return on_step

    def _log(self, update, fps, loss_vals, elapsed):
        T = self.n_steps
        rows = [('serial_timesteps', update * T), ('n_updates', update), ('total_timesteps', self.num_timesteps),
                ('fps', fps), ('explained_variance', explained_variance(self.buffer.values[:T], self.buffer.returns))]
        if len(self.ep_info_buf) > 0:
            rows += [('ep_reward_mean', float(np.mean([ep['r'] for ep in self.ep_info_buf]))),
                     ('ep_len_mean', float(np.mean([ep['l'] for ep in self.ep_info_buf])))]
        rows.append(('time_elapsed', elapsed))
        rows += list(zip(LOSS_NAMES, (float(v) for v in loss_vals)))
        text = [(key, '%-8.3g' % value if isinstance(value, float) else str(value)) for key, value in rows]
        width = max(len(key) for key, _ in text), max(len(value) for _, value in text)
        dashes = '-' * (width[0] + width[1] + 7)
        print('\n'.join([dashes] + ['| %s | %s |' % (key.ljust(width[0]), value.ljust(width[1])) for key, value in text]
                        + [dashes]), flush=True)

    # -------------------------------------------------------------- predict
    def predict(self, observation, state=None, mask=None, deterministic=False):
        """Actions of every row of ``observation`` ([rows, obs_dim], numpy or a CUDA tensor) -> (actions [rows, 1] of
        the same kind, None).  ``DevicePolicy.act``: the Gaussian's mean plus noise, or the mean alone with
        ``deterministic``, clipped to the action Box."""
        as_tensor = torch.is_tensor(observation)
        obs = observation if as_tensor else torch.from_numpy(np.ascontiguousarray(observation, dtype=np.float32))
        obs = obs.reshape(-1, self.obs_dim).to(self.device, torch.float32).contiguous()
        log_std = self.device_policy.log_std
        if deterministic:
            self.device_policy.set_log_std(None)
        try:
            actions = self.device_policy.act(obs)
        finally:
            self.device_policy.set_log_std(log_std)
        actions = actions.reshape((-1,) + self.action_shape)
        return (actions if as_tensor else actions.cpu().numpy()), None

    # -------------------------------------------------------------- parameters and files
    def get_parameters(self):
        """OrderedDict of stable-baselines' MlpPolicy names -> float32 numpy arrays in TF layouts (``PARAMETER_MAP``)."""
        return sb_parameters(self.model)

    def load_parameters(self, load_path_or_dict, exact_match=True):
        """Read parameters in stable-baselines' names from a dict or from the ``parameters`` member of a zip that
        ``save`` or stable-baselines wrote; the device policy takes them at once."""
        params = load_path_or_dict
        if not isinstance(params, dict):
            params = read_zip(params)[1]
        load_sb_parameters(self.model, params, exact_match)
        load_model(self.device_policy, self.model)

    def _data(self):
        data = {}
        for key in _HYPERPARAMETERS:
            value = getattr(self, key)
            if not callable(value):          # stable-baselines cloudpickles schedules; they are not kept here
                data[key] = value
        data['n_envs'] = self.n_envs
        return data

    def save(self, save_path):
        """stable-baselines' zip: ``data`` (JSON of the plain hyperparameters; spaces, policy class and callable
        schedules are not written), ``parameters`` (npz) and ``parameter_list`` (JSON).  A path without an extension
        gets '.zip'.  Under a group only rank 0 writes."""
        if self.group is not None:
            import torch.distributed as dist
            if dist.get_rank(self.group) != 0:
                return
        write_zip(save_path, self._data(), self.get_parameters())

    @classmethod
    def load(cls, load_path, env=None, **kwargs):
        """A model from a zip of ``save`` or of stable-baselines: the plain hyperparameters of its ``data`` (serialized
        entries are ignored), overridden by ``kwargs``, and its ``parameters``."""
        data, params = read_zip(load_path)
        hyper = plain_hyperparameters(data)
        hyper.update(kwargs)
        model = cls(MlpPolicy, env, _init_setup_model=False, **hyper)
        if 'model/pi_fc0/w:0' not in params:
            raise ValueError('%s holds no MlpPolicy parameters' % load_path)
        obs_dim = int(np.shape(params['model/pi_fc0/w:0'])[0])
        if model.obs_dim is not None and model.obs_dim != obs_dim:
            raise ValueError('the saved model reads obs_dim %d, the env has %d' % (obs_dim, model.obs_dim))
        model.obs_dim = obs_dim
        model.setup_model()
        model.load_parameters(params)
        return model


def _has_extension(path):
    import os
    return os.path.splitext(path)[1] != ''


def plain_hyperparameters(data):
    """The constructor arguments among the ``data`` entries of a saved model, without stable-baselines' serialized
    (cloudpickled) ones."""
    return {key: value for key, value in data.items()
            if key in _HYPERPARAMETERS and not (isinstance(value, dict) and ':serialized:' in value)}


def write_zip(save_path, data, params):
    """stable-baselines 2.10's ``_save_to_file_zip``: members ``data`` (JSON), ``parameters`` (``np.savez`` of
    ``params``) and ``parameter_list`` (JSON list of their names, in order).  A path without an extension gets '.zip'."""
    raw = io.BytesIO()
    np.savez(raw, **params)
    if isinstance(save_path, str) and not _has_extension(save_path):
        save_path += '.zip'
    with zipfile.ZipFile(save_path, 'w') as file_:
        file_.writestr('data', json.dumps(data, indent=4))
        file_.writestr('parameters', raw.getvalue())
        file_.writestr('parameter_list', json.dumps(list(params.keys()), indent=4))


def read_zip(path):
    """(data dict, OrderedDict of parameters in ``parameter_list`` order) of a zip that ``write_zip`` or
    stable-baselines wrote."""
    if isinstance(path, str) and not _has_extension(path) and not zipfile.is_zipfile(path):
        path += '.zip'
    if not zipfile.is_zipfile(path):
        raise ValueError('%s is not a zip archive (stable-baselines\' older cloudpickle files are not read)' % path)
    with zipfile.ZipFile(path) as file_:
        names = file_.namelist()
        if 'parameters' not in names:
            raise ValueError('%s has no "parameters" member' % path)
        data = json.loads(file_.read('data')) if 'data' in names else {}
        order = json.loads(file_.read('parameter_list')) if 'parameter_list' in names else None
        arrays = np.load(io.BytesIO(file_.read('parameters')))
        params = OrderedDict((name, arrays[name]) for name in (order or arrays.files))
    return data, params
