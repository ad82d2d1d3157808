"""The Adam baseline on the device: Keras' Adam drives the fused env batch, one learning rate per env.

The reference scores its learned optimiser against Keras' Adam (``search_baseline_hyperparam.py``: an optuna
search over Adam's learning rate, one ``model.fit`` per trial).  ``DeviceAdam`` runs that baseline on the
batch the agent trains on: every env keeps its weights, its minibatch stream and its reward, done flag,
info statistics and episode bookkeeping, and only the update rule changes (``b2e_step_adam``,
include/b200env.h).  With one learning rate per env a whole sweep is one batch::

    env = BatchedOptEnv(spec, features, targets, num_envs=4096, ...)
    adam = DeviceAdam(env, lr=torch.logspace(-5, -1, 4096, device=env.device))
    env.reset()
    monitor = DeviceEpisodeMonitor(env.num_envs, 'adam')      # .mon.csv rows, as for the agent
    adam.run(steps, on_step=monitor.on_step)

The update is Keras 2.2 ``Adam.get_updates`` with ``amsgrad=False``, restated from its source; it has not
been run against Keras itself.  SGD needs no class of its own: the constant action ``4 + log10(lr)``
(MultiOptLRs' action version 0) already gives ``w - lr * g0`` with the env's batch-SUM gradient ``g0``.
"""
from __future__ import annotations

import ctypes

import torch

from custom_envs_b200 import _lib
from custom_envs_b200.batched_env import BatchedOptEnv


def _ptr(tensor):
    return ctypes.c_void_p(0 if tensor is None else tensor.data_ptr())


def _device_batch(env):
    """The ``BatchedOptEnv`` behind ``env`` (itself, or the batch of a device-backed ``OptVecEnv``)."""
    if isinstance(env, BatchedOptEnv):
        return env
    from custom_envs_b200.vectorize.optvecenv import OptVecEnv
    if isinstance(env, OptVecEnv):
        if not env.is_device_backed:
            raise ValueError('DeviceAdam needs an OptVecEnv whose envs are fused into one device batch; this one '
                             'runs on the host fallback, which has no device batch to drive')
        return env._impl.env
    raise ValueError('DeviceAdam takes a BatchedOptEnv or a device-backed OptVecEnv, not %s' % type(env).__name__)


class DeviceAdam:
    """Keras' Adam (lr, beta_1, beta_2, epsilon; Keras 2.2 defaults) in place of the agent's actions.

    ``lr``: a float for every env, or a tensor [E] with one learning rate per env.  The moments m and v
    [E, P] (natural parameter order) are held here; step t = 1 of every episode ignores them, so resets,
    auto-resets included, need not touch them.  MultiOptLRs envs only."""

    def __init__(self, env, lr=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        batch = _device_batch(env)
        if batch.env_kind_name != 'optlrs':
            raise ValueError('DeviceAdam drives MultiOptLRs envs; a MultiOptimize action is a weight delta and its '
                             'minibatch never advances')
        if not (0.0 <= beta_1 < 1.0 and 0.0 <= beta_2 < 1.0):
            raise ValueError('beta_1 and beta_2 must lie in [0, 1)')
        if not epsilon > 0.0:
            raise ValueError('epsilon must be positive')
        self.env, self.batch = env, batch
        self.device = batch.device
        self.lr = self._check_lr(lr)
        self.beta_1, self.beta_2, self.epsilon = float(beta_1), float(beta_2), float(epsilon)
        self._opt = _lib.Adam(self.beta_1, self.beta_2, self.epsilon)
        shape = (batch.num_envs, batch.num_params)
        self.m = torch.zeros(shape, dtype=torch.float32, device=self.device)
        self.v = torch.zeros(shape, dtype=torch.float32, device=self.device)

    def _check_lr(self, lr):
        num_envs = self.batch.num_envs
        if torch.is_tensor(lr):
            if tuple(lr.shape) != (num_envs,):
                raise ValueError('lr must be a float or a tensor of shape [%d], not %s' % (num_envs, tuple(lr.shape)))
            lr = lr.detach().to(self.device, torch.float32).clone()     # a copy: later edits of the caller's tensor do not reach it
        else:
            lr = torch.full((num_envs,), float(lr), dtype=torch.float32, device=self.device)
        if not bool(torch.all(torch.isfinite(lr) & (lr > 0))):
            raise ValueError('every learning rate must be positive and finite')
        return lr

    def step(self, ring_only=False):
        """One Adam step of every env -> what ``BatchedOptEnv.step`` returns: (obs [E*P, obs_dim] or None
        with ``ring_only``, reward [E], done [E], info [E, 16]), views of buffers the next step overwrites."""
        batch = self.batch
        obs = None if ring_only else batch.obs
        if obs is None and not ring_only:
            raise _lib.B200EnvError('the env holds no observation matrix (materialize_obs=False): step(ring_only=True)')
        if batch.handle is None:
            raise _lib.B200EnvError('the env is closed')
        batch._check(batch.lib.b2e_step_adam(batch.handle, ctypes.byref(self._opt), _ptr(self.lr), _ptr(self.m),
                                             _ptr(self.v), None, None, _ptr(obs), _ptr(batch.reward),
                                             _ptr(batch.done), _ptr(batch.info), batch._stream()))
        return obs, batch.reward, batch.done, batch.info

    @torch.no_grad()
    def run(self, steps, on_step=None, ring_only=False):
        """``steps`` Adam steps; ``on_step(t, obs, reward, done, info)`` after each (the hook of
        ``device_policy_rollout``, e.g. ``DeviceEpisodeMonitor.on_step``).  Returns (per-env reward sums [E]
        float64, finished episodes)."""
        returns = torch.zeros(self.batch.num_envs, dtype=torch.float64, device=self.device)
        finished = torch.zeros((), dtype=torch.int64, device=self.device)
        for t in range(int(steps)):
            obs, reward, done, info = self.step(ring_only)
            returns.add_(reward)
            finished.add_(done.sum())
            if on_step is not None:
                on_step(t, obs, reward, done, info)
        return returns, int(finished.item())

    def state(self):
        """The optimiser's state: copies of m, v [E, P] and lr [E]."""
        return {'m': self.m.clone(), 'v': self.v.clone(), 'lr': self.lr.clone()}

    def load_state(self, state):
        """Restore ``state()`` (lr optional)."""
        for name in ('m', 'v'):
            value = torch.as_tensor(state[name])
            if tuple(value.shape) != tuple(self.m.shape):
                raise ValueError('%s must have shape %s, not %s' % (name, tuple(self.m.shape), tuple(value.shape)))
            getattr(self, name).copy_(value.to(self.device, torch.float32))
        if 'lr' in state:
            self.lr = self._check_lr(torch.as_tensor(state['lr']))
