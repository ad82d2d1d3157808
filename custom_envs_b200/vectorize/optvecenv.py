"""``OptVecEnv``: the stable-baselines VecEnv whose rows are the per-parameter agents of
many optimise envs (reference vectorize/optvecenv.py:10-91).

Two implementations behind one class:
* device path -- every env is a device-backed ``MultiOptLRs`` / ``MultiOptimize`` of one
  configuration: they are fused into ONE ``BatchedOptEnv`` (E envs in HBM, one kernel
  launch per ``step``), wrappers such as ``Monitor`` keep seeing their env's per-step
  ``(reward, done, info)``;
* generic path -- anything else (e.g. the reference's StubEnv tests) runs thread-per-env
  through ``ThreadVecEnv`` + ``OptEnvRunner`` exactly as the reference does.
"""
import time
from itertools import chain

import numpy as np

from custom_envs_b200.compat import VecEnv
from custom_envs_b200.vectorize.concurrentvecenv import ThreadVecEnv

INFO_KEYS = ('loss', 'batch_loss', 'weights_mean', 'weights_sum', 'actions_mean',
             'actions_std', 'states_mean', 'states_sum', 'grads_mean', 'grads_sum',
             'loss_mean', 'adjusted_loss', 'adjusted_grad', 'grad_diff')


def flatten_dictionary(dictionary):
    """Values of an agent dict ordered by full agent name (lexicographic)."""
    return tuple(value for _, value in sorted(dictionary.items(), key=lambda item: item[0]))


def info_row_to_dict(row):
    """One env's 16 info doubles -> the reference's info dict (multioptlrs.py:111-127,
    baseenvironment.py:40)."""
    info = {key: float(row[i]) for i, key in enumerate(INFO_KEYS)}
    if info['loss'] != info['loss']:
        info['loss'] = None
    info['episode'] = {'r': float(row[14]), 'l': int(row[15])}
    return info


class LazyInfos:
    """``infos`` of the VecEnv contract: one dict per agent row, the same dict object for
    the P rows of an env (optvecenv.py:45), built on first access."""

    def __init__(self, info_array, agents_per_env, overrides=None):
        self._array = info_array
        self._agents = int(agents_per_env)
        self._cache = dict(overrides or {})

    def __len__(self):
        return self._array.shape[0] * self._agents

    def env_info(self, env_index):
        if env_index not in self._cache:
            self._cache[env_index] = info_row_to_dict(self._array[env_index])
        return self._cache[env_index]

    def __getitem__(self, row):
        if isinstance(row, slice):
            return [self[i] for i in range(*row.indices(len(self)))]
        if row < 0:
            row += len(self)
        if not 0 <= row < len(self):
            raise IndexError(row)
        return self.env_info(row // self._agents)

    def __iter__(self):
        for env_index in range(self._array.shape[0]):
            info = self.env_info(env_index)
            for _ in range(self._agents):
                yield info


_COPY_POOL = None
_COPY_CHUNK = 1 << 23            # float32 elements per staged chunk (32 MB)


def _copy_pool():
    """Host threads that stage numpy inputs into pinned memory.  Own pool, because torchrun
    exports OMP_NUM_THREADS=1 and would make torch's host copy single-threaded."""
    global _COPY_POOL
    if _COPY_POOL is None:
        import os
        from concurrent.futures import ThreadPoolExecutor
        cpus = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
        _COPY_POOL = ThreadPoolExecutor(max(1, min(8, cpus)), thread_name_prefix='b2e-stage')
    return _COPY_POOL


def stage_to_device(src, host, dev, chunk=_COPY_CHUNK):
    """numpy ``src`` -> pinned ``host`` -> device ``dev`` (1-D, same length).  Chunks are copied
    into the pinned buffer by the pool (numpy releases the GIL) and each chunk's
    host->device copy is queued as soon as it is staged, so the two overlap."""
    count = src.shape[0]
    staged = host.numpy()
    if count <= chunk:
        np.copyto(staged, src)
        dev.copy_(host, non_blocking=True)
        return
    cuts = list(range(0, count, chunk)) + [count]
    pool = _copy_pool()
    jobs = [pool.submit(np.copyto, staged[lo:hi], src[lo:hi]) for lo, hi in zip(cuts, cuts[1:])]
    for job, lo, hi in zip(jobs, cuts, cuts[1:]):
        job.result()
        dev[lo:hi].copy_(host[lo:hi], non_blocking=True)


class DeviceOptVecEnv(VecEnv):
    """VecEnv over a ``BatchedOptEnv``: numpy in, numpy out, state stays in HBM.

    ``step_async`` copies the actions host->device from pinned memory and launches the
    fused step; ``step_wait`` copies observations / rewards / dones / infos device->host
    into pinned buffers.  ``rewards`` / ``terminals`` / ``infos`` are fresh objects every step
    (the stable-baselines runners append them to their rollout lists without copying).  The
    ``states`` array alone is a view of the pinned observation buffer, valid until the next
    ``step_wait`` / ``reset`` -- the runners copy observations themselves (``self.obs[:] = obs``,
    ``mb_obs.append(self.obs.copy())``) -- unless ``copy_outputs=True`` asks for a private copy of
    the 60-byte-per-agent matrix as well."""

    def __init__(self, batched_env, observation_space=None, action_space=None, callbacks=(),
                 copy_outputs=False, direct_host_obs=None):
        import torch
        from custom_envs_b200.utils import utils_env
        self._torch = torch
        self.env = batched_env
        self.agent_no_list = [batched_env.num_params] * batched_env.num_envs
        self.callbacks = callbacks
        self.copy_outputs = copy_outputs
        # option: the observation kernel writes its rows straight into the pinned host buffer
        # (unified addressing) instead of HBM + a device->host copy.  Measured on a B200 at
        # 2e8 rows: 13.7 k env-steps/s against 14.6 k with the copy engine, so it is off by default.
        if direct_host_obs is None:
            import os
            direct_host_obs = os.environ.get('B2E_DIRECT_HOST_OBS', '0') != '0'
        self.direct_host_obs = bool(direct_host_obs)
        self.waiting = False
        self.closed = False
        self.last_timing = {}
        if observation_space is None:
            observation_space, _ = utils_env.get_obs_version((batched_env.num_params,),
                                                             batched_env.max_history, 3)
        if action_space is None:
            action_space = utils_env.get_action_space_optlrs(2)
        VecEnv.__init__(self, batched_env.num_rows, observation_space, action_space)
        dev = batched_env.device
        rows, dim, envs = batched_env.num_rows, batched_env.obs_dim, batched_env.num_envs
        pin = dict(pin_memory=True)
        self._act_host = torch.empty(rows, dtype=torch.float32, **pin)
        self._act_dev = torch.empty(rows, dtype=torch.float32, device=dev)
        self._obs_host = torch.empty((rows, dim), dtype=torch.float32, **pin)
        self._rew_host = torch.empty(envs, dtype=torch.float32, **pin)
        self._done_host = torch.empty(envs, dtype=torch.uint8, **pin)
        self._info_host = torch.empty((envs, 16), dtype=torch.float64, **pin)
        # the VecEnv surface repeats reward / done once per agent row (optvecenv.py:43-45): host
        # threads expand the per-env values while the observation copy is still on the wire.
        # FRESH arrays every step, like the reference's np.stack: PPO2 / A2C runners keep
        # ``rewards`` / ``dones`` of every step of a rollout without copying them.
        self._rew_rows_np = None
        self._done_rows_np = None
        self._scalars_event = torch.cuda.Event()
        self._event = torch.cuda.Event()

    def _states(self):
        states = self._obs_host.numpy()
        return states.copy() if self.copy_outputs else states

    def _row_outputs(self):
        """(rewards[rows], terminals[rows]): arrays allocated for this step, never reused."""
        return self._rew_rows_np, self._done_rows_np

    def _expand_rows(self):
        envs, agents = self.env.num_envs, self.env.num_params
        reward = self._rew_host.numpy()
        done = self._done_host.numpy().astype(np.bool_)
        self._rew_rows_np = np.empty(envs * agents, dtype=np.float32)
        self._done_rows_np = np.empty(envs * agents, dtype=np.bool_)
        rew_rows = self._rew_rows_np.reshape(envs, agents)
        done_rows = self._done_rows_np.reshape(envs, agents)

        def fill(lo, hi):
            rew_rows[lo:hi] = reward[lo:hi, None]
            done_rows[lo:hi] = done[lo:hi, None]

        if envs * agents <= _COPY_CHUNK:
            fill(0, envs)
            return
        pool = _copy_pool()
        cuts = np.linspace(0, envs, min(envs, 4 * pool._max_workers) + 1).astype(np.int64)
        for job in [pool.submit(fill, int(lo), int(hi)) for lo, hi in zip(cuts, cuts[1:])]:
            job.result()

    def _wait_outputs(self):
        """Block until the step's outputs are in host memory: the per-env scalars arrive
        first and are expanded per agent row while the observation copy is in flight."""
        clock = time.perf_counter
        t0 = clock()
        self._scalars_event.synchronize()
        t1 = clock()
        self._expand_rows()
        t2 = clock()
        self._event.synchronize()
        t3 = clock()
        self.waiting = False
        # host-side phases of the last step in ms (where the end-to-end time goes)
        self.last_timing.update(wait_step=1e3 * (t1 - t0), expand_rows=1e3 * (t2 - t1),
                                wait_obs_copy=1e3 * (t3 - t2))

    def reset(self):
        obs = self.env.reset()
        self._obs_host.copy_(obs, non_blocking=True)
        self._torch.cuda.current_stream(self.env.device).synchronize()
        return self._states()

    def step_async(self, actions):
        actions = np.ascontiguousarray(np.asarray(actions, np.float32).reshape(-1))
        assert actions.size == self.num_envs
        t0 = time.perf_counter()
        stage_to_device(actions, self._act_host, self._act_dev)
        t1 = time.perf_counter()
        obs, reward, done, info = self.env.step(
            self._act_dev, obs_out=self._obs_host if self.direct_host_obs else None)
        self._rew_host.copy_(reward, non_blocking=True)
        self._done_host.copy_(done, non_blocking=True)
        self._info_host.copy_(info, non_blocking=True)
        self._scalars_event.record(self._torch.cuda.current_stream(self.env.device))
        if not self.direct_host_obs:
            self._obs_host.copy_(obs, non_blocking=True)
        self._event.record(self._torch.cuda.current_stream(self.env.device))
        self.waiting = True
        self.last_timing = {'stage_actions': 1e3 * (t1 - t0), 'queue_step': 1e3 * (time.perf_counter() - t1)}

    def step_wait(self):
        self._wait_outputs()
        agents = self.env.num_params
        states = self._states()
        rewards, terminals = self._row_outputs()
        infos = LazyInfos(self._info_host.numpy().copy(), agents)
        for callback in self.callbacks:
            callback(states, rewards, terminals, infos)
        return states, rewards, terminals, infos

    def close(self):
        if self.closed:
            return
        if self.waiting:
            self._event.synchronize()
        self.env.close()
        self.closed = True

    def get_attr(self, attr_name, indices=None):
        value = getattr(self.env, attr_name)
        return [value] * self.env.num_envs

    def set_attr(self, attr_name, value, indices=None):
        raise AttributeError('DeviceOptVecEnv has no per-env Python objects; use OptVecEnv')

    def env_method(self, method_name, *method_args, **method_kwargs):
        raise AttributeError('DeviceOptVecEnv has no per-env Python objects; use OptVecEnv')


class OptEnvRunner:
    """Dict-of-agents env -> rows (reference optvecenv.py:17-54); generic path only."""

    def __init__(self, environment_fn):
        environment = environment_fn()
        self._environment = environment
        self._names = list(environment.action_space.spaces)        # Dict order == sorted keys
        first = self._names[0]
        self.observation_space = environment.observation_space.spaces[first]
        self.action_space = environment.action_space.spaces[first]
        self._num_agents = len(environment.observation_space.spaces)
        assert all(space == self.observation_space
                   for space in environment.observation_space.spaces.values())
        assert all(space == self.action_space for space in environment.action_space.spaces.values())

    def reset(self):
        return flatten_dictionary(self._environment.reset())

    def step(self, actions):
        states, reward, terminal, info = self._environment.step(dict(zip(self._names, actions)))
        agents = self._num_agents
        return flatten_dictionary(states), [reward] * agents, [terminal] * agents, [info] * agents

    def close(self):
        self._environment.close()

    def __getattr__(self, attr):
        if attr.startswith('__'):
            raise AttributeError(attr)
        return getattr(self._environment, attr)


class _GenericOptVecEnv(ThreadVecEnv):
    def __init__(self, environments, callbacks=()):
        super().__init__([(lambda env=env: OptEnvRunner(lambda: env)) for env in environments])
        self.agent_no_list = self.get_attr('_num_agents')
        self.num_envs = sum(self.agent_no_list)
        self.callbacks = callbacks

    def step_async(self, actions):
        grouped, start = [], 0
        for count in self.agent_no_list:
            grouped.append(actions[start:start + count])
            start += count
        super().step_async(grouped)

    def step_wait(self):
        results = [remote.recv() for remote in self.remotes]
        self.waiting = False
        obs, rews, dones, infos = zip(*results)
        states = np.stack(list(chain.from_iterable(obs)))
        rewards = np.stack(list(chain.from_iterable(rews)))
        terminals = np.stack(list(chain.from_iterable(dones)))
        infos = list(chain.from_iterable(infos))
        for callback in self.callbacks:
            callback(states, rewards, terminals, infos)
        return states, rewards, terminals, infos

    def reset(self):
        results = self._ask(self.remotes, 'reset', None)
        return np.stack(list(chain.from_iterable(results)))


def _core_env(env):
    """Innermost env of a wrapper chain."""
    seen = 0
    while hasattr(env, 'env') and seen < 32:
        env = env.env
        seen += 1
    return env


class OptVecEnv(VecEnv):
    """``OptVecEnv(environment_fns, callbacks=())`` -- reference signature and outputs:
    ``reset() -> [sum P, obs_dim]``; ``step(actions[sum P, 1]) -> (states, rewards[sum P],
    terminals[sum P], infos)``; ``num_envs = sum P``; ``agent_no_list``."""

    def __init__(self, environment_fns, callbacks=(), device=None):
        from custom_envs_b200.envs.device_env import DeviceEnvFront, fuse_fronts
        environments = [fn() for fn in environment_fns]
        cores = [_core_env(env) for env in environments]
        self.callbacks = callbacks
        self.waiting = False
        self.closed = False
        self._chains = environments
        self._cores = cores
        fused = (all(isinstance(core, DeviceEnvFront) for core in cores)
                 and len({core.fuse_key() for core in cores}) == 1)
        if fused:
            backend = fuse_fronts(cores, device=device)
            first = cores[0]
            names = list(first.action_space.spaces)
            self._impl = DeviceOptVecEnv(backend, first.observation_space.spaces[names[0]],
                                         first.action_space.spaces[names[0]], copy_outputs=False)
            self._wrapped = [env is not core for env, core in zip(environments, cores)]
            # Fast path for the scripts' usual chain, one callback-free Monitor around each env
            # (search_optimize_hyperparam.py:97-110): per-step bookkeeping is vectorised over the
            # envs and the per-env Python objects are only touched when an episode ends.
            from custom_envs_b200.utils.utils_logging import Monitor as _LenientMonitor
            self._fast_monitor = all(
                (env is core) or (type(env) is _LenientMonitor and env.env is core and not env.callbacks)
                for env, core in zip(environments, cores))
            self._ep_sum = np.zeros(len(cores), np.float64)
            self._ep_len = np.zeros(len(cores), np.int64)
            self._steps = np.zeros(len(cores), np.int64)
            if self._fast_monitor:
                for slot, core in enumerate(cores):
                    core._shared_steps = (self._steps, slot)
        else:
            self._impl = _GenericOptVecEnv(environments)
            self._wrapped = None
        self.agent_no_list = self._impl.agent_no_list
        VecEnv.__init__(self, self._impl.num_envs, self._impl.observation_space,
                        self._impl.action_space)

    @property
    def is_device_backed(self):
        return self._wrapped is not None

    def reset(self):
        states = self._impl.reset()
        if self.is_device_backed:
            self._ep_sum[:] = 0.0
            self._ep_len[:] = 0
            self._steps[:] = 0
            for env, core in zip(self._chains, self._cores):
                core._host_reset_done()
                if env is not core:
                    env.reset()                   # wrappers (Monitor) see the reset
        return states

    def step_async(self, actions):
        self._impl.step_async(actions)
        self.waiting = True

    def step_wait(self):
        self.waiting = False
        if not self.is_device_backed:
            states, rewards, terminals, infos = self._impl.step_wait()
        else:
            impl = self._impl
            impl._wait_outputs()
            states = impl._states()
            info_array = impl._info_host.numpy().copy()
            infos = self.replay_env_step(impl._rew_host.numpy(), impl._done_host.numpy().astype(bool), info_array)
            rewards, terminals = impl._row_outputs()
        for callback in self.callbacks:
            callback(states, rewards, terminals, infos)
        return states, rewards, terminals, infos

    def replay_env_step(self, reward_env, done_env, info_array):
        """Per-env bookkeeping of one step of the fused batch (device-backed path): every env's step counter, and its
        result replayed through its wrappers, so that Monitors write their ``.mon.csv`` rows, ``get_episode_rewards``
        grows and ``info['episode']`` is the Monitor's.  ``reward_env`` float32 [E], ``done_env`` bool [E] and
        ``info_array`` float64 [E, 16] are host arrays of that step (``info_array`` is kept by the result).  Returns
        the step's ``LazyInfos``.  ``step_wait`` and the device trainer (``custom_envs_b200.ppo2.PPO2``) both call it."""
        overrides = {}
        if self._fast_monitor:
            # sum(self.rewards) in Monitor.step adds the float rewards in step order: a
            # running float64 sum per env is the same arithmetic
            self._ep_sum += reward_env.astype(np.float64)
            self._ep_len += 1
            self._steps[:] = info_array[:, 15].astype(np.int64)
            for e in np.nonzero(done_env)[0]:
                env, core = self._chains[e], self._cores[e]
                self._steps[e] = 0
                if env is not core:
                    info = info_row_to_dict(info_array[e])
                    env._finish_episode(float(self._ep_sum[e]), int(self._ep_len[e]),
                                        float(reward_env[e]), info)
                    overrides[e] = info
                    env.rewards = []                       # what Monitor.reset does
                    env.current_episode += 1
                self._ep_sum[e] = 0.0
                self._ep_len[e] = 0
        for e, (env, core) in enumerate(() if self._fast_monitor else zip(self._chains, self._cores)):
            core._host_step_done(info_array[e], bool(done_env[e]))
            if env is core:
                continue
            # replay this env's result through its wrappers (Monitor bookkeeping)
            core._pending = (float(reward_env[e]), bool(done_env[e]), info_row_to_dict(info_array[e]))
            _, _, done, info = env.step(None)
            overrides[e] = info
            if done:
                env.reset()
        return LazyInfos(info_array, self._impl.env.num_params, overrides)

    def close(self):
        if self.closed:
            return
        if self.is_device_backed:
            # the reference's worker closes its env chain (concurrentvecenv.py:45-47): a Monitor writes the
            # episodes it still holds (chunk_size > 1) from its close()
            for env in self._chains:
                env.close()
        self._impl.close()
        self.closed = True

    def get_attr(self, attr_name, indices=None):
        if not self.is_device_backed:
            return self._impl.get_attr(attr_name, indices)
        if attr_name == '_num_agents':
            return list(self.agent_no_list)
        return [getattr(env, attr_name) for env in self._select(indices)]

    def set_attr(self, attr_name, value, indices=None):
        if not self.is_device_backed:
            return self._impl.set_attr(attr_name, value, indices)
        return [setattr(env, attr_name, value) for env in self._select(indices)]

    def env_method(self, method_name, *method_args, **method_kwargs):
        if not self.is_device_backed:
            return self._impl.env_method(method_name, *method_args, **method_kwargs)
        return [getattr(env, method_name)(*method_args, **method_kwargs) for env in self._chains]

    def _select(self, indices):
        if indices is None:
            return self._chains
        if isinstance(indices, int):
            indices = [indices]
        return [self._chains[i] for i in indices]

    def get_images(self):
        return []

    def render(self, *args, **kwargs):
        return None
