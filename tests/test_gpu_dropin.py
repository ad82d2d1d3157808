"""GPU tests of the drop-in surface: the reference's env / problem / VecEnv tests
(tests/envs/test_env.py, tests/problems/test_base_problem.py, tests/vectorize/test_optvecenv.py)
re-expressed against the device-backed classes, reached through the ``custom_envs`` alias."""
import os
import tempfile
from functools import partial

import numpy as np
import pandas as pd
import pytest

from oracle import optenv_oracle as orc

pytestmark = pytest.mark.gpu


def test_env_step_and_reset_types():
    from custom_envs.envs import SINGLE_AGENT_ENVIRONMENTS
    for env_cls in SINGLE_AGENT_ENVIRONMENTS:
        env = env_cls()       # defaults: Rosenbrock (MultiOptLRs), iris + (256, 256) stack (MultiOptimize)
        state = env.reset()
        assert env.current_step == 0 and env.observation_space.contains(state)
        action = env.action_space.sample()
        if env_cls.__name__ == 'MultiOptimize':
            # +-4 is a step of +-10 on every weight (multioptimize.py:95-98): keep the run inside
            # the declared +-1e6 observation box
            action = type(action)((key, value * 0.25) for key, value in action.items())
        for i in range(1, 10):
            state, reward, terminal, info = env.step(action)
            assert env.current_step == i
            assert env.observation_space.contains(state)
            assert isinstance(reward, float) and isinstance(terminal, bool) and isinstance(info, dict)
            assert info['episode'] == {'r': reward, 'l': i}
            if terminal:
                break
        env.close()


def test_multioptlrs_nn_on_iris_matches_oracle():
    from custom_envs.envs import MultiOptLRs
    from custom_envs import load_data
    data = load_data('iris', 32)
    env = MultiOptLRs(problem='nn', max_batches=8, max_history=5,
                      problem_kwargs=dict(layers=(), data_set=data))
    env.seed(3)
    state = env.reset()
    assert len(state) == 15 and all(np.all(v == -1) for v in state.values())
    spec = orc.ProblemSpec('softmax', 4, (), 3)
    perm = np.arange(150)
    rs = np.random.RandomState()
    rs.set_state(env.random_generator.get_state())
    rs.shuffle(perm)
    ref = orc.BatchedOptEnvOracle(spec, data.features.astype(np.float32), data.targets.argmax(1), 1,
                                  batch_size=32, config=orc.EnvConfig.multioptlrs(8, 5), perms=perm[None])
    ref.reset(init_params=env.model.get_parameters()[None].astype(np.float32))
    rng = np.random.RandomState(0)
    for t in range(8):
        nat = rng.uniform(0, 3, size=15).astype(np.float32)
        action = {'parameter-%d' % i: np.array([nat[i]], np.float32) for i in range(15)}
        state, reward, terminal, info = env.step(action)
        want_obs, want_rew, want_done, want_info = ref.step(nat[None])
        got = np.stack([state['parameter-%d' % i] for i in range(15)])
        err = np.abs(got - want_obs[0]) / np.maximum(1, np.abs(want_obs[0] + 1))
        assert err.max() < 2e-4, (t, err.max())
        assert abs(reward - want_rew[0]) < 1e-4 and terminal == bool(want_done[0])
        assert (info['loss'] is None) == (not terminal)
        assert abs(info['batch_loss'] - want_info['batch_loss'][0]) < 1e-5
    assert terminal
    env.close()


@pytest.mark.parametrize('name', ['func', 'nn', 'nn-default'])
def test_base_problem_contract(name):
    from custom_envs.problems import get_problem
    kwargs = dict(layers=(8,)) if name == 'nn' else {}    # nn-default: the reference's (256, 256)
    default = name == 'nn-default'
    name = name.split('-')[0]
    problem = get_problem(name, **kwargs)
    assert not default or problem.size == 4 * 256 + 256 + 256 * 256 + 256 + 256 * 3 + 3
    old = np.random.rand(problem.size)
    problem.set_parameters(old)
    assert np.allclose(problem.get_parameters(), old, atol=1e-6)        # set -> get round trip
    gradient, loss, params = problem.get()
    assert np.array(gradient).ndim == 1 and np.array(params).ndim == 1 and float(loss) == float(loss)
    assert np.allclose(gradient, problem.get_gradient()) and np.isclose(loss, problem.get_loss())
    assert np.allclose(params, problem.parameters)
    problem.reset()
    assert not np.allclose(problem.get_parameters(), old)
    if name == 'nn':
        before = problem.get_loss()
        problem.next()
        assert problem.get_loss() != before                             # next minibatch
    with pytest.raises(RuntimeError):
        get_problem('other')


def test_optvecenv_fuses_monitored_envs():
    from custom_envs.vectorize import OptVecEnv
    from custom_envs.utils.utils_logging import Monitor
    from custom_envs_b200.compat import make
    from custom_envs import load_data
    data = load_data('iris', 32)
    keys = ('loss', 'actions_mean', 'weights_mean', 'actions_std', 'states_mean', 'grads_mean')
    with tempfile.TemporaryDirectory() as tmp:
        fns = [partial(Monitor, partial(make, 'MultiOptLRs-v0', problem='nn', max_batches=5,
                                        problem_kwargs=dict(layers=(), data_set=data)),
                       os.path.join(tmp, 'env%d' % i), info_keywords=keys) for i in range(3)]
        seen = []
        vec = OptVecEnv(fns, callbacks=(lambda s, r, t, i: seen.append(len(s)),))
        assert vec.is_device_backed and vec.num_envs == 45 and vec.agent_no_list == [15, 15, 15]
        states = vec.reset()
        assert states.shape == (45, 15) and np.all(states == -1)
        for t in range(11):
            actions = np.random.RandomState(t).uniform(0, 2, size=(45, 1)).astype(np.float32)
            states, rewards, terminals, infos = vec.step(actions)
            assert states.shape == (45, 15) and rewards.shape == (45,) and terminals.shape == (45,)
            assert len(infos) == 45 and infos[0] is infos[14] and infos[15] is not infos[0]
            assert np.all(rewards[:15] == rewards[0])
            if (t + 1) % 5 == 0:
                assert terminals.all() and np.all(states == -1)          # auto-reset observation
                assert infos[0]['loss'] is not None and infos[0]['episode']['l'] == 5
            else:
                assert not terminals.any() and infos[0]['loss'] is None
                assert infos[0]['episode']['l'] == (t % 5) + 1
        assert len(seen) == 11
        episode_rewards = vec.env_method('get_episode_rewards')
        assert [len(r) for r in episode_rewards] == [2, 2, 2]
        assert vec.get_attr('current_step') == [1, 1, 1]
        vec.close()
        frame = pd.read_csv(os.path.join(tmp, 'env0.mon.csv'))
        assert len(frame) == 2 and set(keys) <= set(frame.columns) and list(frame['l']) == [5, 5]


def test_optvecenv_step_outputs_survive_the_next_step():
    """stable-baselines' runners do ``mb_rewards.append(rewards)`` / ``mb_dones.append(self.dones)``
    without copying (ppo2.py Runner.run), so the rewards / terminals / infos of step N must not be
    rewritten by step N+1 (the reference returns fresh ``np.stack`` results, optvecenv.py:78-88)."""
    from custom_envs.vectorize import OptVecEnv
    from custom_envs_b200.compat import make
    from custom_envs import load_data
    data = load_data('iris', 32)
    fns = [partial(make, 'MultiOptLRs-v0', problem='nn', max_batches=3,
                   problem_kwargs=dict(layers=(), data_set=data)) for _ in range(3)]
    vec = OptVecEnv(fns)
    vec.reset()
    kept, snapshots = [], []
    for t in range(5):
        actions = np.random.RandomState(t).uniform(0, 2, size=(45, 1)).astype(np.float32)
        _, rewards, terminals, infos = vec.step(actions)
        kept.append((rewards, terminals, infos[0]))
        snapshots.append((rewards.copy(), terminals.copy(), dict(infos[0])))
    for (rewards, terminals, info), (rew_then, term_then, info_then) in zip(kept, snapshots):
        assert np.array_equal(rewards, rew_then) and np.array_equal(terminals, term_then)
        assert info == info_then
    assert len({id(k[0]) for k in kept}) == 5 and len({id(k[1]) for k in kept}) == 5
    assert not np.array_equal(kept[0][0], kept[1][0])
    vec.close()


def test_vectorised_monitor_path_equals_per_env_replay():
    """A callback-free Monitor around every env takes the vectorised bookkeeping path of the fused
    OptVecEnv; a Monitor with a callback forces the per-env replay.  Same seeds -> same outputs,
    same episode rows in the .mon.csv files."""
    from custom_envs.vectorize import OptVecEnv
    from custom_envs.utils.utils_logging import Monitor
    from custom_envs_b200.compat import make
    from custom_envs import load_data
    data = load_data('iris', 32)
    keys = ('loss', 'actions_mean', 'weights_mean')

    def build(i, tmp, slow):
        env = make('MultiOptLRs-v0', problem='nn', max_batches=4,
                   problem_kwargs=dict(layers=(5,), data_set=data))
        env.seed(100 + i)
        return Monitor(env, os.path.join(tmp, 'env%d' % i), info_keywords=keys,
                       callbacks=[lambda record: None] if slow else None)

    runs = []
    for slow in (False, True):
        with tempfile.TemporaryDirectory() as tmp:
            vec = OptVecEnv([partial(build, i, tmp, slow) for i in range(4)])
            assert vec.is_device_backed and vec._fast_monitor == (not slow)
            vec.reset()
            outputs = []
            for t in range(10):
                actions = np.random.RandomState(t).uniform(0, 2, size=(vec.num_envs, 1)).astype(np.float32)
                states, rewards, terminals, infos = vec.step(actions)
                outputs.append((states.copy(), rewards.copy(), terminals.copy(),
                                [infos[e * vec.agent_no_list[0]]['episode'] for e in range(4)]))
            steps = vec.get_attr('current_step')
            totals = vec.env_method('get_episode_rewards')
            vec.close()
            frames = [pd.read_csv(os.path.join(tmp, 'env%d.mon.csv' % i)).drop(columns=['t']) for i in range(4)]
            runs.append((outputs, steps, totals, frames))
    fast, slow = runs
    assert fast[1] == slow[1] == [2, 2, 2, 2] and fast[2] == slow[2]
    for (s0, r0, t0, e0), (s1, r1, t1, e1) in zip(fast[0], slow[0]):
        assert np.array_equal(s0, s1) and np.array_equal(r0, r1) and np.array_equal(t0, t1)
        for a, b in zip(e0, e1):
            assert {k: v for k, v in a.items() if k != 't'} == {k: v for k, v in b.items() if k != 't'}
    for a, b in zip(fast[3], slow[3]):
        assert len(a) == 2 and a.equals(b)


def test_device_optvecenv_matches_vecenv_oracle():
    """Host-buffer VecEnv path (lexicographic rows, auto-reset, internal stream) vs the oracle."""
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    from custom_envs_b200.vectorize import DeviceOptVecEnv
    spec = orc.ProblemSpec('softmax', 6, (5,), 3)
    rng = np.random.RandomState(4)
    feats = rng.uniform(size=(50, 6)).astype(np.float32)
    labels = rng.randint(0, 3, 50).astype(np.int32)
    num_envs = 3
    perms = np.stack([orc.env_permutation(50, s) for s in range(num_envs)])
    env = BatchedOptEnv(ProblemSpec('softmax', 6, (5,), 3), feats, labels, num_envs, batch_size=16,
                        max_batches=6, perms=perms, auto_reset=False)
    ref = orc.OptVecEnvOracle(orc.BatchedOptEnvOracle(spec, feats, labels, num_envs, batch_size=16,
                                                      config=orc.EnvConfig.multioptlrs(6, 5), perms=perms))
    vec = DeviceOptVecEnv(env)
    init = np.stack([orc.glorot_uniform_init(spec, rng) for _ in range(num_envs)])
    env.reset(init_params=init)
    ref.reset(init_params=init)
    for t in range(5):
        actions = rng.uniform(0, 2.5, size=(vec.num_envs, 1)).astype(np.float32)
        states, rewards, terminals, infos = vec.step(actions)
        want_s, want_r, want_t, want_i = ref.step(actions[:, 0])
        err = np.abs(states - want_s) / np.maximum(1, np.abs(want_s + 1))
        assert np.mean(err < 1e-4) > 0.97
        assert np.allclose(rewards, want_r, rtol=1e-4, atol=1e-4) and np.array_equal(terminals, want_t)
        assert abs(infos[0]['batch_loss'] - want_i['batch_loss'][0]) < 1e-4
    vec.close()


def test_device_wrappers_match_host_wrappers():
    """DeviceHistoryWrapper / DeviceSubSetWrapper over the fused env batch give what the reference's
    HistoryWrapper / SubSetWrapper (wrappers/optimizewrappers.py:9-70) give env by env, including the
    history refill when an env finishes and is reset inside the step."""
    import torch
    from custom_envs import load_data
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    from custom_envs_b200.wrappers import DeviceHistoryWrapper, DeviceSubSetWrapper
    data = load_data('iris', 32)
    spec, envs, depth, episode = ProblemSpec('softmax', 4, (), 3), 3, 4, 5
    make = partial(BatchedOptEnv, spec, data.features.astype(np.float32), data.targets.argmax(1), envs,
                   batch_size=32, max_batches=episode, max_history=5, seeds=[1, 2, 3], init_seed=7)
    plain, wrapped = make(), DeviceHistoryWrapper(make(), max_history=depth)
    P, dim = plain.num_params, plain.obs_dim
    ring = np.repeat(plain.reset().cpu().numpy()[None], depth, axis=0)          # [depth, rows, dim]
    got = wrapped.reset()
    assert tuple(got.shape) == (envs * P, depth, dim)
    np.testing.assert_array_equal(got.cpu().numpy(), ring.transpose(1, 0, 2))
    gen = torch.Generator(device=plain.device)
    gen.manual_seed(0)
    for t in range(2 * episode + 1):
        actions = torch.rand(plain.num_rows, device=plain.device, generator=gen) * 3
        obs, _, done, _ = plain.step(actions)
        got, _, done_w, _ = wrapped.step(actions)
        obs, done = obs.cpu().numpy(), done.cpu().numpy().astype(bool)
        assert np.array_equal(done, done_w.cpu().numpy().astype(bool))
        assert done.all() == ((t + 1) % episode == 0)
        ring = np.concatenate([obs[None], ring[:-1]], axis=0)                    # newest first
        for e in np.flatnonzero(done):                                           # wrapper.reset() of that env
            ring[:, e * P:(e + 1) * P] = obs[e * P:(e + 1) * P]
        np.testing.assert_array_equal(got.cpu().numpy(), ring.transpose(1, 0, 2))
    # subset: rows of the named agents, env by env, in the order given
    names = ['parameter-%d' % i for i in (12, 0, 7)]
    sub = DeviceSubSetWrapper(make(), names)
    rows_sorted = sorted('parameter-%d' % i for i in range(P))
    full = sub.env.reset().cpu().numpy().copy()
    picked = sub.reset().cpu().numpy()
    want = np.stack([full[e * P + rows_sorted.index(n)] for e in range(envs) for n in names])
    np.testing.assert_array_equal(picked, want)
    step_full = sub.step(torch.ones(plain.num_rows, device=plain.device))[0].cpu().numpy()
    want = np.stack([sub.env.obs.cpu().numpy()[e * P + rows_sorted.index(n)] for e in range(envs) for n in names])
    np.testing.assert_array_equal(step_full, want)
    for env in (plain, wrapped, sub):
        env.close()


def test_device_rollout_matches_a_manual_loop():
    """Policy in the loop on the device: chunked policy evaluation + env.step equals the same
    loop written out with whole-matrix policy calls."""
    import torch
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy, device_rollout
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(150, 4)).astype(np.float32)
    labels = (np.arange(150) % 3).astype(np.int32)
    torch.manual_seed(0)
    policy = SharedMlpPolicy(15).to('cuda:0')
    mean_only = lambda obs: policy.pi(obs).squeeze(-1)            # noqa: E731 (deterministic)
    results = []
    for chunked in (True, False):
        env = BatchedOptEnv(ProblemSpec('softmax', 4, (), 3), feats, labels, 8, batch_size=32,
                            max_batches=6, seeds=list(range(8)), init_seed=5)
        env.reset()
        if chunked:
            seen = []
            returns, finished = device_rollout(env, mean_only, 7, row_chunk=32,
                                               on_step=lambda t, o, r, d, i: seen.append(o.clone()))
            results.append((returns.cpu().numpy(), finished, seen[-1].cpu().numpy()))
        else:
            returns, finished, obs = torch.zeros(8, dtype=torch.float64, device='cuda:0'), 0, env.obs
            with torch.no_grad():
                for _ in range(7):
                    obs, reward, done, _ = env.step(mean_only(obs).clamp(-4.0, 6.0))
                    returns += reward
                    finished += int(done.sum())
            results.append((returns.cpu().numpy(), finished, obs.cpu().numpy()))
        env.close()
    assert results[0][1] == results[1][1] == 8            # every env ended once (max_batches=6)
    assert np.allclose(results[0][0], results[1][0], rtol=1e-6)
    assert np.allclose(results[0][2], results[1][2], rtol=1e-5, atol=1e-6)


def test_device_episode_monitor_in_a_device_rollout(tmp_path):
    """Episode bookkeeping on the device next to a host replay of the same steps: reward sums,
    lengths (max_batches), the terminal `loss` info and the CSV the reference's tools read."""
    import pandas as pd
    import torch
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy, device_rollout
    from custom_envs_b200.wrappers.device_monitor import DeviceEpisodeMonitor
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(150, 4)).astype(np.float32)
    labels = (np.arange(150) % 3).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 4, (), 3), feats, labels, 16, batch_size=32,
                        max_batches=5, seeds=list(range(16)), init_seed=2)
    env.reset()
    torch.manual_seed(1)
    policy = SharedMlpPolicy(env.obs_dim).to(env.device)
    monitor = DeviceEpisodeMonitor(env.num_envs, str(tmp_path / 'run'), info_keywords=('loss', 'batch_loss'),
                                   device=env.device)
    seen = []

    def hook(t, obs, reward, done, info):
        monitor.on_step(t, obs, reward, done, info)
        seen.append((reward.cpu().numpy().copy(), done.cpu().numpy().copy(), info.cpu().numpy().copy()))

    device_rollout(env, policy.act, 12, on_step=hook)
    rows = monitor.close()
    env.close()
    assert len(rows) == 16 * 2                           # every env ends at step 5 and 10 (or earlier if it diverges)
    total = np.zeros(16)
    want = {}
    episode = np.ones(16, int)
    for reward, done, info in seen:
        total += reward
        for e in np.nonzero(done)[0]:
            want[(e, episode[e])] = (total[e], int(info[e, 15]), info[e, 0])
            total[e], episode[e] = 0.0, episode[e] + 1
    for row in rows:
        ret, length, loss = want[(row['env'], row['episode'])]
        assert abs(row['r'] - ret) < 1e-4 and row['l'] == length and abs(row['loss'] - loss) < 1e-9
    frame = pd.read_csv(tmp_path / 'run.mon.csv')
    assert list(frame.columns) == sorted(['env', 'r', 'l', 'current_reward', 'episode', 't', 'loss', 'batch_loss'])
    assert len(frame) == len(rows)


def test_integration_training_loop_snippet(tmp_path):
    """INTEGRATION.md section 5 at a small env count: device data set -> env -> policy rollout ->
    episode monitor, nothing on the host until the flush."""
    import warnings
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    from custom_envs_b200.data import load_data
    from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy, device_rollout
    from custom_envs_b200.wrappers.device_monitor import DeviceEpisodeMonitor
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        data = load_data('mnist-test', batch_size=32, device='cuda:0')       # synthetic bytes offline
    assert tuple(data.features.shape) == (10000, 49) and data.num_classes == 10
    env = BatchedOptEnv(ProblemSpec('softmax', 49, (64,), data.num_classes), data.features, data.targets,
                        num_envs=64, batch_size=32, max_batches=6, max_history=5)
    env.reset()
    policy = SharedMlpPolicy(env.obs_dim).to('cuda:0')
    monitor = DeviceEpisodeMonitor(env.num_envs, str(tmp_path / 'monitor'), info_keywords=('loss', 'actions_mean'))
    returns, finished = device_rollout(env, policy.act, steps=13, on_step=monitor.on_step)
    rows = monitor.flush()
    env.close()
    assert finished == len(rows) >= 2 * 64 and all(row['l'] <= 6 for row in rows)
    assert (tmp_path / 'monitor.mon.csv').is_file()


@pytest.mark.parametrize('shape', ['iris', 'mlp'])
def test_step_replayed_from_a_cuda_graph_equals_eager_steps(shape):
    """include/b200env.h promises that b2e_step only enqueues work on the caller's stream (no hidden
    synchronisation or allocation): the step is captured into a CUDA graph and the replays must
    reproduce the eager trajectory bit for bit, episode ends and auto-resets included."""
    import torch
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    rng = np.random.RandomState(0)
    if shape == 'iris':
        spec, rows, envs = ProblemSpec('softmax', 4, (), 3), 150, 64
    else:
        spec, rows, envs = ProblemSpec('softmax', 784, (64,), 10), 512, 6
    feats = rng.uniform(size=(rows, spec.num_features)).astype(np.float32)
    labels = rng.randint(0, spec.num_outputs, rows).astype(np.int32)

    def make():
        env = BatchedOptEnv(spec, feats, labels, envs, batch_size=32, max_batches=5, init_seed=4)
        env.reset()
        return env

    eager, graphed = make(), make()
    actions = torch.rand(eager.num_rows, device=eager.device, generator=torch.Generator(device=eager.device).manual_seed(9)) * 3
    static = actions.clone()
    graph, period = graphed.capture_step_graph(static)
    assert period == (1 if shape == 'iris' else 2)
    warm = period                                   # capture_step_graph ran `period` warm-up steps
    for _ in range(warm):
        eager.step(actions)
    for replay in range(6):
        graph.replay()
        for _ in range(period):
            obs, reward, done, info = eager.step(actions)
        torch.cuda.synchronize()
        assert torch.equal(graphed.obs, obs) and torch.equal(graphed.reward, reward), (shape, replay)
        assert torch.equal(graphed.done, done)
        assert torch.allclose(graphed.info, info, rtol=0, atol=0, equal_nan=True)
    assert torch.equal(graphed.get_state('params'), eager.get_state('params'))
    eager.close()
    graphed.close()


class _RunnerStandIn:
    """The slice of stable-baselines' on-policy algorithms the reference scripts exercise (PPO2 / A2C
    ``learn`` and ``predict``; stable_baselines/ppo2/ppo2.py Runner.run): n_steps of
    ``env.step(actions)`` with actions [num_envs, 1], rollout lists that keep every step's arrays WITHOUT
    copying them, the episode-info buffer fed from ``info.get('episode')``, and the ``callback(locals,
    globals)`` hook.  No learning: the scripts' contract with the env is what is under test."""

    def __init__(self, policy, env, gamma=0.99, learning_rate=1e-3, verbose=0, nminibatches=4, n_steps=4):
        assert env.num_envs % nminibatches == 0          # ppo2.py: n_batch % nminibatches
        self.env, self.n_steps = env, n_steps
        self.observation_space, self.action_space = env.observation_space, env.action_space
        self.rng = np.random.RandomState(0)
        self.ep_infos, self.rollouts = [], []

    def predict(self, observation, state=None, mask=None, deterministic=False):
        observation = np.asarray(observation).reshape((-1,) + self.observation_space.shape)
        assert observation.shape[0] == self.env.num_envs
        actions = self.rng.uniform(0.0, 2.0, size=(self.env.num_envs,) + self.action_space.shape)
        return np.clip(actions, self.action_space.low, self.action_space.high).astype(np.float32), None

    def learn(self, total_timesteps, callback=None):
        env = self.env
        obs = np.zeros((env.num_envs,) + self.observation_space.shape, dtype=self.observation_space.dtype)
        obs[:] = env.reset()
        dones = [False] * env.num_envs
        for update in range(1, total_timesteps // (env.num_envs * self.n_steps) + 1):
            mb_obs, mb_rewards, mb_dones = [], [], []
            for _ in range(self.n_steps):
                actions, _ = self.predict(obs)
                mb_obs.append(obs.copy())
                mb_dones.append(dones)
                obs[:], rewards, dones, infos = env.step(actions)
                for info in infos:
                    maybe = info.get('episode')
                    if maybe:
                        self.ep_infos.append(maybe)
                mb_rewards.append(rewards)
            self.rollouts.append((np.asarray(mb_obs), np.asarray(mb_rewards), np.asarray(mb_dones[1:] + [dones])))
            if callback is not None and callback(locals(), globals()) is False:
                break
        return self


def test_script_call_sites_of_survey_8b(tmp_path):
    """SURVEY 8b "who calls it", one call site after the other, against the device-backed classes reached
    through the reference's own module paths (the scripts themselves need stable-baselines / TF / optuna,
    absent here; ``_RunnerStandIn`` restates the runner's side of the contract):

    * run_multiagent_exp_single.py:30-49   OptVecEnv(envs), nminibatches=dummy_env.num_envs, learn, close
    * search_optimize_hyperparam.py:27-62, 95-112   Monitor(partial(gym.make, ...), path, info_keywords, chunk_size),
      dummy_env.agent_no_list[0], env_method('get_episode_rewards') from the learn callback
    * eval_multiexp.py:70-92   gym.make(env_name, **kwargs), states = vec_env.reset(), model.predict(states),
      rewards[0], infos[0] extended in place by the caller
    * play_optimize.py:79-98   reset / predict / step until any(dones), close (twice: the finally block)
    * compile_exp.py:8-28      the .mon.csv the Monitor leaves behind"""
    from custom_envs.vectorize.optvecenv import OptVecEnv
    from custom_envs.utils.utils_logging import Monitor
    from custom_envs import load_data
    import custom_envs_b200.compat as compat
    gym_make = compat.make                                    # `gym.make` of the scripts (stand-in registry or real gym)
    data = load_data('iris', 32)
    kwargs = dict(problem='nn', max_batches=6, problem_kwargs=dict(layers=(), data_set=data))
    keys = ('loss', 'actions_mean', 'weights_mean', 'actions_std', 'states_mean', 'grads_mean')
    log_path = str(tmp_path / 'monitor_{:d}')
    wrapped_envs = [partial(Monitor, partial(gym_make, 'MultiOptLRs-v0', **kwargs), log_path.format(i),
                            info_keywords=keys, chunk_size=5) for i in range(2)]

    # ---- search_optimize_hyperparam.py / run_multiagent_exp_single.py: train
    dummy_env = OptVecEnv(wrapped_envs)
    assert dummy_env.is_device_backed
    model = _RunnerStandIn('MlpPolicy', dummy_env, gamma=0.99, learning_rate=1e-3, verbose=1,
                           nminibatches=dummy_env.num_envs)
    assert dummy_env.num_envs == 30 and dummy_env.agent_no_list[0] == 15
    timesteps = 20 * dummy_env.agent_no_list[0] * 2           # total_timesteps * agent_no_list[0], two envs
    totals = []

    def get_total_reward(environment):                        # search_optimize_hyperparam.py:27-33
        return sum(sum(r) for r in environment.env_method('get_episode_rewards'))

    def callback(local_vars, global_vars):
        totals.append(get_total_reward(local_vars['self'].env))

    model.learn(total_timesteps=timesteps, callback=callback)
    assert len(model.rollouts) == 5 and len(totals) == 5      # 600 timesteps / (30 rows x 4 steps)
    # 20 steps at max_batches = 6: three finished episodes per env, each reported once per agent row
    assert len(model.ep_infos) == 20 * 30 and all(set(e) >= {'r', 'l'} for e in model.ep_infos)
    assert totals[-1] != 0 and totals == sorted(totals, key=lambda v: totals.index(v))
    for mb_obs, mb_rewards, mb_dones in model.rollouts:      # kept arrays were not overwritten by later steps
        assert mb_obs.shape == (4, 30, 15) and mb_rewards.shape == (4, 30) and mb_dones.shape == (4, 30)
        assert len({tuple(r) for r in mb_rewards}) == 4       # four distinct steps, not four aliases of the last
    dummy_env.close()
    dummy_env.close()                                         # idempotent (concurrentvecenv.py:112-122)
    frame = pd.read_csv(log_path.format(0) + '.mon.csv')      # compile_exp.py / eval_csv.py read these
    assert len(frame) == 3 and set(keys) | {'r', 'l', 't'} <= set(frame.columns) and list(frame['l']) == [6, 6, 6]

    # ---- eval_multiexp.py:70-92: one env, the caller extends infos[0]
    env = partial(gym_make, 'MultiOptLRs-v0', **dict(kwargs, max_batches=4))
    vec_env = OptVecEnv([env])
    model = _RunnerStandIn('MlpPolicy', vec_env, nminibatches=1)
    states = vec_env.reset()
    info_list, cumulative_reward = [], 0
    for step in range(6):
        actions = model.predict(states, deterministic=False)[0]
        states, rewards, _, infos = vec_env.step(actions)
        cumulative_reward = cumulative_reward + rewards[0]
        info = infos[0]
        info['step'] = step
        info['cumulative_reward'] = cumulative_reward
        info_list.append(info)
    assert [i['step'] for i in info_list] == list(range(6))   # each step handed out its own dict
    assert all(set(orc.INFO_KEYS) <= set(i) for i in info_list)
    assert [i['loss'] is not None for i in info_list] == [False, False, False, True, False, False]
    assert np.isfinite(cumulative_reward)

    # ---- play_optimize.py:79-98: until any(dones)
    observations = vec_env.reset()
    done, steps = False, 0
    while not done:
        action = model.predict(observations)
        observations, rewards, dones, infos = vec_env.step(action[0])
        done = any(dones)
        steps += 1
    assert steps == 4 and np.all(observations == -1)          # the auto-reset observation (concurrentvecenv.py:32-38)
    vec_env.close()


def test_bench_line_carries_the_contract(tmp_path):
    """`python bench.py` at a reduced env count: stdout is ONE JSON line with the keys the driver and the judge read
    (metric, value, roofline against the measured peak, cpu_baseline, e2e with its copy volumes, gpu_launches, clocks),
    the sampled oracle parity of the same run and the device policy loop; --dump-outputs writes the outputs of the
    last timed step."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--envs', '96', '--steps', '6', '--warmup', '3',
                          '--e2e-steps', '2', '--skip-faithful', '--cpu-steps', '2', '--dump-outputs', str(tmp_path / 'out')],
                         capture_output=True, text=True, cwd=root, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline', 'cpu_baseline',
                'parity', 'policy_loop'):
        assert key in line, key
    assert line['metric'] == 'env-steps/sec' and line['n_gpus'] == 1 and line['steps'] == 6 and line['dtype'] == 'f32'
    assert line['higher_is_better'] is True and line['vs_baseline'] is None and line['data'] == 'synthetic'
    assert abs(line['value'] - 96 * 1e3 / line['ms_per_step']) < 1e-6 * line['value']
    roof = line['roofline']
    assert roof['bound'] == 'hbm' and roof['unit'] == 'GB/s' and abs(roof['frac'] - roof['achieved'] / roof['peak']) < 1e-9
    assert {k['name'] for k in roof['kernels']} == {'eval_kernel<w_prev>', 'update_kernel', 'eval_kernel<w_new>', 'obs_kernel'}
    e2e = line['e2e']
    assert e2e['h2d_bytes_per_step'] == 96 * 50890 * 4 and e2e['d2h_bytes_per_step'] > 96 * 50890 * 15 * 4 and e2e['value'] > 0
    assert line['gpu_launches'] >= 5 * 6
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1 and line['cpu_baseline']['value'] > 0
    assert line['parity']['ok'] is True and line['parity']['done_equal'] is True
    assert line['policy_loop']['value'] > 0 and 'error' not in line['policy_loop']
    assert line['config']['episode_end_in_window']['envs_done'] == 96
    dumped = {name[:-4]: np.load(tmp_path / 'out' / name) for name in os.listdir(tmp_path / 'out')}
    assert set(dumped) == {'obs', 'reward', 'done', 'info', 'info_nonfinite'}
    assert dumped['obs'].dtype == np.float32 and dumped['obs'].shape == (1 << 18, 15)        # sampled rows of [96 * 50890, 15]
    assert dumped['reward'].dtype == np.float32 and dumped['reward'].shape == (96,) and np.isfinite(dumped['reward']).all()
    assert dumped['info'].dtype == np.float64 and dumped['info'].shape == (96, 16)
    assert all(np.isfinite(a).all() for a in dumped.values())
    codes = dumped['info_nonfinite']
    assert codes.dtype == np.float32 and codes.shape == (96, 16) and set(np.unique(codes)) <= {0, 1, 2, 3}
    assert (codes[:, 0] == 1).all()                  # the loss is NaN (the reference's None) where no episode ended
    assert not dumped['info'][codes != 0].any()
    assert dumped['done'].dtype == np.float32 and dumped['done'].shape == (96,)
    assert not dumped['done'].any()                  # the last of the 6 timed steps, not the episode end at step 3
    assert sum(a.nbytes for a in dumped.values()) <= 64 << 20
