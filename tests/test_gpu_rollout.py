"""GPU tests of PPO rollouts on the device: the step kernel (b2p_step / b2p_step_env: value tower, raw actions,
neglogp, bf16 observation store), the GAE kernel (b2p_gae), DeviceRolloutBuffer and device_ppo_rollout.

The clipped actions of a step launch are the action-only kernel's, bit for bit; the value tower is held to a
bf16-rounded torch evaluation like the action tower in test_gpu_policy.py; GAE to a numpy restatement of the
stable-baselines 2 PPO2 Runner."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from custom_envs_b200._lib import B200EnvError
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations
    from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer, device_ppo_rollout, gae,
                                                          reference_values)
    from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy

LOG_STD = -0.5


def make_policy(obs_dim, seed, scale=1.0):
    torch.manual_seed(seed)
    policy = SharedMlpPolicy(obs_dim).cuda()
    with torch.no_grad():
        for tower in (policy.pi, policy.vf):
            for p in tower.parameters():
                p.mul_(scale)
            for m in tower.modules():
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.3, 0.3)
    return policy


def small_env(num_envs=3, max_batches=6, row_order='lexicographic', materialize_obs=True, max_history=5, hidden=(64,)):
    """The config-4 problem shape (MLP 784-64-10) on a small data set, as in test_gpu_policy.py; hidden = () is the
    resident-minibatch pipeline."""
    rng = np.random.RandomState(0)
    rows = 320
    feats = rng.uniform(size=(rows, 784)).astype(np.float32)
    labels = rng.randint(0, 10, rows).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 784, tuple(hidden), 10), feats, labels, num_envs, batch_size=32,
                        max_batches=max_batches, max_history=max_history, row_order=row_order,
                        perms=env_permutations(rows, list(range(num_envs))), init_seed=9,
                        materialize_obs=materialize_obs)
    env.reset()
    return env


def iris_env(num_envs=4, max_batches=3):
    rng = np.random.RandomState(1)
    feats = rng.uniform(size=(150, 4)).astype(np.float32)
    labels = (np.arange(150) % 3).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 4, (), 3), feats, labels, num_envs, batch_size=32, max_batches=max_batches,
                        perms=env_permutations(150, list(range(num_envs))))
    env.reset()
    return env


def obs_store(rows):
    return torch.empty((rows, 16), dtype=torch.bfloat16, device='cuda')


def runner_gae(values, rewards, dones, P, gamma, lam):
    """stable-baselines 2 PPO2 Runner.run (ppo2.py), the advantage loop over per-row arrays, in its own dtypes:
    float32 values / rewards, bool dones, `1.0 - dones` float64, last_gae_lam float64, mb_advs float32.
    Parity unpinned: stable-baselines is not installed here, this restates its code."""
    T = rewards.shape[0]
    mb_rewards = np.repeat(rewards, P, axis=1).astype(np.float32)
    all_dones = np.repeat(dones, P, axis=1).astype(bool)
    mb_values, last_values = values[:T].astype(np.float32), values[T].astype(np.float32)
    mb_dones, final_dones = all_dones[:T], all_dones[T]
    mb_advs = np.zeros_like(mb_rewards)
    last_gae_lam = 0
    for step in reversed(range(T)):
        if step == T - 1:
            nextnonterminal = 1.0 - final_dones
            nextvalues = last_values
        else:
            nextnonterminal = 1.0 - mb_dones[step + 1]
            nextvalues = mb_values[step + 1]
        delta = mb_rewards[step] + gamma * nextvalues * nextnonterminal - mb_values[step]
        mb_advs[step] = last_gae_lam = delta + gamma * lam * nextnonterminal * last_gae_lam
    mb_returns = mb_advs + mb_values
    return mb_advs, mb_returns


def assert_close_ulp(got, want):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    ulp = np.spacing(np.abs(want))
    assert np.all((np.abs(got - want) <= 1e-6 * np.abs(want)) | (np.abs(got - want) <= ulp)), \
        np.abs(got - want).max()


# ------------------------------------------------------------------ step kernel, dense front end
@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
@pytest.mark.parametrize('obs_dim,rows', [(15, 128 * 9), (15, 1), (3, 257), (9, 4321), (15, 100003)])
def test_dense_step_matches_act_and_torch(obs_dim, rows, tanh_mode):
    policy = make_policy(obs_dim, seed=obs_dim + rows)
    gen = torch.Generator(device='cuda').manual_seed(rows)
    obs = torch.randn(rows, obs_dim, device='cuda', generator=gen)
    obs[::7] *= 10.0
    obs[::13, 0] = 99.0
    obs[::17, -1] = -101.0
    low, high = -1.0, 1.5
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD), tanh_mode=tanh_mode, low=low, high=high)
    assert dev.has_value
    store = obs_store(rows)
    actions, raw, values, neglogp, _ = dev.step(obs, seed=7, obs_bf16=store)
    # the clipped actions are the action-only kernel's
    assert torch.equal(actions, dev.act(obs, seed=7))
    assert torch.equal(raw.clamp(low, high), actions)
    # value tower against torch
    want = reference_values(policy.vf, obs)
    exact = reference_values(policy.vf, obs, bf16=False)
    scale = max(1.0, policy.vf[-1].weight.abs().sum().item())
    tol = (2e-3 if tanh_mode == 0 else 1.5e-2) * scale
    assert (values - want).abs().max().item() <= tol
    assert (values - exact).abs().max().item() <= 0.1 * scale
    # neglogp of the raw action under N(mean, std)
    quiet = DevicePolicy.from_torch(policy.pi, tanh_mode=tanh_mode, low=-1e9, high=1e9)
    mean = quiet.act(obs).double()
    std = math.exp(LOG_STD)
    nlp = 0.5 * ((raw.double() - mean) / std) ** 2 + 0.5 * math.log(2 * math.pi) + LOG_STD
    assert (neglogp.double() - nlp).abs().max().item() <= 1e-5
    # observation store: the bf16 row, zero padding
    assert torch.equal(store[:, :obs_dim], obs.to(torch.bfloat16))
    assert not store[:, obs_dim:].float().abs().sum().item()
    # model.value: the value tower alone gives the same bits
    assert torch.equal(dev.value(obs), values)
    dev.close()
    quiet.close()


def test_step_output_subsets_and_errors():
    policy = make_policy(15, seed=3)
    obs = torch.randn(5000, 15, device='cuda')
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD))
    actions, raw, values, neglogp, _ = dev.step(obs, seed=3)
    parts = {name: torch.empty(5000, device='cuda') for name in ('actions', 'actions_raw', 'neglogp')}
    dev._launch(obs, dev._seed(3), **parts)                     # the action tower alone
    assert torch.equal(parts['actions'], actions) and torch.equal(parts['actions_raw'], raw)
    assert torch.equal(parts['neglogp'], neglogp)
    store = obs_store(5000)
    dev._launch(obs, dev._seed(3), obs_bf16=store)              # no tower at all
    assert torch.equal(store[:, :15], obs.to(torch.bfloat16))
    with pytest.raises(B200EnvError, match='every output is NULL'):
        dev._launch(obs, dev._seed(3))
    pi_only = DevicePolicy.from_torch(policy.pi, log_std=torch.tensor(LOG_STD))
    assert not pi_only.has_value and pi_only.step(obs, seed=3)[2] is None
    with pytest.raises(B200EnvError, match='b2p_set_value_weights'):
        pi_only.value(obs)
    with pytest.raises(B200EnvError, match='multiple of P'):
        gae(torch.zeros(2, 10, device='cuda'), torch.zeros(1, 3, device='cuda'),
            torch.zeros(2, 3, dtype=torch.uint8, device='cuda'), 3)
    dev.close()
    pi_only.close()


def test_log_std_change_reaches_noise_and_neglogp():
    """PPO trains log_std: after set_log_std the step samples with the new std and scores with the new log_std."""
    policy = make_policy(15, seed=8)
    obs = torch.randn(20000, 15, device='cuda')
    dev = DevicePolicy.from_torch(policy, low=-1e9, high=1e9)
    assert dev.log_std == pytest.approx(policy.log_std.item())
    quiet = DevicePolicy.from_torch(policy.pi, low=-1e9, high=1e9)
    mean = quiet.act(obs).double()
    before = dev.step(obs, seed=5)
    new_log_std = 0.3
    dev.set_log_std(torch.tensor(new_log_std))
    _, raw, _, neglogp, _ = dev.step(obs, seed=5)
    std = math.exp(new_log_std)
    z = (raw.double() - mean) / std
    assert torch.allclose(z, (before[1].double() - mean) / math.exp(policy.log_std.item()), atol=1e-4)   # same draw
    nlp = 0.5 * z ** 2 + 0.5 * math.log(2 * math.pi) + new_log_std
    assert (neglogp.double() - nlp).abs().max().item() <= 1e-5
    dev.set_log_std(None)
    assert torch.equal(dev.act(obs, seed=5), quiet.act(obs, seed=5))
    dev.close()
    quiet.close()


# ------------------------------------------------------------------ step kernel, ring front end
@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
@pytest.mark.parametrize('row_order,depth', [('lexicographic', 5), ('natural', 5), ('lexicographic', 3), ('natural', 1)])
def test_ring_step_equals_dense_step(row_order, depth, tanh_mode):
    """b2p_step_env on the rings equals b2p_step on the observation rows of the same step in all five outputs, from
    the reset observation through an auto-reset (max_batches = 6, 8 steps); depth 5 is the constant-index ring front
    end, 3 and 1 the run-time-depth one."""
    env = small_env(row_order=row_order, max_history=depth)
    policy = make_policy(env.obs_dim, seed=1, scale=1.5)
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD), tanh_mode=tanh_mode)
    gen = torch.Generator(device='cuda').manual_seed(0)
    for t in range(8):
        ring = dev.step(env, seed=100 + t, obs_bf16=obs_store(env.num_rows))
        dense = dev.step(env.obs, seed=100 + t, obs_bf16=obs_store(env.num_rows))
        for a, b in zip(ring, dense):
            assert torch.equal(a, b), t
        env.step(torch.rand(env.num_rows, device='cuda', generator=gen) * 2.0)
    assert torch.equal(dev.value(env), dev.value(env.obs))
    dev.close()
    env.close()


# ------------------------------------------------------------------ GAE
@pytest.mark.parametrize('gamma,lam', [(0.99, 0.95), (1.0, 1.0)])
@pytest.mark.parametrize('T', [1, 7, 64])
@pytest.mark.parametrize('P,E', [(1, 1000), (15, 67), (50890, 3)])
def test_gae_matches_the_runner(T, P, E, gamma, lam):
    """b2p_gae against the PPO2 Runner's loop (runner_gae; parity unpinned: a restatement of stable-baselines 2 code
    that is not installed here).  Done flags at the first step, at T and in between."""
    rng = np.random.RandomState(T * 7 + P)
    rows = P * E
    values = (rng.standard_normal((T + 1, rows)) * 3.0).astype(np.float32)
    rewards = rng.standard_normal((T, E)).astype(np.float32)
    dones = (rng.uniform(size=(T + 1, E)) < 0.15).astype(np.uint8)
    dones[0, ::2] = 1
    dones[1, 1::3] = 1                       # done returned by step 0
    dones[T, ::4] = 1                        # done returned by the last step
    want_adv, want_ret = runner_gae(values, rewards, dones, P, gamma, lam)
    adv, ret = gae(torch.as_tensor(values).cuda(), torch.as_tensor(rewards).cuda(), torch.as_tensor(dones).cuda(), P,
                   gamma, lam)
    assert_close_ulp(adv.cpu().numpy(), want_adv)
    assert_close_ulp(ret.cpu().numpy(), want_ret)


# ------------------------------------------------------------------ rollouts
def buffers(buf):
    return [buf.obs_bf16, buf.actions_raw, buf.values, buf.neglogp, buf.advantages, buf.returns, buf.rewards, buf.dones]


@pytest.mark.parametrize('hidden', [(64,), ()], ids=['tcgen05', 'resident-minibatch'])
def test_rollout_on_the_rings_equals_rollout_on_observation_rows(hidden):
    """Two rollouts of 4 steps each (the episodes of max_batches = 5 end inside the second one): every buffer field
    is the same, bit for bit, whether the policy reads the rings (ring-only env steps) or the observation rows."""
    policy = make_policy(15, seed=2, scale=1.5)
    results = []
    for ring_only in (True, False):
        env = small_env(num_envs=4, max_batches=5, materialize_obs=not ring_only, hidden=hidden)
        dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD))
        buf = DeviceRolloutBuffer(env, 4)
        snaps, total = [], 0
        for _ in range(2):
            _, finished = device_ppo_rollout(env, dev, buf, ring_only=ring_only)
            total += finished
            snaps.append([t.clone() for t in buffers(buf)])
        results.append((snaps, total))
        dev.close()
        env.close()
    assert results[0][1] == results[1][1] == 4
    for a, b in zip(results[0][0], results[1][0]):
        for i, (x, y) in enumerate(zip(a, b)):
            assert torch.equal(x, y), i


def test_rollout_buffer_holds_what_the_env_returned():
    """Iris-shaped problem (dense front end only): obs_bf16[t] is the bf16 of the observation before step t,
    rewards / dones the env's outputs, dones[0] of the second rollout the last flags of the first, advantages and
    returns the Runner's GAE of the buffer's own values, rewards and dones."""
    env = iris_env()
    policy = make_policy(env.obs_dim, seed=4, scale=1.5)
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD))
    T = 5
    buf = DeviceRolloutBuffer(env, T)
    for rollout in range(2):
        seen = []
        before = env.obs.clone()
        _, finished = device_ppo_rollout(env, dev, buf, ring_only=False,
                                         on_step=lambda t, o, r, d, i: seen.append((o.clone(), r.clone(), d.clone())))
        assert len(seen) == T
        if rollout == 1:
            assert torch.equal(buf.dones[0], last_flags)
        else:
            assert not buf.dones[0].any()
        for t in range(T):
            obs_t = before if t == 0 else seen[t - 1][0]
            assert torch.equal(buf.obs_bf16[t, :, :env.obs_dim], obs_t.to(torch.bfloat16)), t
            assert torch.equal(buf.rewards[t], seen[t][1]) and torch.equal(buf.dones[t + 1], seen[t][2]), t
        assert finished == int(sum(d.sum().item() for _, _, d in seen))
        last_flags = seen[-1][2]
        # values[T] is model.value of the last observation
        assert torch.equal(buf.values[T], dev.value(env.obs))
        want_adv, want_ret = runner_gae(buf.values.cpu().numpy(), buf.rewards.cpu().numpy(), buf.dones.cpu().numpy(),
                                        env.num_params, 0.99, 0.95)
        assert_close_ulp(buf.advantages.cpu().numpy(), want_adv)
        assert_close_ulp(buf.returns.cpu().numpy(), want_ret)
    assert buf.dones[1:].any()                       # max_batches = 3: episodes ended inside the rollouts
    buf.reset()
    assert not buf.dones.any()
    dev.close()
    env.close()


def test_rollout_buffer_checks_free_memory():
    env = iris_env()
    with pytest.raises(MemoryError, match='n_steps'):
        DeviceRolloutBuffer(env, 10 ** 12)
    env.close()


# ------------------------------------------------------------------ guard bands
def test_step_outputs_stay_inside_their_buffers():
    """Every step output written through a window of a NaN-filled buffer (dense front end at ragged row counts, ring
    front end, a value-only launch; GAE outputs): nothing outside the window changes, nothing inside stays NaN."""
    pad = 1024
    policy = make_policy(15, seed=6)
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD))

    def windows(rows):
        bufs = [torch.full((rows + 2 * pad,), float('nan'), device='cuda') for _ in range(4)]
        store = torch.full(((rows + 2 * pad) * 16,), float('nan'), dtype=torch.bfloat16, device='cuda')
        return bufs, store, [b[pad:pad + rows] for b in bufs], store[pad * 16:(pad + rows) * 16].view(rows, 16)

    def check(bufs, store, rows, which=range(4), with_store=True):
        for i in which:
            b = bufs[i]
            assert torch.isnan(b[:pad]).all() and torch.isnan(b[pad + rows:]).all(), (rows, i)
            assert not torch.isnan(b[pad:pad + rows]).any(), (rows, i)
        if with_store:
            assert torch.isnan(store[:pad * 16]).all() and torch.isnan(store[(pad + rows) * 16:]).all(), rows
            assert not torch.isnan(store[pad * 16:(pad + rows) * 16]).any(), rows

    for rows in (1, 127, 128, 129, 100003):
        obs = torch.randn(rows, 15, device='cuda')
        bufs, store, win, swin = windows(rows)
        dev._launch(obs, dev._seed(1), *win, obs_bf16=swin)
        check(bufs, store, rows)
        bufs, store, win, swin = windows(rows)
        dev.value(obs, out=win[2])
        check(bufs, store, rows, which=[2], with_store=False)
        assert torch.isnan(bufs[0]).all() and torch.isnan(bufs[3]).all()
    env = small_env(num_envs=3, max_batches=3, materialize_obs=False)
    gen = torch.Generator(device='cuda').manual_seed(1)
    for t in range(4):                                         # the third step ends every episode
        bufs, store, win, swin = windows(env.num_rows)
        dev._launch(env, dev._seed(None), *win, obs_bf16=swin)
        check(bufs, store, env.num_rows)
        bufs, store, win, swin = windows(env.num_rows)
        dev.value(env, out=win[2])
        check(bufs, store, env.num_rows, which=[2], with_store=False)
        env.step(torch.rand(env.num_rows, device='cuda', generator=gen) * 2, ring_only=True)
    env.close()
    T, E, P = 3, 5, 77
    rows = E * P
    adv = torch.full((T * rows + 2 * pad,), float('nan'), device='cuda')
    ret = torch.full((T * rows + 2 * pad,), float('nan'), device='cuda')
    gae(torch.randn(T + 1, rows, device='cuda'), torch.randn(T, E, device='cuda'),
        torch.zeros(T + 1, E, dtype=torch.uint8, device='cuda'), P, advantages=adv[pad:pad + T * rows].view(T, rows),
        returns=ret[pad:pad + T * rows].view(T, rows))
    for b in (adv, ret):
        assert torch.isnan(b[:pad]).all() and torch.isnan(b[pad + T * rows:]).all()
        assert not torch.isnan(b[pad:pad + T * rows]).any()
    dev.close()
