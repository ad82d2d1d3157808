"""GPU tests of the device PPO2 (custom_envs_b200.ppo2): learn against the hand-written loop of device_ppo_rollout +
device_ppo_update, seeds, the Monitor bookkeeping of the reference's OptVecEnv chain, callbacks that stop training,
predict, save / load and process groups."""
import multiprocessing
from functools import partial

import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import torch.distributed as dist

    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations
    from custom_envs_b200.ppo2 import PPO2, MlpPolicy, frac_of, tf_adam, update_seeds
    from custom_envs_b200.sharding import shard_range
    from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer, device_ppo_rollout,
                                                          device_ppo_update, reference_actions)
    from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy


def mlp_env(num_envs=3, first=0, device='cuda:0'):
    """The config-4 problem shape (MLP 784-64-10): the env keeps rings, and writes no rows."""
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(320, 784)).astype(np.float32)
    labels = rng.randint(0, 10, 320).astype(np.int32)
    return BatchedOptEnv(ProblemSpec('softmax', 784, (64,), 10), feats, labels, num_envs, batch_size=32,
                         max_batches=5, max_history=5, seeds=list(range(first, first + num_envs)), init_seed=9,
                         materialize_obs=False, device=device, env_base=first)


def iris_env(num_envs=4):
    """A small problem (softmax 4 -> 3, P = 15): dense observation rows only."""
    rng = np.random.RandomState(1)
    feats = rng.uniform(size=(150, 4)).astype(np.float32)
    labels = (np.arange(150) % 3).astype(np.int32)
    return BatchedOptEnv(ProblemSpec('softmax', 4, (), 3), feats, labels, num_envs, batch_size=32, max_batches=5,
                         perms=env_permutations(150, list(range(num_envs))), init_seed=3)


def params_of(model):
    return [p.detach().clone() for p in model.model.parameters()]


def LR(frac):
    return 3e-4 * frac


def CLIP(frac):
    return 0.1 + 0.1 * frac


def hand_loop(env, initial, seed, n_updates, T, low, high, ring_only, cliprange_vf):
    """INTEGRATION section 6's loop with PPO2's seeds, optimizer and schedules."""
    env.reset()
    model = SharedMlpPolicy(env.obs_dim).cuda()
    model.load_state_dict(initial)
    policy = DevicePolicy.from_torch(model, low=low, high=high)
    buf = DeviceRolloutBuffer(env, T)
    opt = tf_adam(model.parameters(), LR(1.0))
    for update in range(1, n_updates + 1):
        frac = frac_of(update, n_updates)
        for group in opt.param_groups:
            group['lr'] = LR(frac)
        rollout_seed, permutation_seed = update_seeds(seed, update)
        device_ppo_rollout(env, policy, buf, ring_only=ring_only, seed=rollout_seed)
        device_ppo_update(model, policy, buf, opt, n_epochs=4, n_minibatches=4, cliprange=CLIP(frac),
                          cliprange_vf=cliprange_vf, seed=permutation_seed)
    policy.close()
    return [p.detach().clone() for p in model.parameters()]


@pytest.mark.parametrize('source', ['rings', 'dense'])
def test_learn_equals_the_hand_loop(source):
    make = mlp_env if source == 'rings' else iris_env
    T, cliprange_vf = 4, (None if source == 'rings' else 0.15)
    env = make()
    model = PPO2(MlpPolicy, env, n_steps=T, learning_rate=LR, cliprange=CLIP, cliprange_vf=cliprange_vf, seed=11)
    initial = {k: v.detach().clone() for k, v in model.model.state_dict().items()}
    model.learn(3 * model.n_batch)
    assert model._ring_only == (source == 'rings')
    assert model.num_timesteps == 3 * model.n_batch
    want = hand_loop(make(), initial, 11, 3, T, model.action_low, model.action_high, source == 'rings', cliprange_vf)
    got = params_of(model)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    assert not all(torch.equal(a, initial[k]) for a, k in zip(got, model.model.state_dict()))


def test_seeds_decide_the_run():
    runs = []
    for seed in (5, 5, 6):
        model = PPO2('MlpPolicy', iris_env(), n_steps=4, seed=seed)
        model.learn(2 * model.n_batch)
        runs.append(params_of(model))
    assert all(torch.equal(a, b) for a, b in zip(runs[0], runs[1]))
    assert not any(torch.equal(a, b) for a, b in zip(runs[0], runs[2]) if a.numel() > 1)


def test_monitor_rows_are_the_rollouts_rewards(tmp_path):
    """The reference's chain: OptVecEnv over Monitor-wrapped MultiOptLRs.  The .mon.csv rows and get_episode_rewards
    are the per-env sums of buffer.rewards over the rollouts, and a legacy callback sees them grow."""
    from custom_envs.utils.utils_logging import Monitor
    from custom_envs.vectorize.optvecenv import OptVecEnv
    from custom_envs import load_data
    from custom_envs_b200.compat import make
    data = load_data('iris', 32)
    fns = [partial(Monitor, partial(make, 'MultiOptLRs-v0', problem='nn', max_batches=5,
                                    problem_kwargs=dict(layers=(), data_set=data)),
                   str(tmp_path / ('env%d' % i)), info_keywords=('loss',)) for i in range(3)]
    vec = OptVecEnv(fns)
    model = PPO2(MlpPolicy, vec, n_steps=5, nminibatches=5, seed=2, verbose=1)
    assert model.n_envs == 45 and model.n_batch == 225
    rollouts, totals = [], []

    class Keep:
        def on_rollout_end(self):
            rollouts.append((model.buffer.rewards.cpu().numpy().copy(), model.buffer.dones[1:].cpu().numpy().copy()))

    def search_callback(locals_, globals_):       # search_optimize_hyperparam.py's get_total_reward
        totals.append(sum(sum(r) for r in locals_['self'].env.env_method('get_episode_rewards')))

    model.learn(4 * model.n_batch, callback=[Keep(), search_callback])
    assert len(rollouts) == 4 and len(totals) == 20
    rewards = np.concatenate([r for r, _ in rollouts])
    dones = np.concatenate([d for _, d in rollouts]).astype(bool)
    want = [[] for _ in range(3)]
    for e in range(3):
        total, length = 0.0, 0
        for t in range(rewards.shape[0]):
            total += float(np.float64(rewards[t, e]))
            length += 1
            if dones[t, e]:
                want[e].append((total, length))
                total, length = 0.0, 0
    assert all(len(w) >= 3 for w in want)
    episode_rewards = vec.env_method('get_episode_rewards')
    assert episode_rewards == [[r for r, _ in w] for w in want]
    assert totals[-1] == sum(sum(r for r, _ in w) for w in want)
    assert any('t' in ep for ep in model.ep_info_buf)         # the Monitor's episode dicts of finished episodes
    vec.close()
    for e in range(3):
        frame = pd.read_csv(str(tmp_path / ('env%d.mon.csv' % e)))
        assert list(frame['l']) == [length for _, length in want[e]]
        assert np.allclose(frame['r'], [round(r, 6) for r, _ in want[e]], rtol=0, atol=1e-9)


def test_callback_stops_before_the_update():
    T = 4
    model = PPO2(MlpPolicy, iris_env(), n_steps=T, seed=8)
    calls, seen = [], {}

    def stop_at_ten(locals_, globals_):
        calls.append(1)
        if len(calls) == 10:                       # global step 9: update 3, rollout step 1
            seen['dones'] = locals_['dones'].copy()
            return False
        return None

    model.learn(3 * model.n_batch, callback=stop_at_ten)
    assert len(calls) == 10 and model.num_timesteps == 10 * model.n_envs
    twin = PPO2(MlpPolicy, iris_env(), n_steps=T, seed=8)
    twin.learn(2 * twin.n_batch)
    assert all(torch.equal(a, b) for a, b in zip(params_of(model), params_of(twin)))
    assert seen['dones'].any()                    # max_batches = 5: every env ended at its 10th step
    assert np.array_equal(model.buffer.dones[T].cpu().numpy().astype(bool), seen['dones'])
    model.learn(model.n_batch, reset_num_timesteps=False)
    assert np.array_equal(model.buffer.dones[0].cpu().numpy().astype(bool), seen['dones'])
    assert model.num_timesteps == 10 * model.n_envs + model.n_batch


def test_predict_save_and_load(tmp_path):
    env = iris_env()
    model = PPO2(MlpPolicy, env, n_steps=4, seed=4)
    model.learn(model.n_batch)
    obs = np.random.RandomState(0).normal(size=(300, 15)).astype(np.float32) * 2
    actions, state = model.predict(obs, deterministic=True)
    assert state is None and isinstance(actions, np.ndarray) and actions.shape == (300, 1)
    with torch.no_grad():
        want = reference_actions(model.model.pi, torch.as_tensor(obs, device='cuda'), model.action_low,
                                 model.action_high)
    assert np.abs(actions[:, 0] - want.cpu().numpy()).max() < 5e-3
    on_device, _ = model.predict(torch.as_tensor(obs, device='cuda'), deterministic=True)
    assert on_device.is_cuda and np.array_equal(on_device.cpu().numpy(), actions)
    noisy, _ = model.predict(obs)
    assert not np.array_equal(noisy, actions)
    assert (noisy >= model.action_low).all() and (noisy <= model.action_high).all()

    model.save(str(tmp_path / 'model.pkl'))
    loaded = PPO2.load(str(tmp_path / 'model.pkl'))
    assert loaded.n_steps == 4 and loaded.obs_dim == 15 and loaded.env is None
    assert np.array_equal(loaded.predict(obs, deterministic=True)[0], actions)
    for name, value in model.get_parameters().items():
        assert np.array_equal(loaded.get_parameters()[name], value), name
    with_env = PPO2.load(str(tmp_path / 'model.pkl'), env=iris_env(), n_steps=8)
    assert with_env.n_steps == 8 and np.array_equal(with_env.predict(obs, deterministic=True)[0], actions)

    params = model.get_parameters()
    params['model/pi/b:0'] = np.array([2e4], np.float32)           # a mean beyond the Box: clipped to its high end
    loaded.load_parameters(params)
    assert (loaded.predict(obs, deterministic=True)[0] == np.float32(model.action_high)).all()
    assert (loaded.predict(obs)[0] <= model.action_high).all()


def test_rejects_the_host_fallback_env():
    from custom_envs_b200.vectorize.optvecenv import OptVecEnv

    vec = OptVecEnv.__new__(OptVecEnv)
    vec._wrapped = None                          # what the constructor sets on the thread-per-env fallback
    assert not vec.is_device_backed
    with pytest.raises(ValueError, match='host fallback'):
        PPO2(MlpPolicy, vec)
    with pytest.raises(ValueError, match='BatchedOptEnv'):
        PPO2(MlpPolicy, object())


# ------------------------------------------------------------------ process groups
E_TOTAL = 4


def train(rank, world, group):
    first, count = shard_range(E_TOTAL, world, rank)
    env = mlp_env(count, first, device='cuda:%d' % rank)
    model = PPO2(MlpPolicy, env, n_steps=4, seed=100 + rank, group=group)   # rank 0's seed is used everywhere
    model.learn(2 * model.n_batch)
    return [p.cpu() for p in params_of(model)], model.num_timesteps


def _worker(rank, world, store, out):
    device = torch.device('cuda', rank)
    torch.cuda.set_device(device)
    dist.init_process_group('nccl', init_method='file://' + store, rank=rank, world_size=world, device_id=device)
    try:
        torch.save(train(rank, world, dist.group.WORLD), out % rank)
    finally:
        dist.destroy_process_group()


def spawn_ranks(world, tmp_path, timeout=600):
    ctx = multiprocessing.get_context('spawn')
    store, out = str(tmp_path / 'store'), str(tmp_path / 'rank%d.pt')
    procs = [ctx.Process(target=_worker, args=(r, world, store, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout)
    alive = [p for p in procs if p.is_alive()]
    for p in alive:
        p.kill()
        p.join()
    assert not alive, 'ranks did not finish within %d s' % timeout
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    return [torch.load(out % r, weights_only=False) for r in range(world)]


@pytest.mark.skipif(not (torch.cuda.is_available() and dist.is_nccl_available()), reason='needs NCCL')
def test_one_rank_group_equals_no_group(tmp_path):
    (got,) = spawn_ranks(1, tmp_path)
    want = train(0, 1, None)
    assert got[1] == want[1]
    assert all(torch.equal(a, b) for a, b in zip(got[0], want[0]))


@pytest.mark.skipif(torch.cuda.device_count() < 2 or not dist.is_nccl_available(), reason='needs two GPUs and NCCL')
def test_two_ranks_stay_identical(tmp_path):
    ranks = spawn_ranks(2, tmp_path)
    assert ranks[0][1] == ranks[1][1] == 2 * 4 * E_TOTAL * ProblemSpec('softmax', 784, (64,), 10).size
    assert all(torch.equal(a, b) for a, b in zip(ranks[0][0], ranks[1][0]))
