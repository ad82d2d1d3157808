"""The Adam baseline on the device (b2e_step_adam / DeviceAdam) against the CPU oracle (tests/adam_oracle.py).

Per-step parity from identical states at the bars of test_gpu_parity.py on every step path: the warp-per-env
kernel (config 2), the fused kernel (Rosenbrock, a small MLP), the large-problem pipeline with the thin3, tcgen05
and generic eval kernels; the kernel that ran is named by the profiler.  These parity runs use epsilon = 1e-3:
with Keras' 1e-7 a gradient component at the level of its own fp32 rounding noise moves its weight by lr * sign(g),
which that noise can flip; a larger epsilon makes the update a smooth function of g there.  The formulas are
the same.  Rosenbrock and iris, whose gradient components stay far above that noise, also run at Keras' 1e-7, and
the device-only tests below run Keras' defaults.
"""
import os
import re
import sys

import numpy as np
import pytest
import torch

from oracle import optenv_oracle as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from adam_oracle import AdamOracle  # noqa: E402
from test_gpu_parity import RTOL, check_info, check_obs, make_data, pole_of, product_spec, rel_err, shift_ill  # noqa: E402

pytestmark = pytest.mark.gpu

EPS = 1e-3

# (id, spec, rows, batch, envs, env overrides, kernel of the Adam update, kernel of the evaluations)
CASES = [
    ('tiny_iris', orc.ProblemSpec('softmax', 4, (), 3), 150, 32, 6, {}, r'tiny_env_kernel<5, 4, 3, [^<>]*AdamArgs>', None),
    ('fused_func', orc.ProblemSpec('func', 0, (), 0), 0, None, 4, {}, r'optenv_kernel<5, false, [^<>]*AdamArgs>', None),
    ('fused_mlp_small', orc.ProblemSpec('softmax', 6, (5,), 3), 50, 16, 3, {}, r'optenv_kernel<5, false, [^<>]*AdamArgs>', None),
    ('thin3_784x10', orc.ProblemSpec('softmax', 784, (), 10), 600, 32, 3, {}, r'update_adam_kernel',
     r'thin3_eval_kernel<true>'),
    ('tc2_784x64x10', orc.ProblemSpec('softmax', 784, (64,), 10), 600, 32, 3, {'B2E_TC_CHECK': '1'},
     r'update_adam_kernel', r'tc2_eval_kernel<true, 10>'),
    ('generic_12x16x8x4', orc.ProblemSpec('softmax', 12, (16, 8), 4), 60, 20, 3, {}, r'update_adam_kernel',
     r'gen_eval_kernel'),
]
BY_ID = {case[0]: case for case in CASES}


def _env(spec, rows, batch, num_envs, data=None, **kwargs):
    from custom_envs_b200.batched_env import BatchedOptEnv
    feats, targs = (None, None) if spec.kind == 'func' else (make_data(spec, rows) if data is None else data)
    return BatchedOptEnv(product_spec(spec), feats, targs, num_envs, batch_size=batch, **kwargs), feats, targs


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA})


@pytest.mark.parametrize('case_id', list(BY_ID) + ['fused_func-keras_eps', 'tiny_iris-keras_eps'])
def test_adam_step_parity_from_identical_states(case_id, monkeypatch):
    """7 steps per case with host-supplied minibatches (one ragged env per step), a learning rate per env;
    after every step the oracle continues from the device's parameters, gradient and moments.  ``-keras_eps``:
    Keras' epsilon of 1e-7 on shapes whose gradient components stay far above their rounding noise."""
    eps = 1e-7 if case_id.endswith('-keras_eps') else EPS
    case_id = case_id.split('-')[0]
    from custom_envs_b200.baselines import DeviceAdam
    _, spec, rows, batch, num_envs, env_vars, update_kernel, eval_kernel = BY_ID[case_id]
    for key in ('B2E_TC', 'B2E_THIN2', 'B2E_FORCE_GENERIC', 'B2E_TINY'):
        monkeypatch.delenv(key, raising=False)
    for key, value in env_vars.items():
        monkeypatch.setenv(key, value)
    func = spec.kind == 'func'
    steps, depth = 7, 5
    env, feats, targs = _env(spec, rows, batch, num_envs, max_batches=steps + 1, index_mode='external',
                             auto_reset=False)
    # Rosenbrock: steps of 1e-3 leave g_t - g_{t-1} (grad_diff) at the level of the fp32 gradients' rounding
    lrs = np.geomspace(5e-2, 2e-1, num_envs) if func else np.geomspace(1e-3, 3e-2, num_envs)
    lrs = lrs.astype(np.float32)
    adam = DeviceAdam(env, torch.as_tensor(lrs, device=env.device), epsilon=eps)
    ref_env = orc.BatchedOptEnvOracle(spec, feats, targs, num_envs, batch_size=batch,
                                      config=orc.EnvConfig.multioptlrs(steps + 1, depth),
                                      perms=None if func else np.tile(np.arange(rows), (num_envs, 1)))
    ref = AdamOracle(ref_env, lrs, epsilon=eps)
    num_params = ref_env.num_params
    perm = orc.lexicographic_rows(num_params)
    rng = np.random.RandomState(3)

    def draw_batch():
        if func:
            return None, None
        idx = rng.randint(0, rows, size=(num_envs, batch)).astype(np.int32)
        cnt = np.full(num_envs, batch, np.int32)
        cnt[rng.randint(num_envs)] = rng.randint(1, batch + 1)
        return idx, cnt

    init = np.stack([orc.glorot_uniform_init(spec, rng) for _ in range(num_envs)])
    idx, cnt = draw_batch()
    if not func:
        ref_env.set_batch(idx, cnt)
    ref_env.reset(init_params=init)
    env.reset(init_params=init, batch_idx=idx, batch_cnt=cnt)
    ref_env.raw_g[0] = env.get_state('grad_prev').cpu().numpy().astype(np.float64)
    ill = np.zeros((num_envs, num_params, 3 * depth), bool)
    pole = np.zeros_like(ill)
    for t in range(steps):
        idx, cnt = draw_batch()
        if not func:
            ref_env.set_batch(idx, cnt)
        prev_w = ref_env.weights.astype(np.float64).copy()
        prev_g = ref_env.raw_g[0].copy()
        ref_obs, ref_rew, ref_done, ref_info = ref.step()
        idx_t = None if func else torch.as_tensor(idx, device=env.device)
        cnt_t = None if func else torch.as_tensor(cnt, device=env.device)
        if t == 0:                            # the Adam kernel ran, and the eval kernel the table names
            names = _kernels(lambda: _step(env, adam, idx_t, cnt_t))
            assert any(re.search(update_kernel, n) for n in names), names
            assert eval_kernel is None or any(re.search(eval_kernel, n) for n in names), names
        else:
            _step(env, adam, idx_t, cnt_t)
        obs, rew, done, info = env.obs, env.reward, env.done, env.info
        tag = (case_id, t)
        obs = obs.cpu().numpy().reshape(num_envs, num_params, -1)
        obs_nat = np.empty_like(obs)
        obs_nat[:, perm] = obs
        assert np.array_equal(done.cpu().numpy().astype(bool), ref_done), tag
        new_g = ref_env.raw_g[0]
        g_rms = np.sqrt(np.mean(new_g ** 2, axis=1, keepdims=True)) + 1e-30
        w_rms = np.sqrt(np.mean(prev_w ** 2, axis=1, keepdims=True)) + 1e-30
        ill = shift_ill(ill, depth, np.maximum(np.abs(prev_w), np.abs(ref_env.weights)) < 1e-2 * w_rms,
                        np.maximum(np.abs(prev_g), np.abs(new_g)) < 1e-2 * g_rms)
        pole = shift_ill(pole, depth, np.zeros_like(prev_w, bool), pole_of(prev_g, new_g))
        check_obs(obs_nat, ref_obs, ill, tag, pole)
        np.testing.assert_allclose(rew.cpu().numpy(), ref_rew, rtol=RTOL, atol=RTOL, err_msg=str(tag))
        new_w = env.get_state('params').cpu().numpy()
        werr = rel_err(new_w, ref_env.weights, np.abs(ref_env.weights).mean())
        assert werr.max() <= RTOL, (tag, float(werr.max()))
        m, v = adam.m.cpu().numpy(), adam.v.cpu().numpy()
        assert rel_err(m, ref.m, np.abs(ref.m).mean(axis=1, keepdims=True) + 1e-30).max() <= RTOL, tag
        root_v, ref_root_v = np.sqrt(v), np.sqrt(ref.v)              # conditioned like g, as m is
        assert rel_err(root_v, ref_root_v, ref_root_v.mean(axis=1, keepdims=True) + 1e-30).max() <= 2 * RTOL, tag
        got = env.info_dict(info)
        check_info(got, ref_info, ref_env, ref_obs, prev_g, num_params, tag)   # actions_*: Adam's rates
        # identical states for the next step
        ref_env.weights = new_w.copy()
        ref_env.raw_w[0] = new_w
        ref_env.raw_g[0] = env.get_state('grad_prev').cpu().numpy().astype(np.float64)
        ref.m, ref.v = m.astype(np.float64), v.astype(np.float64)
    env.close()


def _step(env, adam, idx, cnt):
    """b2e_step_adam with host-supplied minibatch indices (DeviceAdam.step uses the on-device stream)."""
    import ctypes
    from custom_envs_b200.baselines import _ptr
    env._check(env.lib.b2e_step_adam(env.handle, ctypes.byref(adam._opt), _ptr(adam.lr), _ptr(adam.m), _ptr(adam.v),
                                     _ptr(idx), _ptr(cnt), _ptr(env.obs), _ptr(env.reward), _ptr(env.done),
                                     _ptr(env.info), env._stream()))


@pytest.mark.parametrize('case_id', ['tiny_iris', 'fused_mlp_small', 'tc2_784x64x10'])
def test_adam_trajectory_across_epoch_wrap_divergence_and_auto_reset(case_id, monkeypatch):
    """Keras' defaults on the on-device minibatch stream with auto-reset: 30 steps of episodes of 12 steps cross
    epoch wraps and auto-resets, and env 1's learning rate of 1e5 makes it diverge (loss > 1e4: done early).  The
    oracle runs alongside from the same initial weights; every reset env starts t = 1 with m and v overwritten by
    stale non-zero values first, which the step must ignore."""
    from custom_envs_b200.baselines import DeviceAdam
    _, spec, rows, batch, num_envs, env_vars, _, _ = BY_ID[case_id]
    for key, value in env_vars.items():
        monkeypatch.setenv(key, value)
    max_batches, rows = 12, min(rows, 200)                   # epochs shorter than an episode
    env, feats, targs = _env(spec, rows, batch, num_envs, max_batches=max_batches, init_seed=5)
    lrs = np.full(num_envs, 1e-2, np.float32)
    lrs[1] = 1e5
    adam = DeviceAdam(env, torch.as_tensor(lrs, device=env.device))
    perms = np.stack([orc.env_permutation(rows, s) for s in range(num_envs)])
    ref_env = orc.BatchedOptEnvOracle(spec, feats, targs, num_envs, batch_size=batch,
                                      config=orc.EnvConfig.multioptlrs(max_batches), perms=perms)
    ref = AdamOracle(ref_env, lrs)
    env.reset()
    ref_env.reset(init_params=env.get_state('params').cpu().numpy())
    stale_envs, diverged, wrapped = 0, False, False
    for t in range(30):
        last_batch = ref_env.stream.cursor == ref_env.stream.num_batches - 1
        obs, rew, done, info = adam.step()
        ref_obs, ref_rew, ref_done, ref_info = ref.step()
        got = env.info_dict(info)
        tag = (case_id, t)
        assert np.array_equal(done.cpu().numpy().astype(bool), ref_done), tag
        ok = ~ref_done | (ref_info['batch_loss'] < 1e4)           # a diverged env's numbers are not comparable
        np.testing.assert_allclose(got['batch_loss'][ok], ref_info['batch_loss'][ok], rtol=1e-3, err_msg=str(tag))
        np.testing.assert_allclose(rew.cpu().numpy()[ok], ref_rew[ok], rtol=1e-3, atol=1e-3, err_msg=str(tag))
        diverged |= bool(ref_done[1] and ref_env.current_step[1] < max_batches)
        wrapped |= bool(np.any(last_batch & ~ref_done))
        if ref_done.any():
            # the device auto-reset these envs; stale moments must not reach their step t = 1
            mask = torch.as_tensor(ref_done, device=env.device)
            adam.m[mask] = 7.0
            adam.v[mask] = 3.0
            stale_envs += int(ref_done.sum())
            ref_env.reset(ref_done, init_params=env.get_state('params').cpu().numpy())
        # identical states: the oracle takes the device's weights and moments (both continue in fp32 / fp64)
        ref_env.weights = env.get_state('params').cpu().numpy()
        ref.m, ref.v = adam.m.cpu().numpy().astype(np.float64), adam.v.cpu().numpy().astype(np.float64)
        ref_env.raw_g[0] = env.get_state('grad_prev').cpu().numpy().astype(np.float64)
        ref_env.raw_w[0] = ref_env.weights
    assert diverged and wrapped and stale_envs >= num_envs, (diverged, wrapped, stale_envs)
    env.close()


@pytest.mark.parametrize('case_id', ['tiny_iris', 'fused_func', 'fused_mlp_small', 'thin3_784x10', 'tc2_784x64x10'])
def test_adam_learning_rate_sweep_is_per_env(case_id, monkeypatch):
    """Env e of a batch with lr = logspace(-4, -1) runs bit for bit what a one-env batch with lr_e and
    env_base = e runs (same Glorot draw, same minibatch stream), over 6 steps with auto-reset."""
    from custom_envs_b200.baselines import DeviceAdam
    _, spec, rows, batch, num_envs, env_vars, _, _ = BY_ID[case_id]
    for key, value in env_vars.items():
        monkeypatch.setenv(key, value)
    num_envs = 4
    data = None if spec.kind == 'func' else make_data(spec, rows)
    lrs = torch.logspace(-4, -1, num_envs, device='cuda')
    big, _, _ = _env(spec, rows, batch, num_envs, data=data, max_batches=4, init_seed=9)
    adam = DeviceAdam(big, lrs)
    big.reset()
    outs = []
    for _ in range(6):
        obs, rew, done, info = adam.step()
        outs.append((obs.clone(), rew.clone(), done.clone(), info.clone(), big.get_state('params').clone(),
                     adam.m.clone(), adam.v.clone()))
    P = big.num_params
    for e in range(num_envs):
        one, _, _ = _env(spec, rows, batch, 1, data=data, max_batches=4, init_seed=9, env_base=e)
        single = DeviceAdam(one, lrs[e:e + 1].clone())
        one.reset()
        for t in range(6):
            obs, rew, done, info = single.step()
            want = outs[t]
            assert torch.equal(obs, want[0][e * P:(e + 1) * P]), (e, t)
            assert torch.equal(rew, want[1][e:e + 1]) and torch.equal(done, want[2][e:e + 1]), (e, t)
            assert torch.equal(info.nan_to_num(), want[3][e:e + 1].nan_to_num()), (e, t)
            assert torch.equal(one.get_state('params'), want[4][e:e + 1]), (e, t)
            assert torch.equal(single.m, want[5][e:e + 1]) and torch.equal(single.v, want[6][e:e + 1]), (e, t)
        one.close()
    big.close()


@pytest.mark.parametrize('case_id', ['thin3_784x10', 'tc2_784x64x10', 'generic_12x16x8x4'])
def test_ring_only_adam_step_is_the_same_env_step(case_id, monkeypatch):
    """Two identical batches, one stepping Adam with observation rows and one ring-only (without an observation
    matrix): parameters, moments, rings, rewards, done flags and info agree step by step across an episode end
    (the statistics the two paths sum in different groupings to 2e-6 relative)."""
    from custom_envs_b200.baselines import DeviceAdam
    _, spec, rows, batch, _, env_vars, _, _ = BY_ID[case_id]
    for key, value in env_vars.items():
        monkeypatch.setenv(key, value)
    data = make_data(spec, rows)
    dense, _, _ = _env(spec, rows, batch, 3, data=data, max_batches=4, init_seed=2)
    ring, _, _ = _env(spec, rows, batch, 3, data=data, max_batches=4, init_seed=2, materialize_obs=False)
    lrs = torch.tensor([1e-3, 1e-2, 3e-2], device='cuda')
    a_dense, a_ring = DeviceAdam(dense, lrs), DeviceAdam(ring, lrs)
    dense.reset()
    ring.reset()
    with pytest.raises(Exception):
        a_ring.step()                                   # no observation matrix: ring_only=True is required
    for t in range(7):
        _, rew_d, done_d, info_d = a_dense.step()
        obs_r, rew_r, done_r, info_r = a_ring.step(ring_only=True)
        assert obs_r is None
        assert torch.equal(rew_d, rew_r) and torch.equal(done_d, done_r), t
        assert torch.equal(a_dense.m, a_ring.m) and torch.equal(a_dense.v, a_ring.v), t
        exact = [i for i in range(16) if i not in (6, 7, 12, 13)]
        assert torch.equal(info_d[:, exact].nan_to_num(), info_r[:, exact].nan_to_num()), t
        # a weight or gradient that was exactly 0 (the zero biases before step 1) makes its ratio nan_to_num(x / 0)
        # = FLT_MAX; a sum holding one overflows to inf in one grouping and not in the other: both are huge
        summed_r, summed_d = info_r[:, [6, 7, 12, 13]], info_d[:, [6, 7, 12, 13]]
        huge = summed_d.abs() > 1e30
        assert torch.equal(huge, summed_r.abs() > 1e30), t
        torch.testing.assert_close(summed_r[~huge], summed_d[~huge], rtol=2e-6, atol=0)
        for name in ('params', 'grad_prev', 'adj_weights', 'adj_grads', 'adj_losses', 'step', 'cursor'):
            assert torch.equal(dense.get_state(name), ring.get_state(name)), (t, name)
    dense.close()
    ring.close()


def test_device_adam_run_writes_monitor_rows(tmp_path):
    """DeviceAdam.run with DeviceEpisodeMonitor.on_step: one .mon.csv row per finished episode, whose return,
    length and info columns are what the per-step rewards and infos say."""
    from custom_envs_b200.baselines import DeviceAdam
    from custom_envs_b200.wrappers.device_monitor import DeviceEpisodeMonitor
    spec, rows, batch = orc.ProblemSpec('softmax', 4, (), 3), 150, 32
    env, _, _ = _env(spec, rows, batch, 5, max_batches=6, init_seed=4)
    adam = DeviceAdam(env, torch.logspace(-3, -1, 5, device='cuda'))
    env.reset()
    path = str(tmp_path / 'adam')
    monitor = DeviceEpisodeMonitor(5, path, info_keywords=('loss', 'actions_mean'), device=env.device)
    steps, rewards, infos = [], [], []

    def record(t, obs, reward, done, info):
        monitor.on_step(t, obs, reward, done, info)
        rewards.append(reward.double().cpu().numpy())
        infos.append(info.cpu().numpy())
        steps.append(done.cpu().numpy().astype(bool))

    returns, finished = adam.run(14, on_step=record)
    rows_out = monitor.close()
    assert finished == 10 and len(rows_out) == 10                   # two episodes of 6 steps per env
    rewards, infos, dones = np.array(rewards), np.array(infos), np.array(steps)
    np.testing.assert_allclose(returns.cpu().numpy(), rewards.sum(axis=0), rtol=1e-12)
    for row in rows_out:
        e, k = row['env'], row['episode']
        ends = np.nonzero(dones[:, e])[0]
        end, start = ends[k - 1], (ends[k - 2] + 1 if k > 1 else 0)
        assert row['l'] == end - start + 1 == 6
        assert abs(row['r'] - round(rewards[start:end + 1, e].sum(), 6)) <= 1e-6
        assert row['loss'] == pytest.approx(infos[end, e, 0], rel=1e-12)
        assert row['actions_mean'] == pytest.approx(infos[end, e, 4], rel=1e-12)
    with open(path + '.mon.csv') as fh:
        lines = [line for line in fh.read().splitlines() if line and not line.startswith('#')]
    assert len(lines) == 1 + 10                                        # header + one row per episode
    env.close()
