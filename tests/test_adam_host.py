"""The Adam baseline without a GPU: the oracle's Adam step against a float64 restatement of the Keras 2.2
formulas, and the argument checks of ``DeviceAdam``."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import optenv_oracle as orc

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from adam_oracle import AdamOracle  # noqa: E402


def keras_adam_run(spec, feats, targs, lr, w0, batches, resets, beta_1=0.9, beta_2=0.999, eps=1e-7):
    """Keras' ``Adam.get_updates`` written out: one env, float64 moments, float32 variables.  ``batches``:
    the (idx, cnt) of every step, ``resets``: {step: new weights} where an episode restarts (iterations
    and moments start over with a fresh optimiser).  Returns the weights after every step."""
    b1, b2, eps = (np.float64(np.float32(x)) for x in (beta_1, beta_2, eps))
    w = np.asarray(w0, np.float32)
    m = v = np.zeros(w.size)
    t, out = 0, []
    for step, (idx, cnt) in enumerate(batches):
        if step in resets:
            w, m, v, t = np.asarray(resets[step], np.float32), np.zeros(w.size), np.zeros(w.size), 0
        t += 1
        mask = np.arange(idx.shape[0]) < cnt
        g_sum, _ = orc.loss_and_grad(spec, w[None], feats[idx][None], targs[idx][None], mask[None])
        g = g_sum[0].astype(np.float32).astype(np.float64) / cnt          # the mean loss' gradient
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g ** 2
        lr_t = np.float64(np.float32(lr)) * np.sqrt(1 - b2 ** t) / (1 - b1 ** t)
        w = (w - lr_t * m / (np.sqrt(v) + eps)).astype(np.float32)
        out.append(w)
    return out


def test_oracle_adam_matches_keras_formulas_over_50_steps():
    """Two envs with different learning rates over 50 steps: episodes of 20 steps (t = 1 after each auto-reset),
    150 rows in minibatches of 32 (every fifth batch is the ragged one of 22 rows)."""
    spec = orc.ProblemSpec('softmax', 4, (), 3)
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(150, 4)).astype(np.float32)
    targs = rng.randint(0, 3, 150).astype(np.int32)
    lrs = np.array([1e-3, 3e-2], np.float32)
    env = orc.BatchedOptEnvOracle(spec, feats, targs, 2, batch_size=32, config=orc.EnvConfig.multioptlrs(20),
                                  perms=np.stack([orc.env_permutation(150, s) for s in range(2)]))
    adam = AdamOracle(env, lrs)
    init = np.stack([orc.glorot_uniform_init(spec, rng) for _ in range(2)])
    env.reset(init_params=init)
    batches, resets, weights, counts = [[], []], [{0: init[0]}, {0: init[1]}], [], set()
    for step in range(50):
        idx, cnt = env.current_batch()
        for e in range(2):
            batches[e].append((idx[e].copy(), int(cnt[e])))
            counts.add(int(cnt[e]))
        _, _, done, info = adam.step()
        assert np.all(np.isfinite(info['actions_mean'])) and np.all(info['actions_std'] >= 0)
        weights.append(env.weights.copy())
        if done.any():
            fresh = np.stack([orc.glorot_uniform_init(spec, rng) for _ in range(2)])
            env.reset(done, init_params=fresh)
            for e in np.nonzero(done)[0]:
                resets[e][step + 1] = fresh[e]
    assert counts == {32, 22}
    assert sorted(resets[0]) == [0, 20, 40]
    for e in range(2):
        want = keras_adam_run(spec, feats, targs, lrs[e], init[e], batches[e], resets[e])
        for step in range(50):
            have = weights[step][e]
            scale = np.abs(want[step]).mean()
            assert np.abs(have - want[step]).max() <= 1e-5 * scale, (e, step)


def test_oracle_adam_first_step_ignores_stale_moments():
    """t = 1 starts from zero moments whatever m and v hold."""
    spec = orc.ProblemSpec('func', 0, (), 0)
    env = orc.BatchedOptEnvOracle(spec, None, None, 1, config=orc.EnvConfig.multioptlrs(5))
    adam = AdamOracle(env, 1e-2)
    env.reset()
    adam.m[:] = 123.0
    adam.v[:] = 456.0
    m, v, rate = adam.update()
    g, _ = env.evaluate()
    b1, b2 = np.float64(np.float32(0.9)), np.float64(np.float32(0.999))    # the fp32 constants of the C ABI
    np.testing.assert_allclose(m, (1 - b1) * g, rtol=1e-12)     # Rosenbrock: cnt = 0, g = g0
    np.testing.assert_allclose(v, (1 - b2) * g * g, rtol=1e-12)


# ----------------------------------------------------------------------------- DeviceAdam argument checks
def _fake_batch(env_kind='optlrs', num_envs=3, num_params=5):
    """A BatchedOptEnv shell on the CPU: the attributes DeviceAdam reads before it touches the library."""
    from custom_envs_b200.batched_env import BatchedOptEnv
    env = BatchedOptEnv.__new__(BatchedOptEnv)
    env.env_kind_name, env.num_envs, env.num_params = env_kind, num_envs, num_params
    env.device, env.handle = torch.device('cpu'), None
    return env


def test_device_adam_holds_moments_and_per_env_rates():
    from custom_envs_b200.baselines import DeviceAdam
    adam = DeviceAdam(_fake_batch(), lr=torch.tensor([1e-4, 1e-3, 1e-2]))
    assert adam.m.shape == adam.v.shape == (3, 5) and adam.m.dtype == torch.float32
    assert torch.equal(adam.lr, torch.tensor([1e-4, 1e-3, 1e-2]))
    assert torch.equal(DeviceAdam(_fake_batch()).lr, torch.full((3,), 1e-3))
    sweep = torch.tensor([1e-4, 1e-3, 1e-2])
    copy = DeviceAdam(_fake_batch(), lr=sweep)
    sweep[0] = 5.0                                            # the caller's tensor is not the optimiser's
    assert float(copy.lr[0]) == pytest.approx(1e-4)
    state = adam.state()
    state['m'] += 1.0
    other = DeviceAdam(_fake_batch(), lr=0.5)
    other.load_state(state)
    assert torch.equal(other.m, torch.ones(3, 5)) and torch.equal(other.lr, adam.lr)
    with pytest.raises(ValueError):
        other.load_state({'m': torch.zeros(3, 4), 'v': torch.zeros(3, 5)})


@pytest.mark.parametrize('lr', [0.0, -1e-3, float('nan'), float('inf'), torch.tensor([1e-3, 0.0, 1e-3]),
                                torch.full((4,), 1e-3), torch.full((3, 1), 1e-3)])
def test_device_adam_rejects_bad_learning_rates(lr):
    from custom_envs_b200.baselines import DeviceAdam
    with pytest.raises(ValueError):
        DeviceAdam(_fake_batch(), lr=lr)


@pytest.mark.parametrize('kwargs', [dict(beta_1=1.0), dict(beta_2=-0.1), dict(epsilon=0.0)])
def test_device_adam_rejects_bad_constants(kwargs):
    from custom_envs_b200.baselines import DeviceAdam
    with pytest.raises(ValueError):
        DeviceAdam(_fake_batch(), **kwargs)


def test_device_adam_rejects_multioptimize_and_host_envs():
    from custom_envs_b200.baselines import DeviceAdam
    from custom_envs_b200.vectorize.optvecenv import OptVecEnv
    with pytest.raises(ValueError, match='MultiOptLRs'):
        DeviceAdam(_fake_batch('optimize'))
    host = OptVecEnv.__new__(OptVecEnv)
    host._wrapped = None                                      # the host fallback: no device batch
    assert not host.is_device_backed
    with pytest.raises(ValueError, match='host fallback'):
        DeviceAdam(host)
    with pytest.raises(ValueError):
        DeviceAdam(object())
