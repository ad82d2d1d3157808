"""Tests of the wide observation rows: obs_dim 16..79 (MultiOptLRs max_history up to 26), for which the policy
kernels' first layer has K1 = 32, 48, 64 or 80 and a stored observation row is W = b2p_obs_width(obs_dim) bf16 wide.

The act / step kernels are held to a bf16-rounded torch evaluation as in test_gpu_policy.py and test_gpu_rollout.py;
the ring front end to the dense one, bit for bit; the PPO gradient to the float64 autograd reference of
test_gpu_ppo_update.py, with width-generic copies of its buffer, parity and update helpers."""
import math
import types

import numpy as np
import pytest
import torch

from custom_envs_b200 import _lib

if torch.cuda.is_available():
    from custom_envs_b200._lib import B200EnvError
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations
    from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer, device_policy_rollout,
                                                          device_ppo_rollout, device_ppo_update, epoch_key,
                                                          ppo_adv_stats, ppo_minibatch_indices, reference_actions,
                                                          reference_values)
    from test_gpu_ppo_update import GRAD_TOL, make_model, ppo2_loss64, tensor_errors

LOG_STD = -0.5
HALF_LOG_2PI = 0.5 * math.log(2 * math.pi)
WIDE = [16, 30, 45, 60, 75, 79]


def width(obs_dim):
    return 16 * ((obs_dim + 16) // 16)


def test_obs_width_table():
    """b2p_obs_width needs no device: W = 16 ceil((obs_dim + 1) / 16) for 1..79, 0 outside."""
    lib = _lib.load()
    for od in range(1, 80):
        assert lib.b2p_obs_width(od) == width(od), od
    assert [lib.b2p_obs_width(od) for od in (15, 16, 31, 32, 47, 48, 63, 64, 79)] == [16, 32, 32, 48, 48, 64, 64, 80, 80]
    for od in (-3, 0, 80, 96, 1000):
        assert lib.b2p_obs_width(od) == 0, od


def make_policy(obs_dim, seed, scale=1.0):
    return make_model(obs_dim, seed, scale)


def small_env(max_history, num_envs=3, max_batches=6, row_order='lexicographic', materialize_obs=True):
    """The config-4 problem shape (MLP 784-64-10, the tcgen05 pipeline) on a small data set."""
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(320, 784)).astype(np.float32)
    labels = rng.randint(0, 10, 320).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 784, (64,), 10), feats, labels, num_envs, batch_size=32,
                        max_batches=max_batches, max_history=max_history, row_order=row_order,
                        perms=env_permutations(320, list(range(num_envs))), init_seed=9, materialize_obs=materialize_obs)
    env.reset()
    return env


@pytest.mark.gpu
def test_width_and_limits_of_the_policy():
    dev = DevicePolicy(79, log_std=LOG_STD)
    assert dev.obs_width == 80
    dev.close()
    assert DevicePolicy(15).obs_width == 16 and DevicePolicy(16).obs_width == 32
    with pytest.raises(B200EnvError, match=r'1\.\.79.*max_history 26'):
        DevicePolicy(80)


# ------------------------------------------------------------------ act, dense rows
def wide_obs(rows, obs_dim, seed):
    gen = torch.Generator(device='cuda').manual_seed(seed)
    obs = torch.randn(rows, obs_dim, device='cuda', generator=gen)
    obs[::7] *= 10.0
    obs[::13, 0] = 99.0
    obs[::17, -1] = -101.0
    return obs


@pytest.mark.gpu
@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
@pytest.mark.parametrize('obs_dim', WIDE)
def test_wide_act_matches_bf16_torch(obs_dim, tanh_mode):
    """3 x 128 + 37 rows: the last tile is ragged."""
    rows = 3 * 128 + 37
    policy = make_policy(obs_dim, seed=obs_dim, scale=2.0)
    obs = wide_obs(rows, obs_dim, obs_dim)
    dev = DevicePolicy.from_torch(policy.pi, tanh_mode=tanh_mode, low=-1e9, high=1e9)
    got = dev.act(obs)
    want = reference_actions(policy.pi, obs, low=-1e9, high=1e9)
    exact = reference_actions(policy.pi, obs, low=-1e9, high=1e9, bf16=False)
    scale = max(1.0, policy.pi[-1].weight.abs().sum().item())
    err = (got - want).abs().max().item()
    assert err <= (2e-3 if tanh_mode == 0 else 1.5e-2) * scale, (err, scale)
    assert (got - exact).abs().max().item() <= 0.1 * scale
    clipped = DevicePolicy.from_torch(policy.pi, tanh_mode=tanh_mode, low=-0.05, high=0.07)
    assert torch.equal(clipped.act(obs), got.clamp(-0.05, 0.07))
    clipped.close()
    # a matrix whose rows are not 16-byte aligned (4-byte aligned base, odd obs_dim strides)
    base = torch.empty(rows * obs_dim + 1, device='cuda')
    odd = base[1:].view(rows, obs_dim)
    odd.copy_(obs)
    assert torch.equal(dev.act(odd), got)
    dev.close()


# ------------------------------------------------------------------ rings against rows
def obs_store(rows, W):
    return torch.empty((rows, W), dtype=torch.bfloat16, device='cuda')


@pytest.mark.gpu
@pytest.mark.parametrize('row_order', ['lexicographic', 'natural'])
@pytest.mark.parametrize('depth', [6, 10, 25, 26])
def test_rings_equal_rows(depth, row_order):
    """act_env == act and step(env) == step(env.obs) in all five outputs, the observation store included, from the
    reset observation through a filling and a full history and across an auto-reset (max_batches = 6, 8 steps)."""
    env = small_env(depth, row_order=row_order)
    assert env.obs_dim == 3 * depth
    W = width(env.obs_dim)
    policy = make_policy(env.obs_dim, seed=depth, scale=1.5)
    tanh_mode = depth % 3
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD), tanh_mode=tanh_mode)
    quiet = DevicePolicy.from_torch(policy.pi, tanh_mode=tanh_mode)
    gen = torch.Generator(device='cuda').manual_seed(0)
    for t in range(8):
        assert torch.equal(quiet.act_env(env), quiet.act(env.obs)), t
        ring = dev.step(env, seed=100 + t, obs_bf16=obs_store(env.num_rows, W))
        dense = dev.step(env.obs, seed=100 + t, obs_bf16=obs_store(env.num_rows, W))
        for a, b in zip(ring, dense):
            assert torch.equal(a, b), t
        assert torch.equal(ring[4][:, :env.obs_dim], env.obs.to(torch.bfloat16)) and not ring[4][:, env.obs_dim:].any()
        env.step(torch.rand(env.num_rows, device='cuda', generator=gen) * 2.0)
    assert torch.equal(dev.value(env), dev.value(env.obs))
    dev.close()
    quiet.close()
    env.close()


# ------------------------------------------------------------------ step, dense rows
@pytest.mark.gpu
@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
@pytest.mark.parametrize('obs_dim,rows', [(30, 100003), (45, 421), (79, 421), (79, 100003)])
def test_wide_step(obs_dim, rows, tanh_mode):
    policy = make_policy(obs_dim, seed=obs_dim + rows)
    obs = wide_obs(rows, obs_dim, rows)
    low, high = -1.0, 1.5
    W = width(obs_dim)
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD), tanh_mode=tanh_mode, low=low, high=high)
    store = obs_store(rows, W)
    actions, raw, values, neglogp, _ = dev.step(obs, seed=7, obs_bf16=store)
    assert torch.equal(actions, dev.act(obs, seed=7))
    assert torch.equal(raw.clamp(low, high), actions)
    want = reference_values(policy.vf, obs)
    scale = max(1.0, policy.vf[-1].weight.abs().sum().item())
    assert (values - want).abs().max().item() <= (2e-3 if tanh_mode == 0 else 1.5e-2) * scale
    quiet = DevicePolicy.from_torch(policy.pi, tanh_mode=tanh_mode, low=-1e9, high=1e9)
    mean = quiet.act(obs).double()
    nlp = 0.5 * ((raw.double() - mean) / math.exp(LOG_STD)) ** 2 + HALF_LOG_2PI + LOG_STD
    assert (neglogp.double() - nlp).abs().max().item() <= 1e-5
    assert torch.equal(store[:, :obs_dim], obs.to(torch.bfloat16))
    assert not store[:, obs_dim:].float().abs().sum().item()
    assert torch.equal(dev.value(obs), values)
    quiet.close()
    dev.close()


@pytest.mark.gpu
def test_wide_step_outputs_stay_inside_their_buffers():
    """Every output of a step launch, the W-wide observation store included, written through a window of a NaN-filled
    buffer: dense rows at ragged counts and the rings across an auto-reset."""
    pad = 1024
    obs_dim = 45
    W = width(obs_dim)
    policy = make_policy(obs_dim, seed=6)
    dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD))

    def windows(rows):
        bufs = [torch.full((rows + 2 * pad,), float('nan'), device='cuda') for _ in range(4)]
        store = torch.full(((rows + 2 * pad) * W,), float('nan'), dtype=torch.bfloat16, device='cuda')
        return bufs, store, [b[pad:pad + rows] for b in bufs], store[pad * W:(pad + rows) * W].view(rows, W)

    def check(bufs, store, rows):
        for b in bufs:
            assert torch.isnan(b[:pad]).all() and torch.isnan(b[pad + rows:]).all(), rows
            assert not torch.isnan(b[pad:pad + rows]).any(), rows
        assert torch.isnan(store[:pad * W]).all() and torch.isnan(store[(pad + rows) * W:]).all(), rows
        assert not torch.isnan(store[pad * W:(pad + rows) * W]).any(), rows

    for rows in (1, 127, 129, 100003):
        bufs, store, win, swin = windows(rows)
        dev._launch(torch.randn(rows, obs_dim, device='cuda'), dev._seed(1), *win, obs_bf16=swin)
        check(bufs, store, rows)
    env = small_env(15, max_batches=3, materialize_obs=False)
    gen = torch.Generator(device='cuda').manual_seed(1)
    for t in range(4):                                         # the third step ends every episode
        bufs, store, win, swin = windows(env.num_rows)
        dev._launch(env, dev._seed(None), *win, obs_bf16=swin)
        check(bufs, store, env.num_rows)
        act = torch.full((env.num_rows + 2 * pad,), float('nan'), device='cuda')
        dev.act_env(env, act[pad:pad + env.num_rows])
        assert torch.isnan(act[:pad]).all() and torch.isnan(act[pad + env.num_rows:]).all()
        assert not torch.isnan(act[pad:pad + env.num_rows]).any()
        env.step(torch.rand(env.num_rows, device='cuda', generator=gen) * 2, ring_only=True)
    env.close()
    dev.close()


# ------------------------------------------------------------------ rollouts at max_history 10
def buffers(buf):
    return [buf.obs_bf16, buf.actions_raw, buf.values, buf.neglogp, buf.advantages, buf.returns, buf.rewards, buf.dones]


@pytest.mark.gpu
def test_wide_ppo_rollout_on_the_rings_equals_rollout_on_rows():
    policy = make_policy(30, seed=2, scale=1.5)
    results = []
    for ring_only in (True, False):
        env = small_env(10, num_envs=4, max_batches=5, materialize_obs=not ring_only)
        dev = DevicePolicy.from_torch(policy, log_std=torch.tensor(LOG_STD))
        buf = DeviceRolloutBuffer(env, 4)
        assert buf.obs_bf16.shape == (4, env.num_rows, 32) and buf.bytes_per_row_step == 2 * 32 + 20
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
    env = small_env(10)
    with pytest.raises(MemoryError, match=r'n_steps.*x 84 B per step'):
        DeviceRolloutBuffer(env, 10 ** 12)
    env.close()


@pytest.mark.gpu
def test_wide_policy_rollout_on_the_rings_equals_rollout_on_rows():
    """device_policy_rollout at max_history 10: rows, rings and the graph-captured ring loop give the same returns,
    episode count and parameters."""
    policy = make_policy(30, seed=2, scale=1.5)
    results = []
    for ring_only, use_graph in ((False, False), (True, False), (True, True)):
        env = small_env(10, num_envs=4, max_batches=5, materialize_obs=not ring_only)
        dev = DevicePolicy.from_torch(policy.pi)
        returns, finished = device_policy_rollout(env, dev, 8, ring_only=ring_only, use_graph=use_graph)
        results.append((returns.cpu().numpy(), finished, env.get_state('params').cpu().numpy()))
        dev.close()
        env.close()
    for r in results[1:]:
        assert r[1] == results[0][1] == 4
        assert np.array_equal(r[0], results[0][0]) and np.array_equal(r[2], results[0][2])


# ------------------------------------------------------------------ PPO gradient
def synthetic_buffer(model, T, rows, tanh_mode, c, c_vf, seed):
    """test_gpu_ppo_update.synthetic_buffer with W-wide stored rows: every PPO2 branch occurs."""
    gen = torch.Generator(device='cuda').manual_seed(seed)
    od = model.pi[0].in_features
    W = width(od)
    n = T * rows
    obs16 = torch.zeros((n, W), dtype=torch.bfloat16, device='cuda')
    obs16[:, :od] = (torch.randn(n, od, device='cuda', generator=gen) * 1.5).to(torch.bfloat16)
    x = obs16[:, :od].float()
    quiet = DevicePolicy.from_torch(model.pi, tanh_mode=tanh_mode, low=-1e30, high=1e30)
    dev = DevicePolicy.from_torch(model, tanh_mode=tanh_mode)
    mu, V = quiet.act(x), dev.value(x)
    quiet.close()
    dev.close()
    sigma = math.exp(LOG_STD)
    z = torch.randn(n, device='cuda', generator=gen)
    act = mu + sigma * z
    nlp = 0.5 * ((act.double() - mu.double()) / sigma) ** 2 + HALF_LOG_2PI + LOG_STD
    u = torch.rand(n, device='cuda', generator=gen, dtype=torch.float64)
    band = torch.randint(0, 3, (n,), device='cuda', generator=gen)
    lo, hi = math.log(1 - c), math.log(1 + c)
    delta = torch.where(band == 0, lo - 0.05 - 0.3 * u, torch.where(band == 1, (lo + 0.03) + (hi - lo - 0.06) * u,
                                                                     hi + 0.05 + 0.3 * u))
    nlp_old = (nlp + delta).float()
    cv = 0.2 if (c_vf is None or c_vf < 0) else c_vf
    inside = torch.rand(n, device='cuda', generator=gen) < 0.5
    mag = torch.where(inside, 0.8 * cv * torch.rand(n, device='cuda', generator=gen),
                      cv * (1.3 + 2 * torch.rand(n, device='cuda', generator=gen)))
    sign = torch.where(torch.rand(n, device='cuda', generator=gen) < 0.5, -1.0, 1.0)
    v_old = V - sign * mag
    ret = v_old + torch.randn(n, device='cuda', generator=gen) + 0.2
    buf = types.SimpleNamespace(obs_bf16=obs16.view(T, rows, W), actions_raw=act.view(T, rows),
                                neglogp=nlp_old.view(T, rows),
                                values=torch.cat([v_old, torch.zeros(rows, device='cuda')]).view(T + 1, rows),
                                returns=ret.view(T, rows))
    return buf, mu, V


def run_parity(obs_dim, count, tanh_mode, cliprange_vf, check_branches):
    """test_gpu_ppo_update.run_parity on W-wide rows."""
    c = 0.2
    model = make_model(obs_dim, seed=obs_dim * 7 + count + tanh_mode, scale=1.3)
    T = 2
    rows = max(8, (count + T - 1) // T + 5)
    buf, mu_all, v_all = synthetic_buffer(model, T, rows, tanh_mode, c, cliprange_vf, seed=count + obs_dim)
    n = T * rows
    key, begin = 0xABCDEF + count, (n - count) // 2
    idx = ppo_minibatch_indices(n, key, begin, count)
    flat = lambda t: t.reshape(-1)[:n]       # noqa: E731  (values: its first T rows)
    act, nlp_old = flat(buf.actions_raw)[idx], flat(buf.neglogp)[idx]
    v_old, ret = flat(buf.values)[idx], flat(buf.returns)[idx]
    obs16 = buf.obs_bf16.reshape(n, width(obs_dim))[idx]
    A = (ret - v_old).double()
    adv = torch.tensor([A.mean().item(), A.std(unbiased=False).item() if count > 1 else 0.0], dtype=torch.float64,
                       device='cuda')
    dev = DevicePolicy.from_torch(model, tanh_mode=tanh_mode)
    grad, stats = dev.ppo_grad(buf, key, begin, count, adv, cliprange=c, cliprange_vf=cliprange_vf, ent_coef=0.01,
                               vf_coef=0.5)
    loss, want_stats, leaves = ppo2_loss64(model, obs16, act, nlp_old, v_old, ret, adv[0].item(), adv[1].item(), c,
                                           cliprange_vf, 0.01, 0.5, tanh_mode, mu_all[idx], v_all[idx])
    loss.backward()
    errs = tensor_errors(grad, leaves)
    print('tanh_mode %d obs_dim %d count %d cliprange_vf %s: max relative L2 error %.2e' % (tanh_mode, obs_dim, count,
                                                                                          cliprange_vf, max(errs)))
    assert max(errs) <= GRAD_TOL, errs
    got, want = stats.cpu().numpy(), want_stats.cpu().numpy()
    for i in (0, 1, 2, 3, 5):
        assert abs(got[i] - want[i]) <= 1e-4 * max(abs(want[i]), 1e-6), (i, got[i], want[i])
    assert round(got[4] * count) == round(want[4] * count), (got[4], want[4])
    if check_branches:
        mu, V = mu_all[idx].double(), v_all[idx].double()
        An = (A - adv[0]) / (adv[1] + 1e-8)
        nlp = 0.5 * ((act.double() - mu) / math.exp(LOG_STD)) ** 2 + HALF_LOG_2PI + LOG_STD
        clipped = ((torch.exp(nlp_old.double() - nlp) - 1).abs() > c)
        for mask in (clipped & (An > 0), clipped & (An < 0), ~clipped & (An > 0), ~clipped & (An < 0)):
            assert mask.double().mean().item() >= 0.05
        cv = c if cliprange_vf is None else cliprange_vf
        if cv >= 0:
            vclip = (V - v_old.double()).abs() > cv
            assert 0.05 <= vclip.double().mean().item() <= 0.95
    dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize('cliprange_vf', [None, 0.1, -1.0])
@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
@pytest.mark.parametrize('obs_dim', [30, 45, 75, 79])
def test_wide_gradient_matches_float64_autograd(obs_dim, tanh_mode, cliprange_vf):
    run_parity(obs_dim, 100003, tanh_mode, cliprange_vf, check_branches=True)


@pytest.mark.gpu
def test_wide_gradient_across_many_accumulator_flushes():
    """Every group (one per SM on wide rows) reads its TMEM accumulators out at least three times (every 16 tiles)."""
    count = 1000003
    slots = torch.cuda.get_device_properties(0).multi_processor_count
    assert count // 128 // slots >= 3 * 16
    run_parity(45, count, 1, 0.1, check_branches=True)


@pytest.mark.gpu
@pytest.mark.parametrize('count', [1, 129])
def test_wide_gradient_at_small_minibatches(count):
    run_parity(79, count, 0, None, check_branches=False)


@pytest.mark.gpu
@pytest.mark.parametrize('ring_only', [True, False], ids=['rings', 'dense'])
def test_wide_forward_equals_the_rollouts(ring_only):
    """max_history 10: with returns = values the value loss and the value tower's gradient are exactly zero."""
    env = small_env(10, materialize_obs=not ring_only)
    model = make_model(30, seed=5, scale=1.5)
    for tanh_mode in (0, 1, 2):
        dev = DevicePolicy.from_torch(model, tanh_mode=tanh_mode)
        buf = DeviceRolloutBuffer(env, 3)
        device_ppo_rollout(env, dev, buf, ring_only=ring_only)
        T, rows = buf.actions_raw.shape
        buf.returns.copy_(buf.values[:T])
        adv = torch.tensor([0.0, 1.0], dtype=torch.float64, device='cuda')
        grad, stats = dev.ppo_grad(buf, 7, 0, T * rows, adv)
        tower = grad.numel() // 2
        s = stats.cpu().numpy()
        assert s[1] == 0.0, (tanh_mode, s)
        assert not grad[tower:2 * tower].any(), tanh_mode
        assert s[4] == 0.0 and s[3] < 1e-10, (tanh_mode, s)
        dev.close()
    env.close()


@pytest.mark.gpu
def test_wide_gradient_is_deterministic_and_stays_inside_its_buffers():
    model = make_model(45, seed=11)
    buf, _, _ = synthetic_buffer(model, 2, 60000, 0, 0.2, None, seed=1)
    adv = torch.tensor([0.1, 1.2], dtype=torch.float64, device='cuda')
    dev = DevicePolicy.from_torch(model)
    g1, s1 = dev.ppo_grad(buf, 5, 1000, 100003, adv)
    g1, s1 = g1.clone(), s1.clone()
    g2, s2 = dev.ppo_grad(buf, 5, 1000, 100003, adv)
    assert torch.equal(g1, g2) and torch.equal(s1, s2)
    pad = 1024
    gbuf = torch.full((g1.numel() + 2 * pad,), float('nan'), device='cuda')
    sbuf = torch.full((6 + 2 * pad,), float('nan'), dtype=torch.float64, device='cuda')
    size = dev._ppo_ws.numel()
    wbuf = torch.full((size + 2 * 4096,), 0xA5, dtype=torch.uint8, device='cuda')
    dev._ppo_ws = wbuf[4096:4096 + size]
    for count in (1, 129, 100003):
        dev.ppo_grad(buf, 5, 0, count, adv, grad=gbuf[pad:pad + g1.numel()], stats=sbuf[pad:pad + 6])
        for b, n in ((gbuf, g1.numel()), (sbuf, 6)):
            assert torch.isnan(b[:pad]).all() and torch.isnan(b[pad + n:]).all()
            assert not torch.isnan(b[pad:pad + n]).any()
        assert (wbuf[:4096] == 0xA5).all() and (wbuf[4096 + size:] == 0xA5).all()
    g3, s3 = dev.ppo_grad(buf, 5, 1000, 100003, adv)
    assert torch.equal(g3, g1) and torch.equal(s3, s1)
    narrow = types.SimpleNamespace(**vars(buf))
    narrow.obs_bf16 = buf.obs_bf16[:, :, :16].contiguous()
    with pytest.raises(AssertionError, match='obs_width'):
        dev.ppo_grad(narrow, 5, 0, 10, adv)
    dev.close()


# ------------------------------------------------------------------ device_ppo_update at max_history 10
def reference_update(model, buf, optimizer, seed, n_epochs, n_minibatches, tanh_mode=0, **kw):
    """test_gpu_ppo_update.reference_update on W-wide rows."""
    T, rows = buf.actions_raw.shape
    n = T * rows
    mb = n // n_minibatches
    W = buf.obs_bf16.shape[-1]
    params = [p for tower in (model.pi, model.vf) for lin in tower if isinstance(lin, torch.nn.Linear)
              for p in (lin.weight, lin.bias)] + [model.log_std]
    total = np.zeros(6)
    for epoch in range(n_epochs):
        order = ppo_minibatch_indices(n, epoch_key(seed, epoch), 0, n)
        for m in range(n_minibatches):
            idx = order[m * mb:(m + 1) * mb]
            pick = lambda t: t.reshape(-1)[:n][idx]    # noqa: E731
            ret, v_old = pick(buf.returns), pick(buf.values)
            A = (ret - v_old).double()
            loss, stats, leaves = ppo2_loss64(model, buf.obs_bf16.reshape(n, W)[idx], pick(buf.actions_raw),
                                              pick(buf.neglogp), v_old, ret, A.mean().item(), A.std(unbiased=False).item(),
                                              kw['cliprange'], kw['cliprange_vf'], kw['ent_coef'], kw['vf_coef'],
                                              tanh_mode)
            loss.backward()
            for p, leaf in zip(params, leaves):
                p.grad = leaf.grad.to(p.dtype).reshape(p.shape).clone()
            torch.nn.utils.clip_grad_norm_(params, kw['max_grad_norm'])
            optimizer.step()
            total += stats.cpu().numpy()
    return total / (n_epochs * n_minibatches)


@pytest.mark.gpu
def test_wide_update_matches_the_torch_reference_loop_and_lowers_the_loss():
    env = small_env(10)
    model = make_model(30, seed=21, scale=1.5)
    dev = DevicePolicy.from_torch(model)
    buf = DeviceRolloutBuffer(env, 4)
    device_ppo_rollout(env, dev, buf, ring_only=True)
    twin = make_model(30, seed=21, scale=1.5)
    start = [p.detach().clone() for p in model.parameters()]
    kw = dict(cliprange=0.2, cliprange_vf=None, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5)
    opt = torch.optim.Adam(model.parameters(), lr=3e-4, eps=1e-5)
    twin_opt = torch.optim.Adam(twin.parameters(), lr=3e-4, eps=1e-5)
    got = device_ppo_update(model, dev, buf, opt, n_epochs=1, n_minibatches=2, seed=4, **kw)
    want = reference_update(twin, buf, twin_opt, 4, 1, 2, **kw)
    for p, q, s in zip(model.parameters(), twin.parameters(), start):
        d, e = (p - s).detach().double(), (q - s).detach().double()
        assert (d - e).norm().item() <= 0.1 * e.norm().item() + 1e-7, p.shape
    mb = buf.actions_raw.numel() // 2
    keep = [0, 1, 2, 3, 5]
    assert np.allclose(got[keep], want[keep], rtol=1e-3, atol=1e-6), (got, want)
    assert abs(got[4] - want[4]) <= 2.0 / mb, (got, want)
    # 20 update steps lower the loss
    T, rows = buf.actions_raw.shape
    n = T * rows
    adv = ppo_adv_stats(buf, 1, n)[0]
    before = dev.ppo_grad(buf, 1, 0, n, adv)[1][5].item()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, eps=1e-5)
    device_ppo_update(model, dev, buf, opt, n_epochs=5, n_minibatches=4, seed=2)
    after = dev.ppo_grad(buf, 1, 0, n, adv)[1][5].item()
    assert after < before, (before, after)
    dev.close()
    env.close()
