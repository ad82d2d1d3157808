"""GPU tests of PPO updates on the device: the minibatch permutation (b2p_ppo_indices), the advantage statistics
(b2p_ppo_adv_stats), the fused clipped-surrogate gradient kernel (b2p_ppo_grad, DevicePolicy.ppo_grad) and
device_ppo_update.

The gradient is held to torch float64 autograd of stable-baselines 2's PPO2 loss (a restatement: stable-baselines is
not installed here), rounding to bf16 where the kernel does: the observation rows, the weights of both MMAs, h1 before
the second MMA, and the dPre tiles of the backward.  The reference takes the action mean and the value of each row
from the kernel's own forward (b2p_act / b2p_step, whose bits the gradient kernel reproduces), so that rows near a clip
boundary take the same branch on both sides; the backward through each tower is the reference's."""
import ctypes
import math
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from custom_envs_b200 import _lib
    from custom_envs_b200._lib import B200EnvError
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations
    from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer, device_ppo_rollout,
                                                          device_ppo_update, epoch_key, ppo_adv_stats,
                                                          ppo_minibatch_indices, tanh_bf16_table)
    from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy

LOG_STD = -0.5
HALF_LOG_2PI = 0.5 * math.log(2 * math.pi)
M64 = (1 << 64) - 1


# ------------------------------------------------------------------ numpy restatement of the permutation
def mix64(z):
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over='ignore'):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def feistel_np(key, n, positions, rounds=6):
    """Position p -> flat sample index: a Feistel network on 2 x bits bits (4^bits >= n), round keys
    mix64(key + golden * (r + 1)), round function mix64(R ^ k_r) & mask, cycle-walked until the value is < n."""
    bits = 1
    while (1 << (2 * bits)) < n:
        bits += 1
    mask, b = np.uint64((1 << bits) - 1), np.uint64(bits)
    keys = [np.uint64(int(mix64(np.uint64((key + 0x9E3779B97F4A7C15 * (r + 1)) & M64)))) for r in range(rounds)]
    v = np.asarray(positions, dtype=np.uint64).copy()
    todo = np.ones(v.shape, dtype=bool)
    while todo.any():
        x = v[todo]
        L, R = x >> b, x & mask
        for k in keys:
            L, R = R, L ^ (mix64(R ^ k) & mask)
        v[todo] = (L << b) | R
        todo = v >= np.uint64(n)
    return v.astype(np.int64)


@pytest.mark.parametrize('n', [1, 2, 127, 1000003])
def test_indices_are_the_restated_permutation(n):
    key = 0x1234567 + n
    got = ppo_minibatch_indices(n, key, 0, n).cpu().numpy()
    assert np.array_equal(np.sort(got), np.arange(n))
    assert np.array_equal(got, feistel_np(key, n, np.arange(n)))
    if n > 2:
        begin, count = n // 3, n // 2
        assert np.array_equal(ppo_minibatch_indices(n, key, begin, count).cpu().numpy(), got[begin:begin + count])
        assert not np.array_equal(ppo_minibatch_indices(n, key + 1, 0, n).cpu().numpy(), got)


def test_indices_permute_beyond_int32():
    """2^31 + 5 samples: every index is hit exactly once (device-side bitmap over the whole order), and a slice matches
    the numpy restatement."""
    n = 2 ** 31 + 5
    idx = ppo_minibatch_indices(n, 99, 0, n)
    assert int(idx.min()) == 0 and int(idx.max()) == n - 1
    seen = torch.zeros(n, dtype=torch.uint8, device='cuda')
    seen[idx] = 1
    assert bool(seen.all())
    del seen
    tail = idx[n - 1000:].cpu().numpy()
    del idx
    assert np.array_equal(tail, feistel_np(99, n, np.arange(n - 1000, n)))


def test_bf16_tanh_table_is_a_bf16_tanh():
    """b2p_tanh_table: for every finite bf16 input, within two bf16 steps of tanh of that input (subnormal results
    may flush to zero), odd, and bf16."""
    table = tanh_bf16_table()
    x = torch.arange(65536, dtype=torch.int32, device='cuda').to(torch.int16).view(torch.bfloat16).float()
    finite = torch.isfinite(x)
    exact = torch.tanh(x.double())
    step = torch.clamp(exact.abs() * 2.0 ** -6, min=2.0 ** -126)
    assert ((table.double() - exact).abs() <= step)[finite].all()
    assert torch.equal(table[finite], table[finite].to(torch.bfloat16).float())
    assert torch.equal(table[32768:][finite[32768:]], -table[:32768][finite[:32768]])


# ------------------------------------------------------------------ float64 reference of PPO2's loss
class _RoundGrad(torch.autograd.Function):
    """Identity forward; the incoming gradient rounded to bf16 (the kernel's dPre tiles)."""
    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype)


def _st(t):
    """bf16 rounding in the forward, identity in the backward."""
    return t + (t.to(torch.bfloat16).to(t.dtype) - t).detach()


_TANH_TABLE = {}


def _bf16_tanh(pre):
    """The kernels' tanh.approx.bf16x2 of bf16(pre): looked up in the device's own table (b2p_tanh_table), indexed
    by the bit pattern of the fp32 accumulator rounded to bf16."""
    if 'table' not in _TANH_TABLE:
        _TANH_TABLE['table'] = tanh_bf16_table().double()
    bits = pre.float().to(torch.bfloat16).view(torch.int16).to(torch.int64) & 0xFFFF
    return _TANH_TABLE['table'][bits]


class _Tanh(torch.autograd.Function):
    """tanh as the kernel evaluates it, with the kernel's derivative 1 - h^2 taken from the h it computed (the bf16
    operand of the next MMA for the first layer, the fp32 or bf16 value of the head for the second)."""
    @staticmethod
    def forward(ctx, pre, mode):
        if mode == 'bf16_table':
            h = _bf16_tanh(pre)
        elif mode == 'round':
            h = torch.tanh(pre).float().to(torch.bfloat16).to(pre.dtype)
        else:
            h = torch.tanh(pre)
        ctx.save_for_backward(h)
        return h

    @staticmethod
    def backward(ctx, g):
        h, = ctx.saved_tensors
        return g * (1 - h * h), None


def tower64(x, params, tanh_mode):
    w1, b1, w2, b2, w3, b3 = params
    pre1 = _RoundGrad.apply(x @ _st(w1).t() + _st(b1))
    h1 = _Tanh.apply(pre1, 'bf16_table' if tanh_mode >= 1 else 'round')
    pre2 = _RoundGrad.apply(h1 @ _st(w2).t() + _st(b2))
    h2 = _Tanh.apply(pre2, 'bf16_table' if tanh_mode == 2 else 'exact')
    return (h2 @ w3.reshape(-1) + b3).reshape(-1)


def model_params64(model):
    out = []
    for tower in (model.pi, model.vf):
        lins = [m for m in tower.modules() if isinstance(m, torch.nn.Linear)]
        out.append([t.detach().double().clone().requires_grad_(True) for lin in lins for t in (lin.weight, lin.bias)])
    return out


def ppo2_loss64(model, obs16, act, nlp_old, v_old, ret, adv_mean, adv_std, cliprange, cliprange_vf, ent_coef, vf_coef,
                tanh_mode, mu_fixed=None, v_fixed=None):
    """PPO2._train_step's loss in float64 (TF gradient rules via torch.where / clamp).  mu_fixed / v_fixed: forward
    values to use (the gradient still flows through the reference towers).  Returns (loss, stats [6], leaves)."""
    pi_p, vf_p = model_params64(model)
    log_std = torch.tensor(float(model.log_std.detach()), dtype=torch.float64, device=obs16.device, requires_grad=True)
    od = model.pi[0].in_features
    x = obs16[:, :od].double()
    mu = tower64(x, pi_p, tanh_mode)
    V = tower64(x, vf_p, tanh_mode)
    if mu_fixed is not None:
        mu = mu_fixed.double() + (mu - mu.detach())
        V = v_fixed.double() + (V - V.detach())
    A = (ret.float() - v_old.float()).double()
    An = (A - adv_mean) / (adv_std + 1e-8)
    nlp = 0.5 * ((act.double() - mu) / torch.exp(log_std)) ** 2 + HALF_LOG_2PI + log_std
    ratio = torch.exp(nlp_old.double() - nlp)
    l1, l2 = -An * ratio, -An * torch.clamp(ratio, 1 - cliprange, 1 + cliprange)
    pg = torch.where(l1 >= l2, l1, l2).mean()
    c_vf = cliprange if cliprange_vf is None else cliprange_vf
    vc = V if c_vf < 0 else v_old.double() + torch.clamp(V - v_old.double(), -c_vf, c_vf)
    f1, f2 = (V - ret.double()) ** 2, (vc - ret.double()) ** 2
    vf = 0.5 * torch.where(f1 >= f2, f1, f2).mean()
    ent = log_std + 0.5 * math.log(2 * math.pi * math.e)
    loss = pg - ent_coef * ent + vf_coef * vf
    with torch.no_grad():
        stats = torch.stack([pg, vf, ent, 0.5 * ((nlp - nlp_old.double()) ** 2).mean(),
                             ((ratio - 1).abs() > cliprange).double().mean(), loss])
    return loss, stats, pi_p + vf_p + [log_std]


def make_model(obs_dim, seed, scale=1.0):
    torch.manual_seed(seed)
    model = SharedMlpPolicy(obs_dim, log_std=LOG_STD).cuda()
    with torch.no_grad():
        for tower in (model.pi, model.vf):
            for p in tower.parameters():
                p.mul_(scale)
            for m in tower.modules():
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.3, 0.3)
    return model


def synthetic_buffer(model, T, rows, tanh_mode, c, c_vf, seed):
    """A rollout buffer in which every PPO2 branch occurs: log-ratios in three bands (below 1 - c, inside, above
    1 + c; away from the boundaries by more than the bf16 forward error), value offsets inside and outside the value
    clip range, advantages of both signs."""
    gen = torch.Generator(device='cuda').manual_seed(seed)
    od = model.pi[0].in_features
    n = T * rows
    obs16 = torch.zeros((n, 16), dtype=torch.bfloat16, device='cuda')
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
    buf = types.SimpleNamespace(obs_bf16=obs16.view(T, rows, 16), actions_raw=act.view(T, rows),
                                neglogp=nlp_old.view(T, rows), values=torch.cat([v_old, torch.zeros(rows, device='cuda')]).view(T + 1, rows),
                                returns=ret.view(T, rows))
    return buf, mu, V


def rel_l2(got, want):
    got, want = got.double(), want.double()
    return (got - want).norm().item() / max(want.norm().item(), 1e-30)


def tensor_errors(grad, leaves):
    out, off = [], 0
    for leaf in leaves:
        k = grad[off:off + leaf.numel()].view_as(leaf)
        off += leaf.numel()
        ref = leaf.grad
        err = (k.double() - ref).norm().item()
        out.append(err / max(ref.norm().item(), 1e-12) if ref.norm().item() > 1e-9 else err)
    assert off == grad.numel()
    return out


# bf16 has 8 significant bits (relative rounding 2^-9 = 2e-3 per operand); each gradient entry is a sum over the
# minibatch of products of two or three rounded factors (dPre, h1 / A1, W2) whose rounding errors are unbiased and
# average out over rows.  The reference reproduces every rounding and the kernels' own bf16 tanh (tabulated on the
# device), so what remains is fp32 against fp64 accumulation and tanh.approx.f32 (2^-11) in the fp32 tanh modes.  A
# per-tensor relative L2 error of 1e-2 is five times the single-rounding bound.
GRAD_TOL = 1e-2


def run_parity(obs_dim, count, tanh_mode, cliprange_vf, check_branches):
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
    obs16 = buf.obs_bf16.reshape(n, 16)[idx]
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
    got = stats.cpu().numpy()
    want = want_stats.cpu().numpy()
    for i in (0, 1, 2, 3, 5):
        assert abs(got[i] - want[i]) <= 1e-4 * max(abs(want[i]), 1e-6), (i, got[i], want[i])
    # the synthetic log-ratios stay 0.03 away from the clip boundaries and both sides use the kernel's forward values:
    # the clipped rows are the same rows
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


@pytest.mark.parametrize('cliprange_vf', [None, 0.1, -1.0])
@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
@pytest.mark.parametrize('obs_dim', [3, 9, 15])
def test_gradient_matches_float64_autograd(obs_dim, tanh_mode, cliprange_vf):
    run_parity(obs_dim, 100003, tanh_mode, cliprange_vf, check_branches=True)


@pytest.mark.parametrize('tanh_mode', [0, 2])
def test_gradient_across_many_accumulator_flushes(tanh_mode):
    """A minibatch large enough that every group reads its TMEM accumulators out several times (every 16 tiles):
    the flush, the restart of the accumulators and of the FFMA sums are held to the float64 reference."""
    count = 2500003
    slots = 2 * torch.cuda.get_device_properties(0).multi_processor_count
    assert count // 128 // slots >= 3 * 16
    run_parity(15, count, tanh_mode, 0.1, check_branches=True)


@pytest.mark.parametrize('tanh_mode', [0, 2])
@pytest.mark.parametrize('count', [1, 127, 128, 129])
def test_gradient_at_small_minibatches(count, tanh_mode):
    run_parity(15, count, tanh_mode, None, check_branches=False)


def test_adv_stats_match_numpy():
    T, rows, mb = 3, 70001, 70001
    gen = torch.Generator(device='cuda').manual_seed(3)
    buf = types.SimpleNamespace(obs_bf16=torch.zeros((T, rows, 16), dtype=torch.bfloat16, device='cuda'),
                                actions_raw=torch.zeros(T, rows, device='cuda'), neglogp=torch.zeros(T, rows, device='cuda'),
                                values=torch.randn(T + 1, rows, device='cuda', generator=gen) * 3 + 50,
                                returns=torch.randn(T, rows, device='cuda', generator=gen) + 51)
    key = 17
    stats = ppo_adv_stats(buf, key, mb).cpu().numpy()
    A = (buf.returns - buf.values[:T]).reshape(-1).double().cpu().numpy()
    order = feistel_np(key, T * rows, np.arange(T * rows))
    for m in range(T * rows // mb):
        a = A[order[m * mb:(m + 1) * mb]]
        assert abs(stats[m, 0] - a.mean()) <= 1e-12 * abs(a.mean()) + 1e-12
        assert abs(stats[m, 1] - a.std()) <= 1e-9 * a.std()
    with pytest.raises(ValueError, match='minibatches'):
        ppo_adv_stats(buf, key, 7)


# ------------------------------------------------------------------ on a real rollout
def small_env(num_envs=3, max_batches=6, materialize_obs=True):
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(320, 784)).astype(np.float32)
    labels = rng.randint(0, 10, 320).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 784, (64,), 10), feats, labels, num_envs, batch_size=32,
                        max_batches=max_batches, max_history=5, perms=env_permutations(320, list(range(num_envs))),
                        init_seed=9, materialize_obs=materialize_obs)
    env.reset()
    return env


@pytest.mark.parametrize('ring_only', [True, False], ids=['rings', 'dense'])
def test_forward_equals_the_rollouts(ring_only):
    """At the rollout's own weights the kernel's forward is the step kernel's, bit for bit: with returns = values the
    value loss and the value tower's gradient are exactly zero, no ratio is clipped and approxkl vanishes."""
    env = small_env(materialize_obs=not ring_only)
    model = make_model(15, seed=5, scale=1.5)
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


def test_gradient_is_deterministic_and_stays_inside_its_buffers():
    model = make_model(15, seed=11)
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
    dev.close()


def test_errors():
    model = make_model(15, seed=12)
    buf, _, _ = synthetic_buffer(model, 2, 1000, 0, 0.2, None, seed=2)
    adv = torch.tensor([0.0, 1.0], dtype=torch.float64, device='cuda')
    bare = DevicePolicy(15, log_std=LOG_STD)
    with pytest.raises(B200EnvError, match='weights not set'):
        bare.ppo_grad(buf, 1, 0, 10, adv)
    bare.close()
    dev = DevicePolicy.from_torch(model)
    flat = torch.zeros(2 * 1000 * 16 + 8, dtype=torch.bfloat16, device='cuda')
    odd = types.SimpleNamespace(**vars(buf))
    odd.obs_bf16 = flat[1:1 + 2 * 1000 * 16].view(2, 1000, 16)
    with pytest.raises(B200EnvError, match='16-byte aligned'):
        dev.ppo_grad(odd, 1, 0, 10, adv)
    with pytest.raises(B200EnvError, match='range outside'):
        dev.ppo_grad(buf, 1, 1995, 10, adv)
    with pytest.raises(B200EnvError, match='range outside'):
        dev.ppo_grad(buf, 1, -1, 10, adv)
    with pytest.raises(B200EnvError, match='count must be'):
        dev.ppo_grad(buf, 1, 0, 0, adv)
    with pytest.raises(B200EnvError, match='cliprange must be'):
        dev.ppo_grad(buf, 1, 0, 10, adv, cliprange=0.0)
    with pytest.raises(B200EnvError, match='count must be'):
        ppo_minibatch_indices(10, 1, 0, 0)
    # an epoch of 2^31 + 2 one-sample minibatches needs more blocks than one launch has; rejected before any access
    lib = _lib.load()
    huge = _lib.PpoBatch(buf.obs_bf16.data_ptr(), buf.actions_raw.data_ptr(), buf.neglogp.data_ptr(),
                         buf.values.data_ptr(), buf.returns.data_ptr(), 2, 2 ** 30 + 1)
    assert lib.b2p_ppo_adv_stats(ctypes.byref(huge), 1, 1, ctypes.c_void_p(adv.data_ptr()),
                                 ctypes.c_void_p(adv.data_ptr()), None)
    assert b'too many minibatches' in lib.b2p_last_error(None)
    with pytest.raises(B200EnvError, match='range outside'):
        ppo_minibatch_indices(10, 1, 5, 6)
    dev.close()


# ------------------------------------------------------------------ device_ppo_update
def reference_update(model, buf, optimizer, seed, n_epochs, n_minibatches, tanh_mode=0, **kw):
    """The SB2 learn() inner loop in torch (float64 autograd of ppo2_loss64, same permutation), for small shapes."""
    T, rows = buf.actions_raw.shape
    n = T * rows
    mb = n // n_minibatches
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
            loss, stats, leaves = ppo2_loss64(model, buf.obs_bf16.reshape(n, 16)[idx], pick(buf.actions_raw),
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


def test_update_matches_the_torch_reference_loop():
    env = small_env()
    model = make_model(15, seed=21, scale=1.5)
    dev = DevicePolicy.from_torch(model)
    buf = DeviceRolloutBuffer(env, 4)
    device_ppo_rollout(env, dev, buf, ring_only=True)
    twin = make_model(15, seed=21, scale=1.5)
    start = [p.detach().clone() for p in model.parameters()]
    kw = dict(cliprange=0.2, cliprange_vf=None, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5)
    opt = torch.optim.Adam(model.parameters(), lr=3e-4, eps=1e-5)
    twin_opt = torch.optim.Adam(twin.parameters(), lr=3e-4, eps=1e-5)
    got = device_ppo_update(model, dev, buf, opt, n_epochs=1, n_minibatches=2, seed=4, **kw)
    want = reference_update(twin, buf, twin_opt, 4, 1, 2, **kw)
    # Adam moves each parameter by about lr per step whatever the gradient's size, so the updates are compared: a
    # parameter whose gradient is within bf16 rounding of zero may move differently, which the relative L2 absorbs
    for p, q, s in zip(model.parameters(), twin.parameters(), start):
        d, e = (p - s).detach().double(), (q - s).detach().double()
        assert (d - e).norm().item() <= 0.1 * e.norm().item() + 1e-7, p.shape
    mb = buf.actions_raw.numel() // 2
    keep = [0, 1, 2, 3, 5]
    assert np.allclose(got[keep], want[keep], rtol=1e-3, atol=1e-6), (got, want)
    assert abs(got[4] - want[4]) <= 2.0 / mb, (got, want)      # a row at the clip boundary may fall either way
    assert dev.log_std == pytest.approx(float(model.log_std.detach()))
    dev.close()
    env.close()


def test_update_lowers_the_loss_and_leaves_the_policy_trained():
    env = small_env()
    model = make_model(15, seed=23, scale=1.5)
    dev = DevicePolicy.from_torch(model)
    buf = DeviceRolloutBuffer(env, 4)
    device_ppo_rollout(env, dev, buf, ring_only=True)
    T, rows = buf.actions_raw.shape
    n = T * rows
    adv = ppo_adv_stats(buf, 1, n)[0]
    before = dev.ppo_grad(buf, 1, 0, n, adv)[1][5].item()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, eps=1e-5)
    device_ppo_update(model, dev, buf, opt, n_epochs=5, n_minibatches=4, seed=2)      # 20 minibatch steps
    after = dev.ppo_grad(buf, 1, 0, n, adv)[1][5].item()
    assert after < before, (before, after)
    fresh = DevicePolicy.from_torch(model)
    for a, b in zip(dev.step(env, seed=3)[:4], fresh.step(env, seed=3)[:4]):
        assert torch.equal(a, b)
    fresh.close()
    dev.close()
    env.close()
