"""Data-parallel PPO: env shards that roll out exactly their rows of one unsharded run (env_base / row_base), the
partial + combine form of the gradient and of the advantage statistics, and device_ppo_update over a torch.distributed
group.  The float64 reference of the gradient is the one of test_gpu_ppo_update.py."""
import ctypes
import multiprocessing

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import torch.distributed as dist

    from custom_envs_b200 import _lib
    from custom_envs_b200._lib import B200EnvError
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    from custom_envs_b200.sharding import shard_bases, shard_range
    from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer, _model_params, _set_grads,
                                                          device_ppo_rollout, device_ppo_update, load_model,
                                                          obs_width, ppo_adv_combine, ppo_adv_moments, ppo_adv_stats,
                                                          ppo_minibatch_indices, rank_epoch_key)
    from test_gpu_ppo_update import GRAD_TOL, make_model, ppo2_loss64, synthetic_buffer, tensor_errors

LOG_STD = -0.5


# ------------------------------------------------------------------ 1. shards roll out their rows of the whole batch
def shard_env(first, count, max_history, materialize_obs, device='cuda:0', max_batches=3, env_base=None):
    """Envs [first, first + count) of a batch of the config-4 problem shape (MLP 784-64-10, tcgen05 pipeline); the seeds
    follow the global index as a sharded launcher hands them out, and so does the initialiser (env_base = first)."""
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(320, 784)).astype(np.float32)
    labels = rng.randint(0, 10, 320).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 784, (64,), 10), feats, labels, count, batch_size=32,
                        max_batches=max_batches, max_history=max_history, seeds=list(range(100 + first, 100 + first + count)),
                        init_seed=9, materialize_obs=materialize_obs, device=device,
                        env_base=first if env_base is None else env_base)
    env.reset()
    return env


def row_buffers(buf):
    return [buf.obs_bf16, buf.actions_raw, buf.values, buf.neglogp, buf.advantages, buf.returns]


@pytest.mark.parametrize('ring_only', [True, False])
@pytest.mark.parametrize('max_history', [5, 10])
def test_shards_roll_out_their_rows_of_the_unsharded_run(max_history, ring_only):
    E, world, T = 5, 2, 4
    model = make_model(3 * max_history, seed=31, scale=1.5)
    runs = []
    for first, count in [(0, E)] + [shard_range(E, world, r) for r in range(world)]:
        env = shard_env(first, count, max_history, materialize_obs=not ring_only)
        env_base, row_base = shard_bases(E, world, 1, env.num_params) if first else (0, 0)
        assert env_base == first and row_base == first * env.num_params
        dev = DevicePolicy.from_torch(model)
        dev.set_row_base(row_base)
        buf = DeviceRolloutBuffer(env, T)
        snaps, finished = [], 0
        for _ in range(2):                       # max_batches 3 < T: both rollouts cross an auto-reset
            finished += device_ppo_rollout(env, dev, buf, ring_only=ring_only)[1]
            snaps.append([t.clone() for t in row_buffers(buf)] + [buf.rewards.clone(), buf.dones.clone()])
        runs.append((first, count, env.num_params, snaps, finished))
        dev.close()
        env.close()
    whole = runs[0][3]
    assert runs[0][4] == sum(r[4] for r in runs[1:]) > 0
    for first, count, P, snaps, _ in runs[1:]:
        rows, envs = slice(first * P, (first + count) * P), slice(first, first + count)
        for want, got in zip(whole, snaps):
            for i in range(6):
                assert torch.equal(want[i][:, rows], got[i]), (first, i)
            assert torch.equal(want[6][:, envs], got[6]) and torch.equal(want[7][:, envs], got[7]), first


def test_env_base_moves_the_initial_parameters():
    """With its seed but without env_base, env 2 alone starts from env 0's initial weights, not from its own: the offset
    is what makes the shards above hold."""
    whole, shard, plain = shard_env(0, 3, 5, True), shard_env(2, 1, 5, True), shard_env(2, 1, 5, True, env_base=0)
    params = [env.get_state('params') for env in (whole, shard, plain)]
    assert torch.equal(params[0][2:3], params[1])
    assert not torch.equal(params[0][2:3], params[2])
    for env in (whole, shard, plain):
        env.close()


# ------------------------------------------------------------------ 2. one rank is the single-GPU path, bit for bit
def random_buffer(obs_dim, T, rows, seed):
    """Any rollout buffer: bit equality does not depend on the data."""
    import types
    gen = torch.Generator(device='cuda').manual_seed(seed)
    W, n = obs_width(obs_dim), T * rows
    obs16 = torch.zeros((n, W), dtype=torch.bfloat16, device='cuda')
    obs16[:, :obs_dim] = (torch.randn(n, obs_dim, device='cuda', generator=gen) * 1.5).to(torch.bfloat16)
    rnd = lambda k: torch.randn(k, device='cuda', generator=gen)     # noqa: E731
    return types.SimpleNamespace(obs_bf16=obs16.view(T, rows, W), actions_raw=rnd(n).view(T, rows),
                                 neglogp=(1.0 + 0.1 * rnd(n)).view(T, rows), values=rnd(n + rows).view(T + 1, rows),
                                 returns=(rnd(n) + 0.3).view(T, rows))


@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
@pytest.mark.parametrize('obs_dim', [3, 15, 30, 79])
def test_one_rank_partial_and_combine_equal_the_single_gpu_calls(obs_dim, tanh_mode):
    model = make_model(obs_dim, seed=obs_dim + tanh_mode, scale=1.3)
    T, rows, n_mb = 2, 60000, 4
    buf = random_buffer(obs_dim, T, rows, seed=obs_dim)
    n = T * rows
    mb = n // n_mb
    key = rank_epoch_key(11, 1, 0)
    adv = ppo_adv_stats(buf, key, mb)
    moments = ppo_adv_moments(buf, key, mb)
    assert moments.shape == (n_mb, 4) and (moments[:, 0] == mb).all()
    assert torch.equal(ppo_adv_combine(moments[None].contiguous()), adv)
    dev = DevicePolicy.from_torch(model, tanh_mode=tanh_mode)
    assert dev.ppo_partial_size == 2 * (64 * obs_dim + 64 + 64 * 64 + 64 + 64 + 1) + 5
    for m in (0, n_mb - 1):
        kw = dict(cliprange=0.2, cliprange_vf=0.1, ent_coef=0.01, vf_coef=0.5)
        grad, stats = dev.ppo_grad(buf, key, m * mb, mb, adv[m], **kw)
        partial = dev.ppo_grad_partial(buf, key, m * mb, mb, mb, adv[m], **kw)
        g2, s2 = dev.ppo_combine(partial[None].contiguous(), mb, ent_coef=0.01, vf_coef=0.5)
        assert torch.equal(grad, g2) and torch.equal(stats, s2), m
    dev.close()


# ------------------------------------------------------------------ 3. two shards in one process against float64
@pytest.mark.parametrize('tanh_mode', [0, 1, 2])
def test_two_shards_combine_to_the_union_minibatch(tanh_mode):
    """Shards of 3 and 2 of 5 envs (shard_range's uneven split): the combined statistics are numpy's over the union of
    both shards' minibatch rows, and the combined gradient is float64 autograd of PPO2's loss over that union."""
    c, c_vf, obs_dim, T, P, n_mb, seed = 0.2, 0.1, 15, 2, 7001, 4, 5
    model = make_model(obs_dim, seed=40 + tanh_mode, scale=1.3)
    shards = []
    for r in range(2):
        _, count = shard_range(5, 2, r)
        buf, mu, V = synthetic_buffer(model, T, count * P * n_mb // 2, tanh_mode, c, c_vf, seed=r + 10 * tanh_mode)
        shards.append((buf, mu, V))
    Ns = [s[0].actions_raw.numel() for s in shards]
    assert Ns[0] != Ns[1] and all(N % n_mb == 0 for N in Ns)
    mbs = [N // n_mb for N in Ns]
    n_m = sum(mbs)
    keys = [rank_epoch_key(seed, 0, r) for r in range(2)]
    adv = ppo_adv_combine(torch.stack([ppo_adv_moments(s[0], k, mb) for s, k, mb in zip(shards, keys, mbs)]))
    devs = [DevicePolicy.from_torch(model, tanh_mode=tanh_mode) for _ in range(2)]
    for m in (0, 3):
        parts = []
        for (buf, mu, V), key, mb, N in zip(shards, keys, mbs, Ns):
            idx = ppo_minibatch_indices(N, key, m * mb, mb)
            flat = lambda t: t.reshape(-1)[:N]          # noqa: E731  (values: the first T rows)
            parts.append((buf.obs_bf16.reshape(N, 16)[idx], flat(buf.actions_raw)[idx], flat(buf.neglogp)[idx],
                          flat(buf.values)[idx], flat(buf.returns)[idx], mu[idx], V[idx]))
        union = [torch.cat([p[i] for p in parts]) for i in range(7)]
        A = (union[4] - union[3]).double().cpu().numpy()
        got = adv[m].cpu().numpy()
        assert abs(got[0] - A.mean()) <= 1e-12 * abs(A.mean()) and abs(got[1] - A.std()) <= 1e-12 * A.std(), (got, A.mean(), A.std())
        partials = torch.stack([dev.ppo_grad_partial(s[0], key, m * mb, mb, n_m, adv[m], cliprange=c, cliprange_vf=c_vf)
                                for dev, s, key, mb in zip(devs, shards, keys, mbs)])
        grad, stats = devs[0].ppo_combine(partials, n_m)
        loss, want_stats, leaves = ppo2_loss64(model, union[0], union[1], union[2], union[3], union[4], float(got[0]),
                                               float(got[1]), c, c_vf, 0.01, 0.5, tanh_mode, union[5], union[6])
        loss.backward()
        errs = tensor_errors(grad, leaves)
        assert max(errs) <= GRAD_TOL, errs
        s, w = stats.cpu().numpy(), want_stats.cpu().numpy()
        for i in (0, 1, 2, 3, 5):
            assert abs(s[i] - w[i]) <= 1e-4 * max(abs(w[i]), 1e-6), (i, s[i], w[i])
        assert round(s[4] * n_m) == round(w[4] * n_m)
    for dev in devs:
        dev.close()


# ------------------------------------------------------------------ 4 / 5. device_ppo_update over a process group
ITERS, N_EPOCHS, N_MB, E_TOTAL = 3, 2, 2, 5
KW = dict(cliprange=0.2, cliprange_vf=None, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5)


def train(rank, world, device, group):
    """ITERS PPO iterations (rollout of rank's shard, then device_ppo_update over `group`, or alone for None) ->
    (final parameters on the host, statistics of every update)."""
    torch.cuda.set_device(device)
    model = make_model(15, seed=50, scale=1.5)
    first, count = shard_range(E_TOTAL, world, rank)
    env = shard_env(first, count, 5, materialize_obs=False, device=device)
    dev = DevicePolicy.from_torch(model)
    dev.set_row_base(shard_bases(E_TOTAL, world, rank, env.num_params)[1])
    buf = DeviceRolloutBuffer(env, 4)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, eps=1e-5)
    stats = []
    for it in range(ITERS):
        device_ppo_rollout(env, dev, buf, ring_only=True)
        stats.append(device_ppo_update(model, dev, buf, opt, N_EPOCHS, N_MB, seed=7 + it, group=group, **KW))
    params = [p.detach().cpu() for p in model.parameters()]
    dev.close()
    env.close()
    return params, np.stack(stats)


def emulate(world):
    """The ranks of a `world`-rank run as shards on this device, combined in one process with the building blocks."""
    model = make_model(15, seed=50, scale=1.5)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, eps=1e-5)
    shards = []
    for r in range(world):
        first, count = shard_range(E_TOTAL, world, r)
        env = shard_env(first, count, 5, materialize_obs=False)
        dev = DevicePolicy.from_torch(model)
        dev.set_row_base(first * env.num_params)
        shards.append((env, dev, DeviceRolloutBuffer(env, 4)))
    params, stats = _model_params(model), []
    for it in range(ITERS):
        for env, dev, buf in shards:
            device_ppo_rollout(env, dev, buf, ring_only=True)
        mbs = [buf.actions_raw.numel() // N_MB for _, _, buf in shards]
        total = torch.zeros(6, dtype=torch.float64, device='cuda')
        for epoch in range(N_EPOCHS):
            keys = [rank_epoch_key(7 + it, epoch, r) for r in range(world)]
            adv = ppo_adv_combine(torch.stack([ppo_adv_moments(s[2], k, mb) for s, k, mb in zip(shards, keys, mbs)]))
            for m in range(N_MB):
                for _, dev, _ in shards:
                    load_model(dev, model)
                partials = torch.stack([dev.ppo_grad_partial(buf, k, m * mb, mb, sum(mbs), adv[m], KW['cliprange'],
                                                             KW['cliprange_vf'], KW['ent_coef'], KW['vf_coef'])
                                        for (_, dev, buf), k, mb in zip(shards, keys, mbs)])
                grad, st = shards[0][1].ppo_combine(partials, sum(mbs), KW['ent_coef'], KW['vf_coef'])
                _set_grads(params, grad)
                torch.nn.utils.clip_grad_norm_(params, KW['max_grad_norm'])
                opt.step()
                total += st
        for _, dev, _ in shards:
            load_model(dev, model)
        stats.append((total / (N_EPOCHS * N_MB)).cpu().numpy())
    for env, dev, _ in shards:
        dev.close()
        env.close()
    return [p.detach().cpu() for p in model.parameters()], np.stack(stats)


def _worker(rank, world, store, out):
    device = torch.device('cuda', rank)
    torch.cuda.set_device(device)
    dist.init_process_group('nccl', init_method='file://' + store, rank=rank, world_size=world, device_id=device)
    try:
        torch.save(train(rank, world, device, dist.group.WORLD), out % rank)
    finally:
        dist.destroy_process_group()


def spawn_ranks(world, tmp_path, timeout=600):
    """`world` NCCL ranks in spawned processes, joined with a timeout (a straggler is killed and the test fails)."""
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


def assert_same(a, b):
    assert all(torch.equal(x, y) for x, y in zip(a[0], b[0]))
    assert np.array_equal(a[1], b[1]), (a[1], b[1])


@pytest.mark.skipif(not (torch.cuda.is_available() and dist.is_nccl_available()), reason='needs NCCL')
def test_one_rank_group_equals_the_single_gpu_update(tmp_path):
    (got,) = spawn_ranks(1, tmp_path)
    want = train(0, 1, torch.device('cuda', 0), None)
    assert_same(got, want)
    assert np.isfinite(want[1]).all()


@pytest.mark.skipif(torch.cuda.device_count() < 2 or not dist.is_nccl_available(), reason='needs two GPUs and NCCL')
def test_two_ranks_stay_identical_and_equal_the_emulation(tmp_path):
    ranks = spawn_ranks(2, tmp_path)
    assert_same(ranks[0], ranks[1])
    assert_same(ranks[0], emulate(2))


# ------------------------------------------------------------------ 6. errors
def test_errors():
    model = make_model(15, seed=60)
    buf = random_buffer(15, 2, 1000, seed=1)
    dev = DevicePolicy.from_torch(model)
    adv = torch.tensor([0.0, 1.0], dtype=torch.float64, device='cuda')
    size = dev.ppo_partial_size
    with pytest.raises(ValueError, match='partial buffer'):
        dev.ppo_grad_partial(buf, 1, 0, 500, 500, adv, partial=torch.empty(size - 1, dtype=torch.float64, device='cuda'))
    with pytest.raises(B200EnvError, match='count_total'):
        dev.ppo_grad_partial(buf, 1, 0, 500, 499, adv)
    with pytest.raises(ValueError, match='partials'):
        dev.ppo_combine(torch.zeros((2, size - 1), dtype=torch.float64, device='cuda'), 10)
    lib = _lib.load()
    parts = torch.zeros((1, size), dtype=torch.float64, device='cuda')
    grad, stats = torch.empty(size - 4, device='cuda'), torch.empty(6, dtype=torch.float64, device='cuda')
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())      # noqa: E731
    assert lib.b2p_ppo_combine(dev.handle, ptr(parts), 0, 10, -0.5, 0.01, 0.5, ptr(grad), ptr(stats), None)
    assert b'ranks must be' in lib.b2p_last_error(dev.handle)
    assert lib.b2p_ppo_combine(dev.handle, ptr(parts), 1, 0, -0.5, 0.01, 0.5, ptr(grad), ptr(stats), None)
    assert b'count_total' in lib.b2p_last_error(dev.handle)
    moments = torch.zeros((1, 4, 4), dtype=torch.float64, device='cuda')
    assert lib.b2p_ppo_adv_combine(ptr(moments), 0, 4, ptr(stats), None)
    assert b'ranks must be' in lib.b2p_last_error(None)
    assert lib.b2p_ppo_adv_combine(ptr(moments), 1, 0, ptr(stats), None)
    assert b'nmb' in lib.b2p_last_error(None)
    with pytest.raises(ValueError, match='minibatches of'):
        ppo_adv_moments(buf, 1, 7)
    with pytest.raises(B200EnvError, match='row_base'):
        dev.set_row_base(-1)
    with pytest.raises(B200EnvError, match='env_base'):
        shard_env(-1, 2, 5, True)
    dev.close()
