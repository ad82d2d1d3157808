"""PPO updates on the device (ppo_adv_stats, DevicePolicy.ppo_grad, device_ppo_update): per config, the advantage
statistics pass, the gradient kernel per minibatch (ms, rows/s, tanh/s against the MUFU probe, gathered bytes/s), the
whole update (4 epochs x 4 minibatches, with set_weights' syncs and the torch optimizer), one PPO iteration (rollout +
update) in env-steps/s, and torch autograd of the same loss on the largest micro-batch that fits beside the buffer, as
a per-row rate.

  config 4: 4096 envs, MLP 784-64-10, 60 000-row synthetic set, n_steps = 8, ring-only env steps
  config 3 shape (softmax regression 784 -> 10, 4096 envs), dense rows

    python tests/ppo_update_bench.py [out_path] [envs] [n_steps]

Kernel times are CUDA events over warmed-up launches.  The card's name and power limit are read in the same run, and
the SM clock while the gradient kernel runs; they are printed with the numbers.  At config 4 the gradient kernel is
also timed on an L2-resident buffer, to tell the gather bound from the compute side."""
import os
import subprocess
import sys
import time
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                     # noqa: E402
from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations_device   # noqa: E402
from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer,   # noqa: E402
                                                      device_ppo_rollout, device_ppo_update, epoch_key,
                                                      ppo_adv_stats)
from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy   # noqa: E402

MUFU_PROBE_TANH_PER_S = 4643e9      # profiles/r2_mufu_rate_probe.txt (tanh.approx.f32, all SMs)
GATHER_BYTES_PER_ROW = 160          # 32 B observation sector + four 32 B sectors of the scalars, random rows
N_MINIBATCHES, N_EPOCHS = 4, 4

out_path = sys.argv[1] if len(sys.argv) > 1 else None
envs = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
n_steps = int(sys.argv[3]) if len(sys.argv) > 3 else 8
lines = []


def say(text):
    print(text, flush=True)
    lines.append(text)


def query(fields):
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=' + fields, '--format=csv,noheader', '-i', '0'],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return ''


def card():
    return query('name,power.limit,clocks.max.sm') or torch.cuda.get_device_name(0) + ' (power limit not readable)'


def sm_clock_under(fn, seconds=1.0):
    """The SM clock read while fn() is being launched back to back (the clock the kernel runs at)."""
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        fn()
    clock = query('clocks.sm')
    torch.cuda.synchronize()
    return clock or 'not readable'


def timed(fn, reps):
    fn()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / reps


def torch_rate(model, buf, mb_rows):
    """Rows/s of torch autograd of PPO2's loss (fp32, both towers) on a micro-batch of mb_rows gathered rows."""
    n = buf.actions_raw.numel()
    idx = torch.randint(0, n, (mb_rows,), device='cuda')
    obs = buf.obs_bf16.view(n, 16)[idx][:, :model.pi[0].in_features].float()
    act, nlp_old = buf.actions_raw.view(-1)[idx], buf.neglogp.view(-1)[idx]
    v_old, ret = buf.values[:buf.n_steps].reshape(-1)[idx], buf.returns.view(-1)[idx]

    def step():
        mu, V = model(obs)
        A = ret - v_old
        An = (A - A.mean()) / (A.std(unbiased=False) + 1e-8)
        nlp = 0.5 * ((act - mu) / model.log_std.exp()) ** 2 + 0.9189385 + model.log_std
        ratio = torch.exp(nlp_old - nlp)
        pg = torch.max(-An * ratio, -An * ratio.clamp(0.8, 1.2)).mean()
        vc = v_old + (V - v_old).clamp(-0.2, 0.2)
        vf = 0.5 * torch.max((V - ret) ** 2, (vc - ret) ** 2).mean()
        loss = pg - 0.01 * (model.log_std + 1.4189385) + 0.5 * vf
        model.zero_grad(set_to_none=False)
        loss.backward()
    return mb_rows / (timed(step, 3) * 1e-3)


def run(hidden, ring_only, label):
    feats, labels = bench.synthetic_data()
    perms = env_permutations_device(bench.ROWS, list(range(envs)), 'cuda:0')
    env = BatchedOptEnv(ProblemSpec('softmax', bench.D, hidden, bench.C), feats, labels, envs, batch_size=32,
                        max_batches=400, max_history=5, perms=perms, init_seed=1, materialize_obs=not ring_only)
    env.reset()
    torch.manual_seed(0)
    model = SharedMlpPolicy(env.obs_dim).cuda()
    policy = DevicePolicy.from_torch(model)
    buf = DeviceRolloutBuffer(env, n_steps)
    rows, T = env.num_rows, n_steps
    n = rows * T
    mb = n // N_MINIBATCHES
    say('%s: %d envs, %d agent rows, n_steps %d, %d samples, minibatch %d rows' % (label, envs, rows, T, n, mb))
    device_ppo_rollout(env, policy, buf, ring_only=ring_only)
    torch.cuda.synchronize()
    key = epoch_key(1, 0)
    t_adv = timed(lambda: ppo_adv_stats(buf, key, mb), 3)
    adv = ppo_adv_stats(buf, key, mb)
    grad, stats = policy.ppo_grad(buf, key, 0, mb, adv[0])
    t_grad = timed(lambda: policy.ppo_grad(buf, key, mb, mb, adv[1], grad=grad, stats=stats), 5)
    clock = sm_clock_under(lambda: policy.ppo_grad(buf, key, mb, mb, adv[1], grad=grad, stats=stats))
    tanh = mb * 256
    say('  advantage statistics (one epoch, %d minibatches): %.3f ms' % (N_MINIBATCHES, t_adv))
    say('  gradient kernel (b2p_ppo_grad incl. the slot reduction), one minibatch: %.3f ms, %.3g rows/s, %.0f G tanh/s = '
        '%.2f of the %.0f G/s MUFU probe, %.0f GB/s gathered (%d B of sectors per row)'
        % (t_grad, mb / t_grad * 1e3, tanh / t_grad / 1e6, tanh / t_grad / 1e-3 / MUFU_PROBE_TANH_PER_S,
           MUFU_PROBE_TANH_PER_S / 1e9, mb * GATHER_BYTES_PER_ROW / t_grad / 1e6, GATHER_BYTES_PER_ROW))
    say('  SM clock read while the gradient kernel runs back to back: %s' % clock)
    if ring_only:
        # the same kernel on a buffer that stays in the 126 MB L2 (52 B per row): if the random-row gather from HBM
        # were its bound, this would run faster per row
        small = 1 << 20
        sb = types.SimpleNamespace(obs_bf16=buf.obs_bf16.view(-1, 16)[:small].view(1, small, 16),
                                   actions_raw=buf.actions_raw.view(-1)[:small].view(1, small),
                                   neglogp=buf.neglogp.view(-1)[:small].view(1, small),
                                   values=buf.values.view(-1)[:2 * small].view(2, small),
                                   returns=buf.returns.view(-1)[:small].view(1, small))
        sadv = ppo_adv_stats(sb, key, small)
        t_small = timed(lambda: policy.ppo_grad(sb, key, 0, small, sadv[0], grad=grad, stats=stats), 20)
        say('  gradient kernel on an L2-resident buffer of %d rows: %.3f ms, %.3g rows/s (%.2f x the rate on the '
            'random rows of the full buffer)' % (small, t_small, small / t_small * 1e3,
                                                 (small / t_small) / (mb / t_grad)))
    opt = torch.optim.Adam(model.parameters(), lr=3e-4, eps=1e-5)
    device_ppo_update(model, policy, buf, opt, n_epochs=1, n_minibatches=N_MINIBATCHES, seed=0)     # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    device_ppo_update(model, policy, buf, opt, n_epochs=N_EPOCHS, n_minibatches=N_MINIBATCHES, seed=1)   # ends in a sync
    t_upd = (time.perf_counter() - t0) * 1e3
    say('  device_ppo_update (%d epochs x %d minibatches): %.1f ms = %.1f ms per minibatch step'
        % (N_EPOCHS, N_MINIBATCHES, t_upd, t_upd / (N_EPOCHS * N_MINIBATCHES)))
    t0 = time.perf_counter()
    device_ppo_rollout(env, policy, buf, ring_only=ring_only)
    device_ppo_update(model, policy, buf, opt, n_epochs=N_EPOCHS, n_minibatches=N_MINIBATCHES, seed=2)
    t_it = (time.perf_counter() - t0) * 1e3
    say('  one PPO iteration (rollout of %d steps + update): %.1f ms, %.0f env-steps/s' % (T, t_it, envs * T / t_it * 1e3))
    micro = 1 << 26
    while True:                                        # the largest power-of-two micro-batch that fits beside the buffer
        try:
            rate = torch_rate(model, buf, micro)
            break
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            micro //= 2
    say('  torch autograd of the same loss (fp32, both towers), micro-batch of %d rows: %.3g rows/s per row = %.1f x '
        'slower than the kernel (rate of that micro-batch only, not a whole minibatch)'
        % (micro, rate, (mb / t_grad * 1e3) / rate))
    policy.close()
    del buf
    env.close()
    torch.cuda.empty_cache()


say('device: %s' % card())
run((bench.HID,), True, 'config 4 (MLP 784-64-10), ring-only')
run((), False, 'config 3 shape (softmax regression 784-10), dense rows')
if out_path:
    os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
    with open(out_path, 'w') as f:
        f.write('\n'.join(lines) + '\n')
