"""Wide observation rows (DevicePolicy at max_history > 5): config-4 geometry -- MLP 784-64-10, 4096 envs, ring-only
env steps -- at max_history H = 5 (the narrow kernels, for comparison), 10 and 25 (obs_dim 30 and 75, rows of
W = 32 and 80 bf16 columns).  Per H:

  kernel times (CUDA events over 20 launches after a warm-up): b2p_act_env, b2p_step_env with all five outputs, the
  ring-only env step; rollout env-steps/s (device_ppo_rollout, n_steps the largest of 8 / 4 / 2 the buffer accepts);
  ppo_grad per minibatch (4 minibatches) and torch autograd of the same loss on a micro-batch beside the buffer.

Each kernel's time is set against the larger of two bounds: the special-function units (128 tanh per row for act, 256
for step and grad, at the 4.64 T/s tanh.approx.f32 probe of profiles/r2_mufu_rate_probe.txt) and HBM bytes per row
from shapes (ring reads 8H, observation store 2W, outputs 4 each, gather 2W + 16) at the data sheet's 7.7 TB/s.

    python tests/wide_obs_bench.py [out_path] [envs]

The card's name, power limit and SM clock are read in the same run and printed with the numbers."""
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                     # noqa: E402
from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations_device   # noqa: E402
from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer,   # noqa: E402
                                                      device_ppo_rollout, epoch_key, obs_width, ppo_adv_stats)
from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy   # noqa: E402

MUFU_PROBE_TANH_PER_S = 4643e9      # profiles/r2_mufu_rate_probe.txt (tanh.approx.f32, all SMs)
HBM_PEAK = 7.7e12                   # B200 data sheet, bytes/s
N_MINIBATCHES = 4

out_path = sys.argv[1] if len(sys.argv) > 1 else None
envs = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
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


def bound(ms, rows, tanh_per_row, bytes_per_row):
    """'x of the <unit> bound' for the larger of the two bounds of a kernel that took ms."""
    t_sfu = rows * tanh_per_row / MUFU_PROBE_TANH_PER_S * 1e3
    t_hbm = rows * bytes_per_row / HBM_PEAK * 1e3
    which, t = ('SFU', t_sfu) if t_sfu >= t_hbm else ('HBM', t_hbm)
    return '%.2f of the %s bound (SFU %.2f ms, HBM %.2f ms at %d B/row)' % (t / ms, which, t_sfu, t_hbm, bytes_per_row)


def torch_rate(model, buf, mb_rows):
    """Rows/s of torch autograd of PPO2's loss (fp32, both towers) on a micro-batch of mb_rows gathered rows."""
    n = buf.actions_raw.numel()
    idx = torch.randint(0, n, (mb_rows,), device='cuda')
    obs = buf.obs_bf16.view(n, buf.obs_width)[idx][:, :model.pi[0].in_features].float()
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


def run(H):
    feats, labels = bench.synthetic_data()
    perms = env_permutations_device(bench.ROWS, list(range(envs)), 'cuda:0')
    env = BatchedOptEnv(ProblemSpec('softmax', bench.D, (bench.HID,), bench.C), feats, labels, envs, batch_size=32,
                        max_batches=400, max_history=H, perms=perms, init_seed=1, materialize_obs=False)
    env.reset()
    torch.manual_seed(0)
    model = SharedMlpPolicy(env.obs_dim).cuda()
    policy = DevicePolicy.from_torch(model)
    rows, W = env.num_rows, obs_width(env.obs_dim)
    buf = None
    for T in (8, 4, 2):
        try:
            buf = DeviceRolloutBuffer(env, T)
            break
        except MemoryError as e:
            say('  (n_steps %d: %s)' % (T, e))
    say('max_history %d (obs_dim %d, W %d): %d envs, %d agent rows, n_steps %d (the largest of 8 / 4 / 2 the buffer '
        'accepts), buffer %.1f GB' % (H, env.obs_dim, W, envs, rows, T, rows * T * buf.bytes_per_row_step / 1e9))
    for _ in range(3):                                   # a filled history
        env.step(policy.act_env(env), ring_only=True)
    torch.cuda.synchronize()
    t_act = timed(lambda: policy.act_env(env, buf.actions), 20)
    say('  b2p_act_env: %.3f ms, %s' % (t_act, bound(t_act, rows, 128, 8 * H + 4)))
    t_step = timed(lambda: policy._launch(env, policy._seed(None), buf.actions, buf.actions_raw[0], buf.values[0],
                                          buf.neglogp[0], buf.obs_bf16[0]), 20)
    say('  b2p_step_env, all five outputs: %.3f ms, %s' % (t_step, bound(t_step, rows, 256, 8 * H + 2 * W + 16)))
    clock = query('clocks.sm')
    t_env = timed(lambda: env.step(buf.actions, ring_only=True), 20)
    say('  env step (ring-only): %.3f ms' % t_env)
    device_ppo_rollout(env, policy, buf, ring_only=True)                       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    device_ppo_rollout(env, policy, buf, ring_only=True)                       # ends in a host sync
    t_roll = (time.perf_counter() - t0) * 1e3
    say('  rollout (device_ppo_rollout, %d steps + value + GAE): %.1f ms, %.0f env-steps/s'
        % (T, t_roll, envs * T / t_roll * 1e3))
    n = rows * T
    mb = n // N_MINIBATCHES
    key = epoch_key(1, 0)
    adv = ppo_adv_stats(buf, key, mb)
    grad, stats = policy.ppo_grad(buf, key, 0, mb, adv[0])
    t_grad = timed(lambda: policy.ppo_grad(buf, key, mb, mb, adv[1], grad=grad, stats=stats), 5)
    say('  ppo_grad, one minibatch of %d rows: %.3f ms, %.3g rows/s, %s'
        % (mb, t_grad, mb / t_grad * 1e3, bound(t_grad, mb, 256, 2 * W + 16)))
    say('  SM clock read after the step kernel ran: %s' % (clock or 'not readable'))
    micro = 1 << 26
    while True:                                        # the largest power-of-two micro-batch that fits beside the buffer
        try:
            rate = torch_rate(model, buf, micro)
            break
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            micro //= 2
    say('  torch autograd of the same loss (fp32, both towers), micro-batch of %d rows: %.3g rows/s; the kernel is '
        '%.1f x faster per row' % (micro, rate, (mb / t_grad * 1e3) / rate))
    policy.close()
    del buf
    env.close()
    torch.cuda.empty_cache()


say('device: %s' % (query('name,power.limit,clocks.max.sm') or torch.cuda.get_device_name(0) + ' (power limit not readable)'))
for H in (5, 10, 25):
    run(H)
if out_path:
    os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
    with open(out_path, 'w') as f:
        f.write('\n'.join(lines) + '\n')
