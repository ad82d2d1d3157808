"""PPO rollouts on the device (DevicePolicy.step / value, b2p_gae, device_ppo_rollout): ms per rollout step split
into env step / step kernel / amortised GAE, env-steps/s of the whole rollout, the step kernel's tanh rate and the
GAE kernel's share of the HBM peak and of a plain device copy's rate on the same card.

  config 4: 4096 envs, MLP 784-64-10, 60 000-row synthetic set, n_steps = 8, ring-only env steps (policy on the rings)
  config 3 shape (softmax regression 784 -> 10, 4096 envs), dense path: the env writes observation rows

    python tests/ppo_rollout_bench.py [out_path] [envs] [n_steps]

The card's name and power limit are read in the same run and printed with the numbers."""
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                     # noqa: E402
from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations_device   # noqa: E402
from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer,   # noqa: E402
                                                      device_ppo_rollout, gae)
from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy   # noqa: E402

MUFU_PROBE_TANH_PER_S = 4643e9      # profiles/r2_mufu_rate_probe.txt (tanh.approx.f32, all SMs)
HBM_PEAK = 7.7e12                   # B200 data sheet, bytes/s

out_path = sys.argv[1] if len(sys.argv) > 1 else None
envs = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
n_steps = int(sys.argv[3]) if len(sys.argv) > 3 else 8
lines = []


def say(text):
    print(text, flush=True)
    lines.append(text)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name(0) + ' (power limit not readable)'


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


def run(hidden, ring_only, label):
    feats, labels = bench.synthetic_data()
    perms = env_permutations_device(bench.ROWS, list(range(envs)), 'cuda:0')
    env = BatchedOptEnv(ProblemSpec('softmax', bench.D, hidden, bench.C), feats, labels, envs, batch_size=32,
                        max_batches=400, max_history=5, perms=perms, init_seed=1, materialize_obs=not ring_only)
    env.reset()
    torch.manual_seed(0)
    policy = DevicePolicy.from_torch(SharedMlpPolicy(env.obs_dim).cuda())
    buf = DeviceRolloutBuffer(env, n_steps)
    rows, T = env.num_rows, n_steps
    say('%s: %d envs, %d agent rows, n_steps %d, buffer %.1f GB' % (label, envs, rows, T,
        sum(t.numel() * t.element_size() for t in (buf.obs_bf16, buf.actions_raw, buf.values, buf.neglogp,
                                                   buf.advantages, buf.returns, buf.rewards, buf.dones)) / 1e9))
    source = env if ring_only else env.obs
    act = torch.empty(rows, device='cuda')
    actions = torch.rand(rows, device='cuda') * 2
    t_act = timed(lambda: policy.act_env(env, act) if ring_only else policy.act(env.obs, act), 5)
    t_step = timed(lambda: policy._launch(source, policy._seed(None), buf.actions, buf.actions_raw[0], buf.values[0],
                                          buf.neglogp[0], buf.obs_bf16[0]), 5)
    t_value = timed(lambda: policy.value(source, out=buf.values[T]), 5)
    t_env = timed(lambda: env.step(actions, ring_only=ring_only), 5)
    t_gae = timed(lambda: gae(buf.values, buf.rewards, buf.dones, buf.rows_per_env, 0.99, 0.95,
                              buf.advantages, buf.returns), 5)
    # the same card's rate for a plain device copy of the same order of size (read T x rows, write T x rows), the
    # yardstick of the streaming GAE kernel
    t_copy = timed(lambda: buf.advantages.copy_(buf.values[:T]), 5)
    copy_bytes = 2 * T * rows * 4
    device_ppo_rollout(env, policy, buf, ring_only=ring_only)          # warm-up rollout
    torch.cuda.synchronize()
    reps = 3
    t0 = time.perf_counter()
    finished = 0
    for _ in range(reps):
        finished += device_ppo_rollout(env, policy, buf, ring_only=ring_only)[1]   # ends in a device sync (.item())
    t_roll = (time.perf_counter() - t0) / reps * 1e3
    gae_bytes = rows * (4 * (T + 1) + 8 * T) + envs * (4 * T + T)
    say('  policy kernel, action only (b2p_act%s): %.3f ms' % ('_env' if ring_only else '', t_act))
    say('  step kernel, all five outputs (b2p_step%s): %.3f ms = %.2f x the action-only kernel; %.0f G tanh/s = %.2f of '
        'the %.0f G/s MUFU probe' % ('_env' if ring_only else '', t_step, t_step / t_act, rows * 256 / t_step / 1e6,
                                     rows * 256 / t_step / 1e-3 / MUFU_PROBE_TANH_PER_S, MUFU_PROBE_TANH_PER_S / 1e9))
    say('  value tower alone (model.value): %.3f ms' % t_value)
    say('  env step (%s): %.3f ms' % ('ring-only' if ring_only else 'with observation rows', t_env))
    say('  GAE over %d steps: %.3f ms (%.3f ms per rollout step), %.2f GB, %.2f TB/s = %.2f of the 7.7 TB/s HBM peak'
        % (T, t_gae, t_gae / T, gae_bytes / 1e9, gae_bytes / t_gae / 1e9, gae_bytes / t_gae / 1e9 / (HBM_PEAK / 1e12)))
    say('  plain device copy (torch copy_, %.2f GB read + written): %.3f ms, %.2f TB/s = %.2f of the HBM peak; GAE runs at '
        '%.2f of this copy rate' % (copy_bytes / 1e9, t_copy, copy_bytes / t_copy / 1e9, copy_bytes / t_copy / 1e9 / 7.7,
                                    (gae_bytes / t_gae) / (copy_bytes / t_copy)))
    say('  rollout (device_ppo_rollout, %d steps + value + GAE): %.2f ms per rollout step = env %.3f + step kernel %.3f '
        '+ final value %.3f + GAE %.3f (both amortised) + rest (copies, launches, Python) %.3f; %.0f env-steps/s '
        '(%d episodes ended in %d rollouts)'
        % (T, t_roll / T, t_env, t_step, t_value / T, t_gae / T, t_roll / T - t_env - t_step - t_value / T - t_gae / T,
           envs * T / t_roll * 1e3, finished, reps))
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
