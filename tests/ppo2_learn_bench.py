"""PPO2.learn against the hand loop of device_ppo_rollout + device_ppo_update (INTEGRATION section 6), in one
invocation and alternated, at config 4: 4096 envs, MLP 784-64-10, 60 000-row synthetic set, n_steps = 8, 4 epochs x 4
minibatches, rings.

Reported: env-steps/s of both (host clock around whole updates that end in a synchronisation), the trainer's per-step
hook (one device-to-host copy, Monitor replay, callbacks) by the host clock and as the device's idle gap between two
CUDA events, and the OptVecEnv Monitor replay (``replay_env_step``) of 4096 Monitor-wrapped envs by the host clock.
The replay runs on an OptVecEnv of small envs (P = 15): its cost depends on the env count only, and 4096 config-4
fronts would each hold a 50 890-entry observation and action Dict on the host.

    python tests/ppo2_learn_bench.py [out_path] [envs] [n_steps] [rounds]

The card's name, power limit and SM clock are read in the same run.  With envs = 4 on a machine without a GPU the
script stops after checking its arguments and the output path (the CPU rehearsal)."""
import os
import subprocess
import sys
import tempfile
import time
from functools import partial

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                                          # noqa: E402
from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations_device  # noqa: E402
from custom_envs_b200.ppo2 import PPO2, MlpPolicy, frac_of, tf_adam, update_seeds   # noqa: E402
from custom_envs_b200.vectorize.device_policy import DevicePolicy, device_ppo_rollout, device_ppo_update   # noqa: E402
from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy                # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else None
envs = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
n_steps = int(sys.argv[3]) if len(sys.argv) > 3 else 8
rounds = int(sys.argv[4]) if len(sys.argv) > 4 else 3
if envs < 1 or n_steps < 1 or rounds < 1:
    raise SystemExit('envs, n_steps and rounds must be positive')
lines = []


def say(text):
    print(text, flush=True)
    lines.append(text)


def write():
    if out_path:
        os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
        with open(out_path, 'w') as f:
            f.write('\n'.join(lines) + '\n')


def query(fields):
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=' + fields, '--format=csv,noheader', '-i', '0'],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return ''


say('config: %d envs, MLP 784-64-10, n_steps %d, 4 epochs x 4 minibatches, %d alternated rounds' % (envs, n_steps, rounds))
if not torch.cuda.is_available():
    say('no CUDA device: arguments and output path checked, nothing measured')
    write()
    raise SystemExit(0)
say('device: %s' % (query('name,power.limit,clocks.max.sm') or torch.cuda.get_device_name(0)))

feats, labels = bench.synthetic_data()
perms = env_permutations_device(bench.ROWS, list(range(envs)), 'cuda:0')


def make_env():
    return BatchedOptEnv(ProblemSpec('softmax', bench.D, (bench.HID,), bench.C), feats, labels, envs, batch_size=32,
                         max_batches=400, max_history=5, perms=perms, init_seed=1, materialize_obs=False)


# ---- PPO2.learn, with its per-step hook timed from outside
env_a = make_env()
model = PPO2(MlpPolicy, env_a, n_steps=n_steps, seed=1)
hook_host, hook_events = [], []
make_hook = model._step_hook


def timed_hook(callbacks, step_infos):
    inner = make_hook(callbacks, step_infos)

    def on_step(*args):
        begin, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        begin.record()
        t0 = time.perf_counter()
        inner(*args)
        hook_host.append(time.perf_counter() - t0)
        end.record()
        hook_events.append((begin, end))
    return on_step


model._step_hook = timed_hook

# ---- the hand loop, from the same initial model, on the same env and rollout buffer (two 87 GB buffers do not fit)
env_b, buf = env_a, model.buffer
twin = SharedMlpPolicy(env_b.obs_dim).cuda()
twin.load_state_dict(model.model.state_dict())
policy = DevicePolicy.from_torch(twin, low=model.action_low, high=model.action_high)
opt = tf_adam(twin.parameters(), 2.5e-4)
hand_updates = [0]


def hand_update():
    hand_updates[0] += 1
    rollout_seed, permutation_seed = update_seeds(1, hand_updates[0])
    for group in opt.param_groups:
        group['lr'] = 2.5e-4 * frac_of(1, 1)
    device_ppo_rollout(env_b, policy, buf, ring_only=True, seed=rollout_seed)
    device_ppo_update(twin, policy, buf, opt, n_epochs=4, n_minibatches=4, seed=permutation_seed)   # ends in a sync


def learn_update():
    model.learn(model.n_batch, reset_num_timesteps=False)
    torch.cuda.synchronize()


learn_update()                                  # warm-up of both (first launches; the first learn resets the env)
hand_update()
hook_host.clear()
hook_events.clear()
times = {'learn': [], 'hand': []}
for r in range(rounds):
    for name, fn in (('learn', learn_update), ('hand', hand_update)) if r % 2 == 0 else \
            (('hand', hand_update), ('learn', learn_update)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        times[name].append(time.perf_counter() - t0)
torch.cuda.synchronize()
clock = query('clocks.sm') or 'not readable'
steps = envs * n_steps
for name in ('learn', 'hand'):
    t = np.array(times[name])
    say('%-5s: one update (rollout + 4 x 4 minibatches) %.1f ms median (min %.1f, max %.1f), %.0f env-steps/s'
        % (name, 1e3 * np.median(t), 1e3 * t.min(), 1e3 * t.max(), steps / np.median(t)))
overhead = np.median(times['learn']) / np.median(times['hand']) - 1
say('PPO2.learn over the hand loop: %+.2f %% of an update (medians)' % (100 * overhead))
gaps = [b.elapsed_time(e) for b, e in hook_events]
say('per-step hook (D2H copy of [E, 18] float64 = %d KB, replay, callbacks): host clock %.3f ms median, device idle '
    'gap between events %.3f ms median, over %d steps' % (envs * 18 * 8 // 1024, 1e3 * np.median(hook_host),
                                                          np.median(gaps), len(gaps)))
say('SM clock after the timed rounds: %s' % clock)
policy.close()
del model, buf
env_a.close()
torch.cuda.empty_cache()

# ---- the Monitor replay of an OptVecEnv of `envs` Monitor-wrapped envs
from custom_envs.utils.utils_logging import Monitor                                      # noqa: E402
from custom_envs.vectorize.optvecenv import OptVecEnv                                    # noqa: E402
from custom_envs import load_data                                                        # noqa: E402
from custom_envs_b200.compat import make                                                 # noqa: E402
data = load_data('iris', 32)
with tempfile.TemporaryDirectory() as tmp:
    fns = [partial(Monitor, partial(make, 'MultiOptLRs-v0', problem='nn', max_batches=400,
                                    problem_kwargs=dict(layers=(), data_set=data)),
                   os.path.join(tmp, 'env%d' % i), info_keywords=('loss',)) for i in range(envs)]
    vec = OptVecEnv(fns)
    vec.reset()
    rng = np.random.RandomState(0)
    info = np.zeros((envs, 16))
    replay = []
    for t in range(50):
        reward = rng.normal(size=envs).astype(np.float32)
        done = np.zeros(envs, bool) if t % 10 else np.ones(envs, bool)        # every env ends an episode every 10th step
        info[:, 15] = t % 10 + 1
        t0 = time.perf_counter()
        vec.replay_env_step(reward, done, info.copy())
        replay.append(time.perf_counter() - t0)
    vec.close()
replay = np.array(replay)
ends = np.arange(50) % 10 == 0
say('OptVecEnv.replay_env_step of %d Monitor-wrapped envs (host clock): %.3f ms median per step without episode ends, '
    '%.2f ms when every env ends one' % (envs, 1e3 * np.median(replay[~ends]), 1e3 * np.median(replay[ends])))
write()
