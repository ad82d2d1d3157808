"""Data-parallel PPO (device_ppo_update over a torch.distributed group, env shards by global index): per rank, the
rollout, the update, the exchange per minibatch (the all-gather of one partial vector) and one PPO iteration in
env-steps/s of the whole job.

  config 4: MLP 784-64-10, 60 000-row synthetic set, max_history 5, ring-only env steps, 4 epochs x 4 minibatches

    torchrun --nproc_per_node=G tests/ppo_dist_bench.py out_path [strong|capability|weak]...

  strong      4096 envs over the G ranks, n_steps = 8
  capability  4096 envs over the G ranks, n_steps = 64 (the buffer of one rank holds 64 steps of 4096 / G envs)
  weak        4096 envs per rank, n_steps = 8

Per rank, the rollout and the update are CUDA-event times on that rank's stream, read before any barrier, so they
show imbalance between ranks (the update's collectives still wait for the slowest rank).  The PPO iteration is a host
clock around rollout + update that ends in a device synchronise and a barrier: the job's wall time.  The strong-scaling
efficiency is against a one-GPU run (``group=None``, all 4096 envs on rank 0) made in the same invocation.  Rank 0
appends the results of every rank and the card name and power limit (read in the same run) to out_path, and a line to
the INDEX.md beside it if there is one."""
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                     # noqa: E402
from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec   # noqa: E402
from custom_envs_b200.sharding import shard_bases, shard_range   # noqa: E402
from custom_envs_b200.vectorize.device_policy import (DevicePolicy, DeviceRolloutBuffer,   # noqa: E402
                                                      device_ppo_rollout, device_ppo_update)
from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy   # noqa: E402

N_EPOCHS, N_MINIBATCHES = 4, 4


def card(index):
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader',
                              '-i', str(index)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ''
    return out or torch.cuda.get_device_name(index) + ' (power limit not readable)'


def synced():
    torch.cuda.synchronize()
    dist.barrier()
    return time.perf_counter()


def events_ms(fn):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop)


def run(mode, rank, world, device, group):
    """One mode on this rank; `group` None = a one-GPU run (rank 0 alone, all envs)."""
    total_envs = 4096 * world if mode == 'weak' else 4096
    n_steps = 64 if mode == 'capability' else 8
    first, count = shard_range(total_envs, world, rank)
    feats, labels = bench.synthetic_data()
    env = BatchedOptEnv(ProblemSpec('softmax', bench.D, (bench.HID,), bench.C), feats, labels, count, batch_size=32,
                        max_batches=400, max_history=5, seeds=list(range(first, first + count)), init_seed=1,
                        materialize_obs=False, device=device, env_base=first)
    env.reset()
    torch.manual_seed(0)
    model = SharedMlpPolicy(env.obs_dim).to(device)
    policy = DevicePolicy.from_torch(model)
    policy.set_row_base(shard_bases(total_envs, world, rank, env.num_params)[1])
    buf = DeviceRolloutBuffer(env, n_steps)
    opt = torch.optim.Adam(model.parameters(), lr=3e-4, eps=1e-5)
    device_ppo_rollout(env, policy, buf)                                              # warm-up of every shape
    device_ppo_update(model, policy, buf, opt, n_epochs=1, n_minibatches=N_MINIBATCHES, seed=0, group=group)
    sync = synced if group is not None else lambda: (torch.cuda.synchronize(), time.perf_counter())[1]
    t0 = sync()
    rollout = events_ms(lambda: device_ppo_rollout(env, policy, buf))
    update = events_ms(lambda: device_ppo_update(model, policy, buf, opt, n_epochs=N_EPOCHS,
                                                 n_minibatches=N_MINIBATCHES, seed=1, group=group))
    t_iter = (sync() - t0) * 1e3
    exchange = 0.0
    if group is not None:       # the exchange alone: one partial vector per rank, as the update gathers it per minibatch
        partial = torch.zeros(policy.ppo_partial_size, dtype=torch.float64, device=device)
        partials = torch.empty((world, partial.numel()), dtype=torch.float64, device=device)
        reps = 50
        dist.all_gather_into_tensor(partials, partial)
        synced()
        exchange = events_ms(lambda: [dist.all_gather_into_tensor(partials, partial) for _ in range(reps)]) / reps
    steps = N_EPOCHS * N_MINIBATCHES
    mine = torch.tensor([count, env.num_rows, rollout, update, update / steps, exchange], dtype=torch.float64, device=device)
    if group is not None:
        table = torch.empty((world, mine.numel()), dtype=torch.float64, device=device)
        dist.all_gather_into_tensor(table, mine)
    else:
        table = mine[None]
    exch_bytes = 8 * policy.ppo_partial_size
    policy.close()
    del buf
    env.close()
    torch.cuda.empty_cache()
    return total_envs, n_steps, table.cpu().tolist(), t_iter, exch_bytes


def main():
    device = torch.device('cuda', int(os.environ.get('LOCAL_RANK', 0)))
    torch.cuda.set_device(device)
    dist.init_process_group('nccl', device_id=device)
    rank, world = dist.get_rank(), dist.get_world_size()
    out_path = sys.argv[1]
    modes = sys.argv[2:] or ['strong']
    lines, summary = [], []
    if rank == 0:
        lines.append('== %d rank(s), one per GPU; GPU 0: %s' % (world, card(device.index)))
    try:
        single = None
        if 'strong' in modes:           # the one-GPU reference of the same invocation: rank 0 alone, group=None
            if rank == 0:
                total_envs, n_steps, table, t_iter, _ = run('strong', 0, 1, device, None)
                single = total_envs * n_steps / t_iter * 1e3
                lines.append('one GPU (group=None, rank 0 alone): 4096 envs, n_steps 8: rollout %.1f ms, update %.1f ms = '
                             '%.1f ms per minibatch step; one PPO iteration %.1f ms, %.0f env-steps/s'
                             % (table[0][2], table[0][3], table[0][4], t_iter, single))
                print(lines[-1], flush=True)
            dist.barrier()
        for mode in modes:
            if mode == 'capability' and world == 1:
                continue                                  # 64 steps of 4096 envs do not fit one card
            total_envs, n_steps, table, t_iter, exch_bytes = run(mode, rank, world, device, dist.group.WORLD)
            rate = total_envs * n_steps / t_iter * 1e3
            if rank == 0:
                lines.append('%s: %d envs in all, n_steps %d, %d epochs x %d minibatches; partial vector %d B per rank'
                             % (mode, total_envs, n_steps, N_EPOCHS, N_MINIBATCHES, exch_bytes))
                for r, (count, rows, rollout, update, per_mb, exchange) in enumerate(table):
                    lines.append('  rank %d: %d envs (%d agent rows): rollout %.1f ms, update %.1f ms = %.1f ms per '
                                 'minibatch step, exchange %.3f ms per minibatch (device events)'
                                 % (r, count, rows, rollout, update, per_mb, exchange))
                eff = ''
                if mode == 'strong':
                    eff = ('; strong-scaling efficiency against the one-GPU %.0f env-steps/s of this run: %.2f'
                           % (single, rate / (single * world)))
                lines.append('  one PPO iteration (rollout + update, wall clock): %.1f ms, %.0f env-steps/s%s'
                             % (t_iter, rate, eff))
                summary.append('%s %.0f env-steps/s' % (mode, rate))
                print('\n'.join(lines[-len(table) - 2:]), flush=True)
    finally:
        if rank == 0:
            os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
            with open(out_path, 'a') as f:
                f.write('\n'.join(lines) + '\n')
            index = os.path.join(os.path.dirname(out_path), 'INDEX.md')
            if summary and os.path.exists(index):          # a row after the last row of its table
                row = ('| `%s` | `tests/ppo_dist_bench.py` under torchrun, %d GPU(s): data-parallel PPO at config 4 '
                       '(ring-only, H = 5), per-rank rollout / update / exchange times, PPO-iteration env-steps/s (%s) |'
                       % (os.path.basename(out_path), world, ', '.join(summary)))
                with open(index) as f:
                    rows = f.read().split('\n')
                last = max([i for i, line in enumerate(rows) if line.startswith('|')], default=len(rows) - 1)
                with open(index, 'w') as f:
                    f.write('\n'.join(rows[:last + 1] + [row] + rows[last + 1:]))
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
