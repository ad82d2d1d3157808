"""Timing of the Adam baseline (b2e_step_adam) next to the action step (b2e_step) on one GPU.

    python tests/adam_bench.py --out DIR [--envs 4096] [--steps 20]

* config 4 (MLP 784-64-10, minibatch 32, 60 000 rows of synthetic MNIST-shaped data, 4096 envs), dense and
  ring-only: per-kernel times of both steps from the pipeline's CUDA-event trace, the two step kinds
  alternated on the same batch; the update kernel's time against the least time its HBM traffic allows
  (Adam: w, g0, m, v read, w, m, v and the ring slot written = 8 words per parameter; the action update:
  w, g0, action read, w and ring slot written = 5)
* config 2 (iris-shaped softmax regression 4 -> 3, 150 rows, 1024 envs): per-step time of both steps,
  eagerly and replayed from a CUDA graph.
Writes DIR/adam_bench.json and prints it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from custom_envs_b200.baselines import DeviceAdam  # noqa: E402
from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec  # noqa: E402

HBM_BYTES_PER_S = 7.7e12              # B200 data sheet, one GPU


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def config4(num_envs, steps):
    rng = np.random.RandomState(0)
    feats = torch.as_tensor(rng.uniform(size=(60000, 784)).astype(np.float32))
    labels = torch.as_tensor(rng.randint(0, 10, 60000).astype(np.int32))
    out = {}
    for ring_only in (False, True):
        env = BatchedOptEnv(ProblemSpec('softmax', 784, (64,), 10), feats, labels, num_envs, batch_size=32,
                            materialize_obs=not ring_only)
        adam = DeviceAdam(env, torch.logspace(-5, -1, num_envs, device=env.device))
        env.reset()
        actions = torch.rand(env.num_rows, device=env.device, generator=torch.Generator('cuda').manual_seed(0))
        env.set_trace(True)
        times = {'step': [], 'step_adam': []}
        for i in range(2 * (steps + 2)):               # alternated: action step, Adam step, ...
            kind = 'step' if i % 2 == 0 else 'step_adam'
            if kind == 'step':
                env.step(actions, ring_only=ring_only)
            else:
                adam.step(ring_only=ring_only)
            torch.cuda.synchronize()
            if i >= 4:                                 # two of each kind as warm-up (the second has m, v to read)
                times[kind].append(env.last_step_kernel_ms())
        env.set_trace(False)
        P, E = env.num_params, env.num_envs
        res = {}
        for kind, rows in times.items():
            med = {k: float(np.median([r[k] for r in rows])) for k in rows[0]}
            words = 8 if kind == 'step_adam' else 5
            bound_ms = words * 4.0 * P * E / HBM_BYTES_PER_S * 1e3
            res[kind] = {'kernel_ms_median': med, 'step_kernels_ms': sum(med.values()),
                         'update_bytes': words * 4 * P * E, 'update_hbm_bound_ms': bound_ms,
                         'update_share_of_hbm_peak': bound_ms / med['update_kernel']}
        out['ring_only' if ring_only else 'dense'] = res
        env.close()
        del env, adam
        torch.cuda.empty_cache()
    return out


def config2(steps):
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(150, 4)).astype(np.float32)
    labels = (np.arange(150) % 3).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 4, (), 3), feats, labels, 1024, batch_size=32)
    adam = DeviceAdam(env, torch.logspace(-4, -1, 1024, device=env.device))
    env.reset()
    actions = torch.rand(env.num_rows, device=env.device)
    calls = {'step': lambda: env.step(actions), 'step_adam': lambda: adam.step()}
    out = {}
    for kind, call in calls.items():
        for _ in range(20):
            call()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            call()
        torch.cuda.synchronize()
        eager = (time.perf_counter() - t0) / steps * 1e6
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            call()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(10):
                call()
        graph.replay()
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(max(steps // 10, 1)):
            graph.replay()
        end.record()
        torch.cuda.synchronize()
        graphed = start.elapsed_time(end) * 1e3 / (max(steps // 10, 1) * 10)
        out[kind] = {'eager_us_per_step': eager, 'graph_us_per_step': graphed}
    env.close()
    return out


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--out', required=True)
    parser.add_argument('--envs', type=int, default=4096)
    parser.add_argument('--steps', type=int, default=20)
    args = parser.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('adam_bench.py measures on a CUDA device; none is visible')
    result = {'card': card(), 'config4_envs': args.envs, 'config4': config4(args.envs, args.steps),
              'config2': config2(2000)}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'adam_bench.json'), 'w') as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == '__main__':
    main()
