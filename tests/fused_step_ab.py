"""Outputs and time of the fused step of one shape, for comparing two builds of the library.

    python tests/fused_step_ab.py --root TREE --out FILE.npz [--steps 40]

Imports custom_envs_b200 from TREE (a built checkout), runs MultiOptLRs softmax 60 -> 64 -> 10 (P = 4554, the
fused register-tiled kernel) at max_history 3 (optenv_kernel<0, true>) over 2 x 148 + 4 envs with seeded data,
actions and auto-reset (episodes of 10 steps), and writes every step's observation rows, rewards, done flags,
info rows and parameters' SHA-256 plus the last step's arrays and the step times (CUDA events) to FILE.npz.
"""
import argparse
import hashlib
import os
import sys

import numpy as np


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--root', required=True)
    parser.add_argument('--out', required=True)
    parser.add_argument('--steps', type=int, default=40)
    args = parser.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import torch
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(3000, 60)).astype(np.float32)
    labels = rng.randint(0, 10, 3000).astype(np.int32)
    env = BatchedOptEnv(ProblemSpec('softmax', 60, (64,), 10), feats, labels, 300, batch_size=32, max_batches=10,
                        max_history=3, init_seed=7)
    env.reset()
    gen = torch.Generator(device='cuda').manual_seed(1)
    actions = [torch.rand(env.num_rows, device='cuda', generator=gen) * 3.0 for _ in range(args.steps)]
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        env.step(actions[0])
        torch.cuda.synchronize()
    names = sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA})
    digest, times = hashlib.sha256(), []
    for t in range(1, args.steps):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        obs, reward, done, info = env.step(actions[t])
        end.record()
        torch.cuda.synchronize()
        times.append(start.elapsed_time(end))
        for x in (obs, reward, done, info, env.get_state('params')):
            digest.update(x.cpu().numpy().tobytes())
    np.savez(args.out, digest=digest.hexdigest(), obs=obs.cpu().numpy(), reward=reward.cpu().numpy(),
             done=done.cpu().numpy(), info=info.cpu().numpy(), params=env.get_state('params').cpu().numpy(),
             times=np.array(times), kernels=np.array(names))
    print(os.path.abspath(args.root), digest.hexdigest(), 'median step %.4f ms' % np.median(times), names)
    env.close()


if __name__ == '__main__':
    main()
