#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched optimise-env step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          # the CUDA path (this repo)
    python bench.py --impl reference --gpus N ...          # the reference algorithm on host CPUs
    python bench.py --envs-total E --gpus N ...            # strong scaling: E envs sharded over N GPUs
    python bench.py ... --dump-outputs DIR                 # also write the last timed step's outputs to DIR/*.npy

Workload (N=1): BASELINE.json configs[3], the configuration the headline target is quoted
on: MultiOptLRs, 2-layer MLP 784->64->10 on synthetic MNIST-shaped data (60000 rows),
minibatch 32, max_history 5, 4096 lock-step envs per GPU (weak scaling: 4096 x N envs).
One "step" = one batched env step over all envs = one b2e_step call (for this workload a
pipeline of four kernels: tcgen05 eval, update, tcgen05 eval, observations + two tiny
bookkeeping launches).  The timed window contains one episode end of every env (the step
counters are advanced so that all envs hit max_batches in the middle of the window and are
re-initialised by the library's auto-reset, as the reference's workers do).

Reported on one JSON line:
  value     env-steps/s with actions already in HBM (device API, CUDA events, max over ranks)
  e2e       the same metric through the reference-facing OptVecEnv.step() with HOST numpy
            buffers: H2D of the actions and D2H of observations/rewards/dones/infos inside
            the timed region
  roofline  SURVEY 8d: algorithmic bytes of the whole step (4*[P*(5H+3)+B*(D+1)] per env-step)
            / step time, against the measured HBM copy bandwidth; the per-kernel figures
            (own algorithmic bytes / own CUDA-event duration) are listed beside it
  parity    one more step after the timed loop, replayed by the oracle for six sampled envs
            (first two, E/3, 2E/3, last two) from the device's own state
  cpu_baseline  the oracle on the host cores, on a bounded sample of the same workload:
            "port" = vectorised numpy (SURVEY 8d path ii), "faithful" = per-env Python
            objects, thread per env over pipes (path i)

--dump-outputs DIR writes what the last timed step returned on rank 0 (see dump_outputs). Data,
permutations, initial weights and actions are all seeded, so two builds run with the same
arguments get the same inputs and their files can be compared array for array.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D, HID, C, BATCH, ROWS, HIST = 784, 64, 10, 32, 60000, 5
MAX_BATCHES = 400                 # the envs' default episode length (envs/multioptlrs.py:39)
NUM_PARAMS = D * HID + HID + HID * C + C
BYTES_PER_ENV_STEP = 4 * (NUM_PARAMS * (5 * HIST + 3) + BATCH * (D + 1))      # 5 800 160
WORKLOAD = 'MultiOptLRs MLP 784-64-10, B=32, H=5, 60000x784 synthetic rows'


def synthetic_data(rows=ROWS):
    rng = np.random.RandomState(0)
    feats = rng.uniform(size=(rows, D)).astype(np.float32)
    lo, hi = feats.min(0), feats.max(0)
    feats = ((feats - lo) / (hi - lo + 1e-8)).astype(np.float32)      # utils_math.normalize
    labels = rng.randint(0, C, size=rows).astype(np.int32)
    return feats, labels


@contextlib.contextmanager
def stdout_to_stderr():
    """File descriptor 1 points at stderr inside the block, so that lines native libraries write to
    stdout do not end up next to the one JSON line."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        yield
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic():
    """DRAM bytes per launch of the step kernel from the committed ncu capture, if any."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh).get('dram_bytes_per_launch')
    return None


class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.lines, self.proc, self.first = index, [], None, 0

    def mark(self):
        """The timed region starts now: earlier samples are dropped."""
        self.first = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY,
                 '--format=csv,noheader,nounits', '-lms', '50'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines[self.first:]:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, flag in zip(names, parts[5:9]):
                if flag.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': max(smax) if smax else None, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------- CPU (oracle) arm
CPU_ROWS = 4096          # data-set rows of the CPU arms (the minibatch stream touches 32 rows per env-step either way)


def cpu_faithful(max_seconds=25.0):
    """SURVEY 8d path (i): per-env Python objects (oracle/faithful_env.py), one thread per env
    over pipes.  The per-agent Python work holds the GIL, so the rate does not grow with the
    thread count; runs E_cpu in {1, min(cores, 4)} for as many steps as the time box allows."""
    from oracle import faithful_env as fe
    from oracle import optenv_oracle as orc
    feats, labels = synthetic_data(CPU_ROWS)
    spec = orc.ProblemSpec('softmax', D, (HID,), C)
    cores = os.cpu_count() or 1
    runs, t_start = [], time.perf_counter()
    for num_envs, steps in ((1, 4), (min(cores, 4), 2)):
        if time.perf_counter() - t_start > max_seconds:
            break
        value, elapsed = fe.env_steps_per_s(spec, feats, labels, num_envs, steps, warmup=0,
                                            batch_size=BATCH, max_batches=400, max_history=HIST)
        runs.append({'envs': num_envs, 'threads': num_envs, 'steps': steps, 'env_steps_per_s': value,
                     'seconds': elapsed})
    best = max(r['env_steps_per_s'] for r in runs)
    return {'value': best, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port-faithful',
            'runs': runs, 'rows': CPU_ROWS,
            'sample': 'per-env Python env objects (History, per-agent dicts, 14 info statistics) over the '
                      'oracle\'s numpy float32 problem, thread per env + pipes; extrapolation to 4096 envs is linear'}


def cpu_env_steps_per_s(envs_per_thread, threads, steps, warmup):
    """The oracle's vectorised numpy path (float32 problem arithmetic, the reference's
    float64 env arithmetic), one oracle instance per host thread."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import optenv_oracle as orc
    feats, labels = synthetic_data(CPU_ROWS)
    spec = orc.ProblemSpec('softmax', D, (HID,), C)
    perm = orc.env_permutation(len(feats), 0)

    def make(i):
        env = orc.BatchedOptEnvOracle(spec, feats, labels, envs_per_thread, batch_size=BATCH,
                                      config=orc.EnvConfig.multioptlrs(400, HIST),
                                      perms=np.tile(perm, (envs_per_thread, 1)),
                                      compute_dtype=np.float32, init_seed=i)
        vec = orc.OptVecEnvOracle(env)
        vec.reset()
        rng = np.random.RandomState(2 + i)
        acts = rng.uniform(0, 3, size=vec.num_envs).astype(np.float32)
        return vec, acts

    workers = [make(i) for i in range(threads)]

    def run(worker, count):
        vec, acts = worker
        for _ in range(count):
            vec.step(acts)

    with ThreadPoolExecutor(threads) as pool:
        list(pool.map(lambda w: run(w, warmup), workers))
        t0 = time.perf_counter()
        list(pool.map(lambda w: run(w, steps), workers))
        elapsed = time.perf_counter() - t0
    return envs_per_thread * threads * steps / elapsed, elapsed


def reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    envs_per_thread = 8
    value, elapsed = cpu_env_steps_per_s(envs_per_thread, threads, args.steps, args.warmup)
    sample = ('%d envs (%d threads x %d) x %d steps of the workload, oracle numpy float32, %d-row data set '
              '(the GPU arm: 60000 rows; 32 rows per env-step are touched either way)' % (
                  envs_per_thread * threads, threads, envs_per_thread, args.steps, CPU_ROWS))
    line = {
        'impl': 'reference', 'metric': 'env-steps/sec', 'value': value, 'unit': 'env-steps/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * elapsed / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'envs_per_step': envs_per_thread * threads,
                   'note': 'reference algorithm (oracle port) on host CPU; TensorFlow/gym '
                           'are not installable so the reference itself cannot run'},
        'cpu_baseline': {'value': value, 'unit': 'env-steps/s', 'cores': threads, 'kind': 'port',
                         'threads': threads, 'envs_per_thread': envs_per_thread, 'rows': CPU_ROWS,
                         'sample': sample},
        'e2e': {'value': value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------- GPU arm
DUMP_OBS_ROWS = 1 << 18           # observation rows written by --dump-outputs: 262144 x 15 float32 = 15.7 MB


def dump_outputs(out_dir, obs, reward, done, info):
    """Write the outputs of one env.step() to out_dir/<name>.npy, every value finite: obs [rows, obs_dim]
    float32, reward [E] float32, done [E] float32 (0 / 1), info [E, 16] float64 and info_nonfinite
    [E, 16] float32.  info holds non-finite values by design, as the reference does: the loss column is
    NaN (the reference's None) unless the episode ended, and sums of ratios that nan_to_num set to the
    float maximum overflow to +inf.  Such entries are written as 0 in info.npy and marked in
    info_nonfinite.npy (0 finite, 1 NaN, 2 +inf, 3 -inf).  At the bench shape the observation matrix
    is 12.5 GB, so only a fixed sample of DUMP_OBS_ROWS of its rows is written:
    np.random.default_rng(0).choice(rows, DUMP_OBS_ROWS, replace=False), sorted (every row when
    there are no more than that)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rows = obs.shape[0]
    if rows > DUMP_OBS_ROWS:
        pick = np.sort(np.random.default_rng(0).choice(rows, DUMP_OBS_ROWS, replace=False))
        obs = obs.index_select(0, torch.as_tensor(pick, device=obs.device))
    info = info.double().cpu().numpy()
    nonfinite = np.select([np.isnan(info), np.isposinf(info), np.isneginf(info)], [1, 2, 3], 0).astype(np.float32)
    arrays = {'obs': obs.float().cpu().numpy(), 'reward': reward.float().cpu().numpy(),
              'done': done.float().cpu().numpy(), 'info': np.where(nonfinite == 0, info, 0.0),
              'info_nonfinite': nonfinite}
    for name, array in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), array)


def sampled_parity(env, feats, labels, actions, max_batches=MAX_BATCHES, depth=HIST, spec=None):
    """One env step checked against the oracle for the sampled envs {0, 1, E/3, 2E/3, E-2, E-1}:
    the oracle (the checker, oracle/step_check.py) is seeded with the device's own state of those
    envs and replays the step; new weights, loss, reward, done and the newest observation
    column of each block at the bar of the parity tests, the older columns bit for bit against
    the previous observation.  Mutates ``env`` by that one step."""
    import torch
    from oracle import optenv_oracle as orc
    from oracle import step_check
    spec = spec or orc.ProblemSpec('softmax', D, (HID,), C)
    num_envs, num_params = env.num_envs, env.num_params
    sample = sorted({0, 1, num_envs // 3, 2 * num_envs // 3, num_envs - 2, num_envs - 1} & set(range(num_envs)))
    pick = torch.as_tensor(sample, device=env.device)
    perm = orc.lexicographic_rows(num_params)

    def rows_of(tensor):                       # [E*P, ...] -> sampled envs, natural parameter order
        rows = tensor.reshape(num_envs, num_params, -1)[pick].cpu().numpy()
        nat = np.empty_like(rows)
        nat[:, perm] = rows
        return nat

    idx, cnt = env.batch_indices()
    state = {'params': env.get_state('params')[pick].cpu().numpy(),
             'grad_prev': env.get_state('grad_prev')[pick].cpu().numpy(),
             'loss_prev': env.get_state('raw_losses')[pick, 0].cpu().numpy(),      # newest entry of the raw loss history
             'step': env.get_state('step')[pick].cpu().numpy(),
             'idx': idx[pick].cpu().numpy(), 'cnt': cnt[pick].cpu().numpy()}
    obs_prev = rows_of(env.obs)
    act_nat = rows_of(actions)[:, :, 0]
    obs, reward, done, info = env.step(actions)
    device = {'params': env.get_state('params')[pick].cpu().numpy(), 'loss': info[pick, 1].cpu().numpy(),
              'reward': reward[pick].cpu().numpy(), 'done': done[pick].cpu().numpy().astype(bool),
              'obs': rows_of(obs), 'obs_prev': obs_prev}
    ref, ref_obs, ref_reward, ref_done, _ = step_check.replay_step(spec, feats, labels, state, act_nat,
                                                                   max_batches=max_batches, depth=depth)
    stats = step_check.compare_step(ref, ref_obs, ref_reward, ref_done, state, device, depth=depth)
    stats['envs'] = sample
    return stats


def gpu_arm(args):
    import torch
    import torch.distributed as dist
    from custom_envs_b200.batched_env import BatchedOptEnv, ProblemSpec, env_permutations_device
    from custom_envs_b200.vectorize.optvecenv import DeviceOptVecEnv

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        with stdout_to_stderr():              # NCCL prints its version banner when the communicator is made
            dist.init_process_group('nccl', device_id=device)
            dist.barrier()
    numa_node = -1
    if os.environ.get('B2E_NUMA_BIND', '1') != '0':
        # one process per GPU: run on (and first-touch the pinned staging buffers of the e2e
        # path in) the NUMA node the GPU hangs off; no-op where the platform reports none
        from custom_envs_b200.sharding import bind_to_gpu_numa, device_pci_bus_id
        try:
            numa_node = bind_to_gpu_numa(device_pci_bus_id(local))
        except (AttributeError, RuntimeError):
            numa_node = -1
    feats, labels = synthetic_data()
    # envs shard by index (custom_envs_b200/sharding.py): weak scaling gives every rank args.envs envs,
    # --envs-total E shards E envs contiguously over the ranks (strong scaling); seeds follow the global index
    if args.envs_total:
        from custom_envs_b200.sharding import shard_range
        first_env, envs = shard_range(args.envs_total, world, rank)
        envs_all = args.envs_total
    else:
        first_env, envs, envs_all = rank * args.envs, args.envs, args.envs * world
    seeds = range(first_env, first_env + envs)
    perms = env_permutations_device(ROWS, list(seeds), device)   # numpy's RandomState(seed).shuffle, generated on the device
    env = BatchedOptEnv(ProblemSpec('softmax', D, (HID,), C), feats, labels, envs,
                        batch_size=BATCH, max_batches=MAX_BATCHES, max_history=HIST,
                        row_order=args.row_order, perms=perms, device=device,
                        init_seed=1234 + rank)
    del perms
    env.reset()
    gen = torch.Generator(device=device)
    gen.manual_seed(2 + rank)
    actions = [torch.rand(env.num_rows, device=device, generator=gen) * 3.0 for _ in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                       # nvidia-smi needs ~1 s to produce its first line
    for i in range(max(args.warmup, 3)):
        env.step(actions[i & 1])
    env.done.sum()                            # load torch's reduction kernel now: the timed window calls it once
    barrier()
    if rank == 0:
        deadline = time.time() + 3.0
        while not sampler.lines and time.time() < deadline:
            time.sleep(0.05)
        sampler.mark()
    # one episode end inside the timed window: every env reaches max_batches at timed step K // 2
    # and is re-initialised by the auto-reset that follows that step
    reset_at = args.steps // 2
    env.set_state('step', torch.full((envs,), MAX_BATCHES - reset_at - 1, dtype=torch.int32, device=device))
    barrier()
    launches0 = env.launch_count
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    done_total = 0
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    start.record()
    for i in range(args.steps):
        env.step(actions[i & 1])
        marks[i].record()                            # per-step profile of the window (read after it)
        if i == reset_at:
            done_total = env.done.sum()              # device tensor, read after the timed region
    stop.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = env.launch_count - launches0
    ms = start.elapsed_time(stop)
    step_ms = [a.elapsed_time(b) for a, b in zip([start] + marks[:-1], marks)]
    done_total = int(done_total.item()) if torch.is_tensor(done_total) else 0
    if world > 1:
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = envs_all * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # env.step() returns these buffers themselves: they hold the last timed step's outputs until the next step
        dump_outputs(args.dump_outputs, env.obs, env.reward, env.done, env.info)

    # ---- parity: one more step, replayed by the oracle for six sampled envs from the device's own state
    parity = sampled_parity(env, feats, labels, actions[0]) if rank == 0 else None

    # ---- cost of a full re-initialisation of every env (b2e_reset), for the amortised figure
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    env.reset()
    ev1.record()
    torch.cuda.synchronize()
    reset_ms = ev0.elapsed_time(ev1)
    for i in range(3):                                  # back to a steady state with valid history rings
        env.step(actions[i & 1])

    # ---- policy in the loop on the device (SURVEY 8f.2): the library's tcgen05 policy kernel reading the env's rings,
    # ring-only env steps; nothing but the action vector and E rewards / flags / info rows exists per step
    policy_loop = None
    if not args.skip_policy_loop:
        try:
            from custom_envs_b200.vectorize.device_policy import DevicePolicy, device_policy_rollout
            from custom_envs_b200.vectorize.device_rollout import SharedMlpPolicy
            torch.manual_seed(5 + rank)
            net = SharedMlpPolicy(env.obs_dim).to(device)
            dev_policy = DevicePolicy.from_torch(net)                   # noise std = exp(log_std) of the network
            device_policy_rollout(env, dev_policy, 3, ring_only=True)
            pl_steps = 10
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            ev0.record()
            device_policy_rollout(env, dev_policy, pl_steps, ring_only=True)
            ev1.record()
            torch.cuda.synchronize()
            pl_ms = ev0.elapsed_time(ev1) / pl_steps
            if world > 1:
                t = torch.tensor([pl_ms], device=device, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                pl_ms = float(t.item())
            policy_loop = {'value': envs_all / (pl_ms * 1e-3), 'unit': 'env-steps/s', 'ms_per_step': pl_ms, 'steps': pl_steps,
                           'what': 'closed loop on the device: b2p_act_env (MlpPolicy 15-64-64-1 tanh, bf16 tcgen05, reads the '
                                   'adjusted-history rings) -> b2e_step(obs_out = NULL); %d agent rows per step and GPU'
                                   % env.num_rows}
            dev_policy.close()
            env.step(actions[0])                                         # a dense step: observation rows are current again
        except Exception as exc:                                        # noqa: BLE001  (auxiliary figure: never lose the line over it)
            policy_loop = {'error': '%s: %s' % (type(exc).__name__, exc)}

    # ---- end to end through the reference-facing VecEnv call with host buffers
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    vec = DeviceOptVecEnv(env)
    host_actions = np.random.RandomState(3 + rank).uniform(0, 3, size=(env.num_rows, 1)).astype(np.float32)
    for _ in range(3):                                       # warm the pinned buffers (first touches
        vec.step(host_actions)                               # of 14 GB of host memory per rank)
    barrier()
    t0 = time.perf_counter()
    e2e_marks, e2e_phases = [t0], {}
    for _ in range(e2e_steps):
        states, rewards, dones, infos = vec.step(host_actions)
        e2e_marks.append(time.perf_counter())
        for name, ms_p in vec.last_timing.items():
            e2e_phases[name] = e2e_phases.get(name, 0.0) + ms_p / e2e_steps
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = envs_all * e2e_steps / e2e_s
    h2d = host_actions.nbytes
    d2h = states.nbytes + env.reward.numel() * 4 + env.done.numel() + env.info.numel() * 8

    # per-kernel durations of the step pipeline (CUDA events recorded inside the library,
    # on the stream the kernels are launched on), averaged over a few extra traced steps
    env.set_trace(True)
    kernel_ms = {}
    traced = 5
    for i in range(traced):
        env.step(actions[i & 1])
        for name, ms_k in env.last_step_kernel_ms().items():
            kernel_ms[name] = kernel_ms.get(name, 0.0) + ms_k / traced
    env.set_trace(False)

    # NCCL is used only for statistics: all-gather per-env episode statistics
    if world > 1:
        from custom_envs_b200.sharding import gather_env_stats
        gather_env_stats(torch.stack([env.reward, env.info[:, 15].float()], dim=1))

    if rank == 0:
        peak, peak_src = measured_peaks()
        # algorithmic bytes of each pipeline kernel per env-step (fp32 words per parameter):
        #   eval: read w (P) + minibatch B*(D+1), write g (P)                        x2
        #   update: read w, g0, action (3P); write w, adj_w (2P)
        #   obs: read g_t, g_prev, 2(H-1) ring slots; write adj_g, 3H observation words
        words = {'eval_kernel<w_prev>': 2 * NUM_PARAMS + BATCH * (D + 1),
                 'update_kernel': 5 * NUM_PARAMS,
                 'eval_kernel<w_new>': 2 * NUM_PARAMS + BATCH * (D + 1),
                 'obs_kernel': (2 + 2 * (HIST - 1) + 1 + 3 * HIST) * NUM_PARAMS}
        if kernel_ms.get('update_kernel', 1.0) < 0.02:
            # fused pipeline: the first eval applies the update in its backward epilogue (reads w
            # and the actions, writes w and the adjusted weights; g0 never reaches HBM)
            kernel_ms.pop('update_kernel')
            kernel_ms = {('eval_kernel<w_prev>+update' if k == 'eval_kernel<w_prev>' else k): v
                         for k, v in kernel_ms.items()}
            words['eval_kernel<w_prev>+update'] = 4 * NUM_PARAMS + BATCH * (D + 1)
        kernels = [{'name': k, 'ms': v, 'bytes': 4 * words[k] * envs,
                    'gbs': 4 * words[k] * envs / (v * 1e-3) / 1e9} for k, v in kernel_ms.items()]
        dominant = max(kernels, key=lambda k: k['ms']) if kernels else None
        launch_ms = ms / args.steps
        step_gbs = BYTES_PER_ENV_STEP * envs / (launch_ms * 1e-3) / 1e9
        cores = os.cpu_count() or 1
        threads = min(cores, 32)
        cpu_steps = args.cpu_steps              # 30: ~12 s of host work on the pool's 16-32 core boxes
        cpu_value, cpu_elapsed = cpu_env_steps_per_s(8, threads, cpu_steps, 1)
        faithful = cpu_faithful() if not args.skip_faithful else None
        line = {
            'metric': 'env-steps/sec', 'value': value, 'unit': 'env-steps/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps,
            'higher_is_better': True, 'scaling': 'strong' if args.envs_total else 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'envs_per_gpu': envs, 'envs_total': envs_all,
                       'agent_rows_total': envs_all * NUM_PARAMS, 'row_order': args.row_order,
                       'actions': 'U[0,3) float32, resident in HBM',
                       'l2': 'per-step working set %.1f GB >> 126 MB L2 (no flush needed)'
                             % (BYTES_PER_ENV_STEP * envs / 1e9),
                       'episode_end_in_window': {'timed_step': reset_at, 'envs_done': done_total,
                                                 'note': 'every env of rank 0 reaches max_batches there and is auto-reset'},
                       'step_ms_in_window': {'median': float(np.median(step_ms)), 'min': float(min(step_ms)),
                                             'max': float(max(step_ms)), 'slowest_step': int(np.argmax(step_ms)),
                                             'note': 'the slowest step is the one that ends every episode and re-initialises the envs'},
                       'full_reset_ms': reset_ms,
                       'reset_amortised_ms_per_step': {'at_400_steps': reset_ms / 400, 'at_100_steps': reset_ms / 100},
                       'obs_tolerance': 'observations: 1e-5 relative on >= 98 % of the well-conditioned entries, '
                                        '20e-5 on all of them (ratios of fp32 quantities, tests/test_gpu_parity.py)',
                       'parallelism': 'env-index shards, dp%d' % world},
            'e2e': {'value': e2e_value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': int(h2d),
                    'd2h_bytes_per_step': int(d2h), 'steps': e2e_steps,
                    'api': 'DeviceOptVecEnv.step(numpy actions) -> numpy states/rewards/dones + infos',
                    'numa_node_bound': numa_node,
                    'host_phase_ms': {k: round(v, 1) for k, v in e2e_phases.items()},
                    'ms_each_step': [round(1e3 * (b - a), 1) for a, b in zip(e2e_marks, e2e_marks[1:])]},
            'gpu_launches': int(launches),
            'clocks': clocks,
            # headline = SURVEY 8d: algorithmic bytes of the WHOLE step / step time (episode end included);
            # the dominant kernel and every pipeline kernel with its own bytes and duration beside it
            'roofline': {'bound': 'hbm', 'achieved': step_gbs, 'peak': peak, 'unit': 'GB/s',
                         'frac': step_gbs / peak, 'traffic': ncu_traffic(), 'peak_source': peak_src,
                         'what': 'whole step: 4*[P*(5H+3)+B*(D+1)] = %d bytes per env-step x %d envs / %.3f ms'
                                 % (BYTES_PER_ENV_STEP, envs, launch_ms),
                         'bytes_per_launch': BYTES_PER_ENV_STEP * envs,
                         'dominant_kernel': ({'name': dominant['name'], 'achieved': dominant['gbs'],
                                              'frac': dominant['gbs'] / peak, 'bytes_per_launch': dominant['bytes'],
                                              'ms': dominant['ms']} if dominant else None),
                         'kernels': [dict(k, frac=k['gbs'] / peak) for k in kernels]},
            'parity': parity,
            'policy_loop': policy_loop,
            'cpu_baseline': {'value': cpu_value, 'unit': 'env-steps/s', 'cores': threads, 'kind': 'port',
                             'threads': threads, 'envs_per_thread': 8, 'rows': CPU_ROWS,
                             'sample': '%d envs x %d steps of the workload (oracle vectorised numpy float32, '
                                       '%d threads x 8 envs, %d-row data set), %.1f s'
                                       % (8 * threads, cpu_steps, threads, CPU_ROWS, cpu_elapsed),
                             'faithful': faithful},
        }
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--gpus', type=int, default=1)
    parser.add_argument('--steps', type=int, default=50)
    parser.add_argument('--warmup', type=int, default=3)
    parser.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    parser.add_argument('--envs', type=int, default=4096, help='envs per GPU')
    parser.add_argument('--row-order', default='lexicographic', choices=['lexicographic', 'natural'])
    parser.add_argument('--e2e-steps', type=int, default=5)
    parser.add_argument('--envs-total', type=int, default=0,
                        help='strong scaling: this many envs sharded over all ranks (overrides --envs)')
    parser.add_argument('--skip-policy-loop', action='store_true', help='skip the device policy-in-the-loop figure')
    parser.add_argument('--skip-faithful', action='store_true', help='skip the ~25 s per-env-object CPU baseline')
    parser.add_argument('--cpu-steps', type=int, default=30, help='steps of the vectorised CPU baseline sample (~12 s at 30)')
    parser.add_argument('--dump-outputs', metavar='DIR', default=None,
                        help='write the outputs of the last timed step (rank 0) to DIR/<name>.npy')
    args = parser.parse_args()
    if args.steps < 1:
        parser.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        parser.error('--dump-outputs writes the outputs of the CUDA path (--impl b200)')
    if args.impl == 'reference':
        reference_arm(args)
        return
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1',
               '--nproc-per-node', str(args.gpus), '--master-addr', '127.0.0.1',
               '--master-port', '29533', os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    gpu_arm(args)


if __name__ == '__main__':
    main()
