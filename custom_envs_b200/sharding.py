"""Multi-GPU: envs shard by index, one process per GPU, no collective on the step path.

Envs never interact (reference vectorize/optvecenv.py:70-88 only concatenates their rows),
so rank r owns the contiguous env range ``shard_range(E, world, r)``, keeps a replica of
the data set and steps its own ``BatchedOptEnv``; the VecEnv row order of the whole job is
the concatenation of the shards.  The only exchange is an all-gather of small per-env
episode statistics (NCCL over NVLink on GPUs, gloo in the CPU tests)."""
import torch
import torch.distributed as dist


def shard_range(num_envs, world_size, rank):
    """Contiguous split of ``num_envs`` envs; the first ``num_envs % world_size`` ranks get
    one extra env.  Returns (first_env, count)."""
    base, extra = divmod(int(num_envs), int(world_size))
    count = base + (1 if rank < extra else 0)
    first = rank * base + min(rank, extra)
    return first, count


def shard_bases(num_envs, world_size, rank, rows_per_env):
    """(env_base, row_base) of rank's shard for data-parallel PPO: ``BatchedOptEnv(..., env_base=env_base)`` draws the
    shard's initial and auto-reset parameters by global env index, and ``DevicePolicy.set_row_base(row_base)`` its
    exploration noise by global agent row (the rows of env e are [e P, (e + 1) P) in both VecEnv row orders), so the
    shard's rollout is exactly its envs' part of one unsharded rollout."""
    first, _ = shard_range(num_envs, world_size, rank)
    return first, first * int(rows_per_env)


def shard_seeds(seeds, world_size, rank):
    """Seeds (one per global env index) of the envs this rank owns."""
    first, count = shard_range(len(seeds), world_size, rank)
    return list(seeds[first:first + count])


def gather_env_stats(local_stats, group=None):
    """All-gather per-env statistics ``[E_local, k]`` into ``[E_total, k]`` in global env order.
    Shards may differ in size by one env, so the payload is padded to the largest shard."""
    if not (dist.is_available() and dist.is_initialized()):
        return local_stats
    world = dist.get_world_size(group)
    local_stats = local_stats.contiguous()
    count = torch.tensor([local_stats.shape[0]], device=local_stats.device, dtype=torch.int64)
    counts = [torch.zeros_like(count) for _ in range(world)]
    dist.all_gather(counts, count, group=group)
    counts = [int(c.item()) for c in counts]
    width = max(counts)
    padded = local_stats.new_zeros((width,) + tuple(local_stats.shape[1:]))
    padded[:local_stats.shape[0]] = local_stats
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    return torch.cat([part[:n] for part, n in zip(parts, counts)], dim=0)


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(','):
        if not part:
            continue
        lo, _, hi = part.partition('-')
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def gpu_numa_node(pci_bus_id, sysfs='/sys'):
    """NUMA node the GPU's PCIe root hangs off (-1 when the platform does not say, e.g. in a
    VM).  ``pci_bus_id`` as CUDA prints it: ``0000:1B:00.0`` (domain may have 8 hex digits)."""
    import os
    domain, _, rest = pci_bus_id.lower().partition(':')
    path = os.path.join(sysfs, 'bus/pci/devices', '%s:%s' % (domain[-4:], rest), 'numa_node')
    try:
        with open(path) as fh:
            return int(fh.read().strip())
    except (OSError, ValueError):
        return -1


def device_pci_bus_id(index):
    """``domain:bus:device.0`` of CUDA device ``index`` (what sysfs names the GPU)."""
    props = torch.cuda.get_device_properties(index)
    return '%04x:%02x:%02x.0' % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)


def bind_to_gpu_numa(pci_bus_id, sysfs='/sys'):
    """Pin this process to the CPUs of the GPU's NUMA node, so that the pinned staging
    buffers of the host-facing VecEnv (12.5 GB of observations per step at config 4) are
    first-touched on the memory next to the GPU's PCIe root and the copy threads run there.
    Call before allocating pinned memory.  Returns the node, or -1 if nothing was changed."""
    import os
    node = gpu_numa_node(pci_bus_id, sysfs)
    if node < 0 or not hasattr(os, 'sched_setaffinity'):
        return -1
    try:
        with open(os.path.join(sysfs, 'devices/system/node/node%d/cpulist' % node)) as fh:
            cpus = _parse_cpulist(fh.read())
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return -1
        os.sched_setaffinity(0, allowed)
    except OSError:
        return -1
    return node
