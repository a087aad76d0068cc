"""Multi-GPU layout of the env step: environment instances are independent (no cross-env state anywhere
in `step()`, SURVEY §8e), so a job of `n_envs_total` instances is split into contiguous slices, one per
rank / GPU, each rank owning its handle, state and output buffers.  There is no data-path collective.
The only exchange is the small all-reduce of the episode / population statistics vector
(`ppg_stats_device`, PPG_N_STATS int64) once per reporting interval: NCCL on GPUs, any
`torch.distributed` backend otherwise (the CPU tests use gloo)."""
import torch
import torch.distributed as dist

from .config import EP_MAX_SLOTS, N_EP_STATS, N_STATS, STAT_NAMES


def shard_range(n_envs_total, rank, world_size):
    """[lo, hi) of the global env indices rank `rank` owns; slices differ by at most one env."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(int(n_envs_total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def global_env_index(local_env, rank, n_envs_total, world_size):
    return shard_range(n_envs_total, rank, world_size)[0] + local_env


def bind_to_gpu_locality(device_index):
    """Pin the calling process to the CPU cores next to GPU `device_index` (NVML's ideal affinity), so that pinned host buffers
    allocated afterwards are first-touched on the GPU's own NUMA node and the rank's device->host copies do not cross sockets
    (one process per GPU on an 8-GPU box).  Returns the number of cores bound to, or 0 if NVML is not available — then
    nothing changes."""
    import os

    try:
        import pynvml

        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(visible.split(",")[device_index]) if visible and visible.split(",")[device_index].isdigit() else device_index
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cores = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cores &= set(os.sched_getaffinity(0))
        if cores:
            os.sched_setaffinity(0, cores)
        return len(cores)
    except Exception:  # noqa: BLE001 — locality is an optimisation, never a requirement
        return 0


def allreduce_stats(stats, group=None):
    """Sum the PPG_N_STATS vector over all ranks in place (int64 tensor on the rank's device; with the
    nccl backend this is `BatchedPredPreyGrass.stats_device()` as is).  Returns a name -> int dict."""
    if stats.dtype != torch.int64 or stats.numel() != N_STATS:
        raise ValueError("stats must be the int64 PPG_N_STATS vector")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return dict(zip(STAT_NAMES, stats.tolist()))


def allreduce_episode_stats(vec, group=None):
    """All-reduce the N_EP_STATS float64 episode-returns vector (`BatchedPredPreyGrass.episode_stats_device()`) in place:
    SUM over every slot except the max and -min of the episode return (slots 6 and 7), which reduce with MAX.  Returns it."""
    if vec.dtype != torch.float64 or vec.numel() != N_EP_STATS:
        raise ValueError("vec must be the float64 PPG_N_EP_STATS vector")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        lo, hi = EP_MAX_SLOTS[0], EP_MAX_SLOTS[1] + 1
        extremes = vec[lo:hi].clone()
        vec[lo:hi] = 0.0
        dist.all_reduce(vec, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(extremes, op=dist.ReduceOp.MAX, group=group)
        vec[lo:hi] = extremes
    return vec


def max_over_ranks(value, device, group=None):
    """max of a python float over ranks (device-timed step durations are reported as the max)."""
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())
