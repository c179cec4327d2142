"""Per-task episode statistics across GPUs: the only collective on this path (DESIGN.md 6).

Each rank reduces its own environments into a [14, 3] float64 buffer on the device (sag_task_stats:
sum of finished-episode returns, sum of costs, number of episodes per task id); the buffers are summed
with one all-reduce (NCCL over NVLink on GPUs, gloo in the CPU tests).  A batch with user-defined tasks has a row for
each of them after the 14 registry rows (``env.task_id_of``): the sum is right when every rank defines the same tasks
in the same order."""
import torch
import torch.distributed as dist


def reduce_task_stats(env, reset: bool = False, group=None) -> torch.Tensor:
    stats = env.task_stats(reset=reset)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def summarize(stats: torch.Tensor):
    """{task_name: (mean_return, mean_cost, episodes)} for tasks that finished at least one episode."""
    from safe_adaptation_gym_b200.benchmark import TASK_IDS
    out = {}
    s = stats.detach().cpu()
    for name, tid in TASK_IDS.items():
        n = float(s[tid, 2])
        if n > 0:
            out[name] = (float(s[tid, 0]) / n, float(s[tid, 1]) / n, int(n))
    return out
