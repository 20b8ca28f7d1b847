"""Multi-GPU plumbing (SURVEY 8e): columns are independent, so they are sharded contiguously over
the ranks (one process per GPU) and the forward/reverse kernels need NO collective.  The only
exchange is the calibration step with parameters SHARED by all columns: one all-reduce of
[loss_sum, n_columns, unusable, dL/dalpha[L], dL/dn[L], dL/dksat[L]] (3 + 3L doubles) per optimiser
step, over NCCL (NVLink 5 / NVSwitch) on the GPU box or gloo in the CPU tests.  The reference has
no distributed code at all (agents/DifferentiableLGAR.py trains one column on one CPU)."""
from __future__ import annotations

import torch
import torch.distributed as dist


def shard_range(num_columns: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block [lo, hi) of columns owned by `rank`; sizes differ by at most one."""
    base, rem = divmod(num_columns, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def allreduce_loss_and_grads(loss_sum: torch.Tensor, count, grads: list[torch.Tensor], group=None, unusable=False):
    """Sum a local loss sum, a column count, this rank's `unusable` flag and the local gradient sums of the shared
    parameters over all ranks with ONE collective, on the loss's device (NCCL needs a CUDA vector even where the
    parameters live on the host).  Returns (mean loss, [mean gradients on the devices of `grads`], unusable): the same
    decision on every rank, true when any rank flagged its gradient or a reduced value is not finite."""
    dev = loss_sum.device
    flat = torch.cat([loss_sum.reshape(1).to(torch.float64),
                      torch.tensor([float(count), float(unusable)], dtype=torch.float64, device=dev)]
                     + [g.reshape(-1).to(dev, torch.float64) for g in grads])
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    unusable = not bool((torch.isfinite(flat).all() & (flat[2] == 0)).item())
    total = flat[1]
    out, o = [], 3
    for g in grads:
        out.append((flat[o:o + g.numel()] / total).reshape(g.shape).to(g.device, g.dtype))
        o += g.numel()
    return flat[0] / total, out, unusable


def step_if_usable(params, mean_grads, unusable: bool, optimizer, overflowed: int = 0) -> None:
    """Never step on a broken gradient: a non-finite entry or a column whose tape arena was exhausted (its gradient
    is NaN, ColumnEnsemble.last_tape_overflow) would poison the parameters and the optimiser's moments for good.
    Either every rank steps on the mean gradients, or every rank zeroes its gradients and raises."""
    if unusable:
        optimizer.zero_grad()
        raise RuntimeError(f"gradient not usable on some rank (non-finite, or columns with an exhausted tape arena; "
                           f"{overflowed} on this rank): the optimiser step was skipped")
    for p, g in zip(params, mean_grads):
        p.grad = g
    optimizer.step()


def calibration_step(shared_params, ensemble_fn, loss_fn, optimizer, group=None, ensemble=None):
    """One data-parallel calibration step with parameters shared by every column of every rank.
    `ensemble_fn(params) -> per-column outputs` runs this rank's shard (lgar_columns);
    `loss_fn(outputs) -> (loss_sum, n_columns)` on the local shard.  `ensemble`: the ColumnEnsemble of the shard, whose
    tape-overflow flags are then checked too (without it only the finiteness of the gradients is)."""
    optimizer.zero_grad(set_to_none=True)
    outputs = ensemble_fn(shared_params)
    loss_sum, count = loss_fn(outputs)
    loss_sum.backward()
    overflowed = ensemble.check_tape_overflow(raise_error=False) if ensemble is not None else 0
    grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in shared_params]
    loss, mean_grads, unusable = allreduce_loss_and_grads(loss_sum.detach(), count, grads, group, overflowed > 0)
    step_if_usable(shared_params, mean_grads, unusable, optimizer, overflowed)
    return loss
