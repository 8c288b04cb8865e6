"""Sample-sharded Monte-Carlo NMSE sweep -- the loop of the reference's ``Bussgang_GMM.py:284-289`` (per SNR:
quantise the validation channels, estimate, accumulate ``sum |h_est - h|^2``), with the i.i.d. observation batch
split contiguously over the ranks of a ``torch.distributed`` job (one process per GPU, parameters replicated).

The only exchange on the path is ONE all-reduce of the ``[n_snr, 3]`` accumulators
``(sum |h_est - h|^2, sum |h|^2, count)`` after the sweep (NCCL over NVLink on GPUs; any backend works -- the
CPU tests use gloo).  Results are invariant to the number of ranks up to the summation order of those three
scalars.
"""
import numpy as np
import torch
import torch.distributed as dist


def shard_range(n_total, rank, world):
    """Contiguous split ``[lo, hi)`` of ``n_total`` observations for ``rank`` (sizes differ by at most one)."""
    base, rem = divmod(int(n_total), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def allreduce_accumulators(acc):
    """Sum the float64 accumulators (``[n_snr, 3]``, or ``[n_snr, 8]`` with the rate sums) over all ranks (no-op without an
    initialised process group)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    return acc


def nmse_from_accumulators(acc, n_antennas):
    """The scripts' metric ``sum |h_est - h|^2 / h.size`` per SNR (Bussgang_GMM.py:289; utils.py:617-618)."""
    acc = acc.detach().cpu().numpy() if isinstance(acc, torch.Tensor) else np.asarray(acc)
    return acc[:, 0] / (acc[:, 2] * n_antennas)


def nmse_sweep(step_fn, n_total, snrs, n_antennas, device='cpu'):
    """Run ``step_fn(snr_index, snr_dB, lo, hi) -> (err, power, count)`` on this rank's shard for every SNR and
    all-reduce once.  ``step_fn`` is the per-SNR hot path (``DenseModel.pipeline`` on the GPU)."""
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    lo, hi = shard_range(n_total, rank, world)
    acc = torch.zeros((len(snrs), 3), dtype=torch.float64, device=device)
    for i, snr in enumerate(snrs):
        out = step_fn(i, snr, lo, hi)
        acc[i] += torch.as_tensor(out, dtype=torch.float64, device=device)
    allreduce_accumulators(acc)
    return nmse_from_accumulators(acc, n_antennas), acc


def nmse_rate_sweep(step_fn, n_total, snrs, n_antennas, device='cpu'):
    """:func:`nmse_sweep` with the scripts' second number, the achievable-rate lower bound: ``step_fn(snr_index, snr_dB, lo, hi)``
    returns the three NMSE sums followed by the five rate sums of ``engine.RateModel.accumulate``.  One all-reduce of the
    ``[n_snr, 8]`` accumulators; returns ``(nmse [n_snr], rate [n_snr], acc [n_snr, 8])``."""
    from .utils import rate_from_accumulators
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    lo, hi = shard_range(n_total, rank, world)
    acc = torch.zeros((len(snrs), 8), dtype=torch.float64, device=device)
    for i, snr in enumerate(snrs):
        out = step_fn(i, snr, lo, hi)
        acc[i] += torch.as_tensor(out, dtype=torch.float64, device=device)
    allreduce_accumulators(acc)
    return nmse_from_accumulators(acc[:, :3], n_antennas), rate_from_accumulators(acc[:, 3:]), acc
