#!/usr/bin/env python
"""BASELINE.json configs[4]: the sample-sharded scaling run -- Bussgang-GMM 'full', 1 bit, 64 antennas, K = 256 components,
N_TOTAL observations (default 1e8) split contiguously over the ranks, parameters replicated, ONE NCCL all-reduce of the
[n_snr, 3] NMSE accumulators at the end (quantized_channel_estimation_b200/montecarlo.py; reference loop: Bussgang_GMM.py:284-289).

    python tools/run_config5.py [--n-total 1e8]                                   # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 \
        tools/run_config5.py                                                      # 8 GPUs

Nothing of the 102 GB a complex128 copy of the observations would take is ever materialised: channels and noise are drawn
on the device per chunk of 2^20 observations of a GLOBAL chunk grid (seeded by chunk index, so the draws do not depend on the
number of ranks), quantised and estimated by the fused pipeline, and only the accumulators survive.  Prints one JSON line
(rank 0): estimates/s of the hot path (CUDA events around the pipeline calls, max over ranks), wall time, NMSE per SNR.

--rate adds the scripts' second number, the achievable-rate lower bound (Bussgang_GMM.py:291-309): the pipeline also writes the
chunk's estimates, engine.RateModel.accumulate adds the five rate sums of the chunk (B and C_q of the global model
sum_k w_k C_k), the all-reduce carries [n_snr, 3 + 5], and the hot-path time covers both calls."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import quantized_channel_estimation_b200 as qce
from quantized_channel_estimation_b200 import synthetic
from quantized_channel_estimation_b200 import engine, montecarlo, utils

N_ANT, N_COMP, CHUNK = 64, 256, 1 << 20
SNRS = list(range(-10, 31, 5))


def draw_channels(Lc, w, n, gen, dev):
    """h_b = C_k^{1/2} g_b, k ~ Cat(w): complex64 like the reference's SCM3GPP channels."""
    lab = torch.multinomial(w, n, replacement=True, generator=gen)
    order = torch.argsort(lab)
    counts = torch.bincount(lab, minlength=N_COMP).tolist()
    g = torch.view_as_complex(torch.randn((n, N_ANT, 2), generator=gen, device=dev, dtype=torch.float32)) * np.sqrt(0.5)
    h = torch.empty((n, N_ANT), dtype=torch.complex64, device=dev)
    pos = 0
    for k, c in enumerate(counts):
        if c:
            idx = order[pos:pos + c]
            h[idx] = g[idx] @ Lc[k].T
            pos += c
    return h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n-total', type=float, default=1e8)
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--rate', action='store_true', help='also accumulate the achievable-rate lower bound')
    args = ap.parse_args()
    n_total = int(args.n_total)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    means, covs, w = synthetic.random_psd_gmm(N_COMP, N_ANT, seed=0)
    gmm = qce.Gmm_nbit(n_components=N_COMP, covariance_type='full').set_parameters(means, covs, w, zero_mean=True, detect_structure=False)
    eye = np.eye(N_ANT, dtype=complex)
    models = [gmm._prepared(eye, s, 1, 'uniform', None) for s in SNRS]
    quant = engine.Quantizer.get(1)
    if args.rate:
        c_glob = np.einsum('k,kij->ij', w, covs)
        rate_models = [engine.RateModel(*utils.rate_params(c_glob, s, 1)) for s in SNRS]
        racc = torch.zeros((len(SNRS), 5), dtype=torch.float64, device=dev)
    Lc = torch.linalg.cholesky(torch.as_tensor(covs, device=dev)).to(torch.complex64)
    wt = torch.as_tensor(w, device=dev)

    lo, hi = montecarlo.shard_range(n_total, rank, world)
    acc = torch.zeros((len(SNRS), 3), dtype=torch.float64, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    hot_ms = 0.0
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for c in range(lo // CHUNK, (hi + CHUNK - 1) // CHUNK):
        a, b = max(lo, c * CHUNK), min(hi, (c + 1) * CHUNK)
        gen = torch.Generator(device=dev).manual_seed(args.seed * 1000003 + c)
        h = draw_channels(Lc, wt, CHUNK, gen, dev)[a - c * CHUNK:b - c * CHUNK].contiguous()      # whole global chunk, then this rank's part
        for i, snr in enumerate(SNRS):
            noise = torch.view_as_complex(torch.randn((CHUNK, N_ANT, 2), generator=gen, device=dev, dtype=torch.float64)) * np.sqrt(0.5)
            noise = noise[a - c * CHUNK:b - c * CHUNK].contiguous()
            ev[0].record()
            if args.rate:
                h_est, _ = models[i].pipeline(quant, h, noise, 10 ** (-snr / 20), 'all', 'auto', want_est=True, acc=acc[i])
                rate_models[i].accumulate(h_est, h, acc=racc[i])
            else:
                models[i].pipeline(quant, h, noise, 10 ** (-snr / 20), 'all', 'auto', acc=acc[i])
            ev[1].record()
            ev[1].synchronize()
            hot_ms += ev[0].elapsed_time(ev[1])
    if args.rate:
        both = montecarlo.allreduce_accumulators(torch.cat([acc, racc], dim=1))      # the path's only exchange
        acc, racc = both[:, :3], both[:, 3:]
    else:
        montecarlo.allreduce_accumulators(acc)              # the path's only exchange
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    t = torch.tensor([hot_ms, wall * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        hot_ms, wall_ms = t.tolist()
        nmse = montecarlo.nmse_from_accumulators(acc, N_ANT)
        assert int(acc[0, 2].item()) == n_total
        out = {
            'config': f"Bussgang-GMM 'full' 1-bit N={N_ANT} K={N_COMP}, {n_total:.3g} observations x {len(SNRS)} SNRs, sample-sharded",
            'n_gpus': world, 'estimates': n_total * len(SNRS), 'hot_path_s': hot_ms / 1e3, 'wall_s': wall_ms / 1e3,
            'estimates_per_s_hot_path': n_total * len(SNRS) / (hot_ms / 1e3),
            'estimates_per_s_wall_incl_generation': n_total * len(SNRS) / (wall_ms / 1e3),
            'tflops_algorithmic_hot_path': 16 * N_COMP * N_ANT * N_ANT * n_total * len(SNRS) / (hot_ms / 1e3) / 1e12,
            'nmse_per_snr': {str(s): float(v) for s, v in zip(SNRS, nmse)}}
        if args.rate:
            out['rate_per_snr'] = {str(s): float(v) for s, v in zip(SNRS, utils.rate_from_accumulators(racc))}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
