#!/usr/bin/env python
"""Cost of the achievable-rate accumulators (engine.RateModel.accumulate, qce_rate.cu) next to the estimate they post-process.
2^20 pilots of channels drawn from the model at 10 dB; every input and output array is larger than the 126 MB L2, so each pass
streams from HBM.  CUDA events around REPS calls; the three variants alternate within each of ROUNDS rounds and the median round
is reported.  Prints one JSON line per configuration with the GPU name and power limit read in the same run:
    (a) the estimate alone    config 2: fused pipeline with the NMSE accumulators only;  config 3: CircModel.estimate
    (b) (a) writing its estimates, then accumulate
    (c) accumulate alone, with pilots/s and the HBM bandwidth of its B (16 N + 8 N) bytes (c128 estimates, c64 channels)."""
import json
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import quantized_channel_estimation_b200 as qce  # noqa: E402
from quantized_channel_estimation_b200 import engine, synthetic, utils  # noqa: E402
from bench_configs import card  # noqa: E402

B, SNR, ROUNDS, REPS = 1 << 20, 10, 5, 5


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / REPS


def compare(config, N, variants, extra):
    for fn in variants.values():          # warm-up of every shape in the timed window
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in variants}
    for _ in range(ROUNDS):
        for k, fn in variants.items():
            ms[k].append(timed(fn))
    med = {k: statistics.median(v) for k, v in ms.items()}
    row = dict(config=config, B=B, **card(), rounds=ROUNDS, reps=REPS, l2='inputs and outputs larger than L2',
               a_ms=med['a'], b_ms=med['b'], c_ms=med['c'], b_over_a=med['b'] / med['a'],
               c_pilots_per_s=B / med['c'] * 1e3, c_hbm_gb_per_s=B * 24 * N / med['c'] / 1e6,
               spread_ms={k: [min(v), max(v)] for k, v in ms.items()}, **extra)
    print(json.dumps(row), flush=True)


def model_channels(covs, w, seed):
    dev = torch.device('cuda')
    gen = torch.Generator(device=dev).manual_seed(seed)
    Lc = torch.linalg.cholesky(torch.as_tensor(covs, device=dev))
    return bench.synth_channels(torch, Lc, torch.as_tensor(w, device=dev), B, gen, dev)


def config2():
    K, N = 64, 64
    means, covs, w = synthetic.random_psd_gmm(K, N, seed=0)
    gmm = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, zero_mean=True, detect_structure=False)
    dm = gmm._prepared(np.eye(N, dtype=complex), SNR, 1, 'uniform', None)
    rm = engine.RateModel(*utils.rate_params(np.einsum('k,kij->ij', w, covs), SNR, 1))
    quant = engine.Quantizer.get(1)
    h, noise = model_channels(covs, w, 1)
    scale = 10 ** (-SNR / 20)
    acc = torch.zeros(3, dtype=torch.float64, device='cuda')
    racc = torch.zeros(5, dtype=torch.float64, device='cuda')
    h_est = dm.pipeline(quant, h, noise, scale, 'all', 'auto', want_est=True)[0]

    def a():
        dm.pipeline(quant, h, noise, scale, 'all', 'auto', acc=acc)

    def b():
        est, _ = dm.pipeline(quant, h, noise, scale, 'all', 'auto', want_est=True, acc=acc)
        rm.accumulate(est, h, acc=racc)

    def c():
        rm.accumulate(h_est, h, acc=racc)
    rate = utils.rate_from_accumulators(rm.accumulate(h_est, h))
    compare("config 2: GMM 'full' 1-bit N=64 K=64, fused pipeline", N, dict(a=a, b=b, c=c), dict(rate=rate))


def config3():
    K, N = 128, 256
    c, covs, w, _ = synthetic.circulant_gmm(K, 16, 16, seed=0)
    qz = qce.get_quantizer([SNR], 3, 'lloyd')[SNR]
    gmm = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant')
    gmm.set_circulant_parameters(c, w, (16, 16))
    cm = gmm._prepared(np.eye(N, dtype=complex), SNR, 3, 'lloyd', qz)
    assert isinstance(cm, engine.CircModel)
    rm = engine.RateModel(*utils.rate_params(np.einsum('k,kij->ij', w, covs), SNR, 3, 'lloyd', qz))
    h, noise = model_channels(covs, w, 2)
    r = qce.get_observation_nbit(h, SNR, n_bits=3, thresholds=qz[0], cluster=qz[1], noise=noise)
    del noise
    h_est = cm.estimate(r, 'all', 'tc')
    racc = torch.zeros(5, dtype=torch.float64, device='cuda')

    def a():
        cm.estimate(r, 'all', 'tc')

    def b():
        rm.accumulate(cm.estimate(r, 'all', 'tc'), h, acc=racc)

    def cc():
        rm.accumulate(h_est, h, acc=racc)
    rate = utils.rate_from_accumulators(rm.accumulate(h_est, h))
    compare('config 3: block-circulant 16x16 3-bit Lloyd-Max N=256 K=128, CircModel.estimate', N, dict(a=a, b=b, c=cc),
            dict(rate=rate))


if __name__ == '__main__':
    config2()
    torch.cuda.empty_cache()
    config3()
