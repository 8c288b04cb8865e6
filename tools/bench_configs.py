#!/usr/bin/env python
"""Throughput of the other BASELINE.json configurations (kernel time with CUDA events, inputs resident).
Not the contract bench (bench.py); prints one JSON line per configuration.  ``--n256`` runs only the dense n_obs = 256 shape."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import quantized_channel_estimation_b200 as qce
from quantized_channel_estimation_b200 import synthetic


def timeit(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def pilots(B, N, nb, qz, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    y = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float64)) * 0.8
    return qce.quant(y, nb, qz[0], qz[1])


def model_pilots(covs, w, B, snr, nb, qz, seed=0):
    """Quantised observations of channels DRAWN FROM THE MIXTURE (h = C_k^{1/2} g, k ~ Cat(w)) at the given SNR: the posteriors --
    and with them the work of the top-n / cumulative / sparse-'all' paths -- are those of the model's own data, not of white noise."""
    import bench
    dev = torch.device('cuda')
    gen = torch.Generator(device=dev).manual_seed(seed)
    Lc = torch.linalg.cholesky(torch.as_tensor(covs, device=dev))
    h, noise = bench.synth_channels(torch, Lc, torch.as_tensor(w, device=dev), B, gen, dev)
    return qce.get_observation_nbit(h, snr, n_bits=nb, thresholds=qz[0], cluster=qz[1], noise=noise)


def card():
    """Name and power limit of the card the numbers were measured on."""
    try:
        pl = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader,nounits', '-i', str(torch.cuda.current_device())],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = 'unknown'
    return dict(gpu=torch.cuda.get_device_name(), power_limit_w=pl)


def n256(out):
    """Dense GMM 'full', N = 256, K = 64 (BASELINE config 3's array as a dense model): 1-bit and 2-bit uniform pilots drawn from the
    model at 10 dB, all four modes, tensor-core path and complex128 kernel on the same pilots."""
    snr, K, N, B = 10, 64, 256, 1 << 18
    means, covs, w = synthetic.random_psd_gmm(K, N, seed=0)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    info = card()
    for nb in (1, 2):
        qz = qce.get_quantizer([snr], nb, 'uniform')[snr] if nb > 1 else (None, None)
        r = model_pilots(covs, w, B, snr, nb, qz)
        for mode in ('all', 1, 4, 0.9):
            row = dict(config=f'GMM full {nb}-bit uniform N=256 K=64 mode={mode}, model-drawn pilots 10 dB', B=B, **info)
            for prec, reps in (('tc', 5), ('fp64', 1)):
                m.precision = prec
                run = lambda: m.estimate_from_y(r, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer=qz)
                ms = timeit(run, reps)
                row[f'{prec}_ms'] = ms
                row[f'{prec}_est_per_s'] = B / ms * 1e3
                row[f'{prec}_tflops_algorithmic'] = 16 * K * N * N * B / ms / 1e9
            row['speedup'] = row['fp64_ms'] / row['tc_ms']
            out.append(row)
            print(json.dumps(row), flush=True)


def main():
    out = []
    if '--n256' in sys.argv:
        n256(out)
        return
    snr = 10
    # C1: GMM full, 1 bit, N=32, K=16
    means, covs, w = synthetic.random_psd_gmm(16, 32, seed=0)
    m = qce.Gmm_nbit(n_components=16).set_parameters(means, covs, w, detect_structure=False)
    r = pilots(1 << 20, 32, 1, (None, None))
    ms = timeit(lambda: m.estimate_from_y(r, snr, 32, n_summands_or_proba='all'))
    out.append(dict(config='C1 GMM full 1-bit N=32 K=16', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3, path='tc'))
    for mode_, path_ in ((1, 'tc fused launch with a running argmax'), (3, 'tc whitening -> selection -> weighted combine')):
        ms = timeit(lambda: m.estimate_from_y(r, snr, 32, n_summands_or_proba=mode_))
        out.append(dict(config=f'C1 GMM full 1-bit N=32 K=16 mode={mode_}', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3, path=path_))
    # C5 shape: GMM full, 1 bit, N=64, K=256
    means, covs, w = synthetic.random_psd_gmm(256, 64, seed=0)
    m = qce.Gmm_nbit(n_components=256).set_parameters(means, covs, w, detect_structure=False)
    r = pilots(1 << 19, 64, 1, (None, None))
    ms = timeit(lambda: m.estimate_from_y(r, snr, 64, n_summands_or_proba='all'))
    out.append(dict(config='C5 GMM full 1-bit N=64 K=256', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3, path='tc',
                    tflops_algorithmic=16 * 256 * 64 * 64 * r.shape[0] / ms / 1e9))
    # C2 other modes on the tensor-core path
    means, covs, w = synthetic.random_psd_gmm(64, 64, seed=0)
    m = qce.Gmm_nbit(n_components=64).set_parameters(means, covs, w, detect_structure=False)
    for tag, r in (('white-noise pilots', pilots(1 << 19, 64, 1, (None, None))), ('model-drawn pilots 10 dB', model_pilots(covs, w, 1 << 19, snr, 1, (None, None)))):
        for mode in ('all', 1, 4, 0.9):
            ms = timeit(lambda: m.estimate_from_y(r, snr, 64, n_summands_or_proba=mode))
            out.append(dict(config=f'C2 GMM full 1-bit N=64 K=64 mode={mode}, {tag}', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3,
                            path='tc fused' if mode == 'all' else ('tc whitening (label) -> bucket -> one-component combine' if mode == 1 else 'tc whitening -> selection -> weighted combine')))
    # C3: block-circulant 16x16, 3-bit Lloyd, N=256, K=128
    c, _, w, _ = synthetic.circulant_gmm(128, 16, 16, seed=0)
    qz = qce.get_quantizer([snr], 3, 'lloyd')[snr]
    m = qce.Gmm_nbit(n_components=128, covariance_type='block-circulant')
    m.covs_cplx = None
    m.set_circulant_parameters(c, w, (16, 16))
    r = pilots(1 << 19, 256, 3, qz)
    ms = timeit(lambda: m.estimate_from_y(r, snr, 256, n_summands_or_proba='all', n_bits=3, quantizer_type='lloyd', quantizer=qz))
    out.append(dict(config='C3 GMM block-circulant 16x16 3-bit Lloyd N=256 K=128', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3,
                    path='circ tc (fp32 fft + split-fp16 mma)', gbytes_per_s=32 * 256 * r.shape[0] / ms / 1e6))
    # C3, plain 'circulant' variant: one 256-point DFT (two-stage 16 x 16 FFT with twiddles), same kernel
    c1, _, w1, _ = synthetic.circulant_gmm(128, 1, 256, seed=0, dense=False)
    m1 = qce.Gmm_nbit(n_components=128, covariance_type='circulant')
    m1.set_circulant_parameters(c1, w1, (1, 256))
    ms = timeit(lambda: m1.estimate_from_y(r, snr, 256, n_summands_or_proba='all', n_bits=3, quantizer_type='lloyd', quantizer=qz))
    out.append(dict(config='C3 GMM circulant 3-bit Lloyd N=256 K=128', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3,
                    path='circ tc (fp32 fft + split-fp16 mma)', gbytes_per_s=32 * 256 * r.shape[0] / ms / 1e6))
    # C4: MFA N=128, K=64, latent 16, 2-bit uniform (dense path, as the reference computes it)
    means, lambdas, psis, amps = synthetic.random_mfa(64, 128, 16, seed=0)
    qz = qce.get_quantizer([snr], 2, 'uniform')[snr]
    mf = qce.Mofa(64, 16, verbose=False).set_parameters(means, lambdas, psis, amps)
    mf.precision = 'fp64'                                 # complex128: the Woodbury kernel
    r = pilots(1 << 15, 128, 2, qz)
    ms = timeit(lambda: mf.estimate_from_y(r, snr, n_summands_or_proba='all', n_bits=2, quantizer_type='uniform', quantizer=qz))
    out.append(dict(config='C4 MFA N=128 K=64 M=16 2-bit uniform', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3, path='woodbury fp64'))
    # C4 through the dense tensor-core split path (whitening launch -> selection -> two row-block launches)
    mf.use_structure = False
    mf.precision = 'tc'
    for tag, r in (('white-noise pilots', pilots(1 << 19, 128, 2, qz)), ('model-drawn pilots 10 dB', model_pilots(mf.covs, amps, 1 << 19, snr, 2, qz))):
        for mode, env in (('all', {}), ('all', {'QCE_TC_PAIRS': '0'}), (1, {}), (4, {}), (0.9, {})):
            os.environ.update(env)
            ms = timeit(lambda: mf.estimate_from_y(r, snr, n_summands_or_proba=mode, n_bits=2, quantizer_type='uniform', quantizer=qz))
            for k in env:
                os.environ.pop(k)
            out.append(dict(config=f'C4 MFA N=128 K=64 M=16 2-bit uniform mode={mode}, {tag}' + (' [dense weighted launch]' if env else ''), B=r.shape[0], ms=ms,
                            est_per_s=r.shape[0] / ms * 1e3, path='dense tc split' + ('' if env or mode == 1 else ', pair-bucketed combine'), tflops_dense_equiv=16 * 64 * 128 * 128 * r.shape[0] / ms / 1e9,
                            tflops_woodbury_equiv=(32 * 64 * 128 * 16 + 8 * 64 * 16 * 16) * r.shape[0] / ms / 1e9))
    # C4 shape with a 3-bit Lloyd-Max quantiser: pilots off the integer grid -> (hi, lo) tile pairs, three passes, one tile per CTA
    qzl = qce.get_quantizer([snr], 3, 'lloyd')[snr]
    r = pilots(1 << 18, 128, 3, qzl)
    ms = timeit(lambda: mf.estimate_from_y(r, snr, n_summands_or_proba='all', n_bits=3, quantizer_type='lloyd', quantizer=qzl))
    out.append(dict(config='C4 shape, MFA N=128 K=64 M=16 3-bit Lloyd-Max', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3,
                    path='dense tc split, off-grid pilots', tflops_dense_equiv=16 * 64 * 128 * 128 * r.shape[0] / ms / 1e9))
    # GMM full, 1 bit, N=128, K=64 (same kernels)
    means, covs, w = synthetic.random_psd_gmm(64, 128, seed=0)
    m = qce.Gmm_nbit(n_components=64).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    r = pilots(1 << 19, 128, 1, (None, None))
    ms = timeit(lambda: m.estimate_from_y(r, snr, 128, n_summands_or_proba='all'))
    out.append(dict(config='GMM full 1-bit N=128 K=64', B=r.shape[0], ms=ms, est_per_s=r.shape[0] / ms * 1e3, path='dense tc split',
                    tflops_algorithmic=16 * 64 * 128 * 128 * r.shape[0] / ms / 1e9))
    for o in out:
        print(json.dumps(o), flush=True)
    n256(out)


if __name__ == '__main__':
    main()
