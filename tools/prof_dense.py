#!/usr/bin/env python
"""The dominant kernel alone (config 2: GMM full, 1 bit, N=64, K=64; qce_format_pilots once, then qce_estimate_formatted in a loop),
optionally as an interleaved in-process A/B of launch-time knobs:  AB="<KEY>=<a>;<KEY>=<b>" python tools/prof_dense.py
(QCE_TC_<KEY>=<value>; without AB the default route alone)."""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import quantized_channel_estimation_b200 as qce
from quantized_channel_estimation_b200 import _lib, engine, precompute, synthetic
from bench_configs import timeit


def main():
    K, N = int(os.environ.get('K', 64)), 64
    B = 1 << int(os.environ.get('LOG2B', 20))
    snrs = [int(x) for x in os.environ.get('SNRS', '-10,10,30').split(',')]
    means, covs, w = synthetic.random_psd_gmm(K, N, seed=0)
    h, noise, _ = synthetic.sample_gmm_channels(means, covs, w, 1 << 14, seed=1)
    lib = _lib.load()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.empty((B, N), dtype=torch.complex128, device='cuda')
    ab = [x for x in os.environ.get('AB', '').split(';') if x] or ['']
    for snr in snrs:
        r = qce.get_observation_nbit(torch.from_numpy(h).cuda(), snr, n_bits=1, noise=torch.from_numpy(noise).cuda()).repeat(B >> 14, 1).contiguous()
        model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1))
        _lib.check(lib.qce_format_pilots(model.handle, stream, C.c_void_p(r.data_ptr()), B))
        run = lambda: _lib.check(lib.qce_estimate_formatted(model.handle, stream, B, C.c_void_p(out.data_ptr()), None, None))
        res = {x: [] for x in ab}
        for _ in range(int(os.environ.get('ROUNDS', 5))):
            for x in ab:
                kvs = [kv.split('=') for kv in x.split(',') if kv]
                for k, v in kvs:
                    os.environ['QCE_TC_' + k] = v
                res[x].append(timeit(run, reps=3))
                for k, _ in kvs:
                    os.environ.pop('QCE_TC_' + k)
        for x in ab:
            v = sorted(res[x])
            ms = v[len(v) // 2]
            print(json.dumps(dict(snr=snr, setting=x, ms_median=ms, est_per_s=B / ms * 1e3, tflops_algorithmic=16 * K * N * N * B / ms / 1e9)), flush=True)


if __name__ == '__main__':
    main()
