#!/usr/bin/env python
"""C3 (block-circulant 16x16, 3-bit Lloyd-Max, N=256, K=128) alone: timing loop for ncu / quick A-B runs."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import quantized_channel_estimation_b200 as qce
from quantized_channel_estimation_b200 import synthetic
from bench_configs import pilots, timeit


def main():
    snr, K = 10, int(os.environ.get('K', 128))
    B = 1 << int(os.environ.get('LOG2B', 19))
    c, _, w, _ = synthetic.circulant_gmm(K, 16, 16, seed=0)
    qz = qce.get_quantizer([snr], 3, 'lloyd')[snr]
    m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant')
    m.set_circulant_parameters(c, w, (16, 16))
    r = pilots(B, 256, 3, qz)
    model = m._prepared(torch.eye(256).numpy(), snr, 3, 'lloyd', qz)
    out = torch.empty_like(r)
    for prec in os.environ.get('PREC', 'tc').split(','):
        ms = timeit(lambda: model.estimate(r, 'all', prec), reps=int(os.environ.get('REPS', 5)))
        print(json.dumps(dict(config=f'C3 K={K}', precision=prec, B=B, ms=ms, est_per_s=B / ms * 1e3, gbytes_per_s=32 * 256 * B / ms / 1e6)), flush=True)
    # interleaved A/B of launch-time knobs (QCE_CIRC_PREFETCH = tiles ahead): AB="PREFETCH=0;PREFETCH=148"
    ab = [x for x in os.environ.get('AB', '').split(';') if x]
    if ab:
        res = {x: [] for x in ab}
        for _ in range(int(os.environ.get('ROUNDS', 7))):
            for x in ab:
                for kv in x.split(','):
                    k, v = kv.split('=')
                    os.environ['QCE_CIRC_' + k] = v
                res[x].append(timeit(lambda: model.estimate(r, 'all', 'tc'), reps=3))
                for kv in x.split(','):
                    os.environ.pop('QCE_CIRC_' + kv.split('=')[0])
        for x in ab:
            v = sorted(res[x])
            print(json.dumps(dict(setting=x, ms_min=v[0], ms_median=v[len(v) // 2], est_per_s_median=B / v[len(v) // 2] * 1e3)), flush=True)


if __name__ == '__main__':
    main()
