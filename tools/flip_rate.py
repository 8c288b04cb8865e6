#!/usr/bin/env python
"""Hard-selection parity of the tensor-core paths against the complex128 kernel on the same pilots.

Per case and mode (top-1, top-n, cumulative rho):
  flips_no_fix   rows whose estimate differs by > 1e-4 when the re-evaluation of near-ties is switched off (QCE_TC_TIE_EPS=0):
                 the flip rate of the plain FP32 log-likelihood path (round-1 behaviour)
  flips          the same with the re-evaluation on (default): must be 0
  fixed          rows the tensor-core path handed to the complex128 kernel (qce_last_fix_count) and their share of the batch
  ms / ms_no_fix CUDA-event time per call with and without the re-evaluation
and the error of the tensor-core log-likelihoods (max / rms over the competitive components) that the gap threshold has to cover.
One JSON line per case; profiles/r02_flip_rate.jsonl and profiles/n256_flip_rate.jsonl are this tool's output.
FLIP_CASES=<substring> runs only the cases whose tag contains it.
"""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import quantized_channel_estimation_b200 as qce                              # noqa: E402
from quantized_channel_estimation_b200 import _lib, engine, precompute, synthetic      # noqa: E402

MODES = {'top1': 1, 'top4': 4, 'cum90': 0.9}


def timed(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1) / reps


def fix_count():
    return int(_lib.load().qce_last_fix_count(C.c_void_p(torch.cuda.current_stream().cuda_stream)))


def run_case(tag, model, r, chunk64=1 << 16):
    B = r.shape[0]
    out = dict(case=tag, pilots=B)
    # log-likelihood error of the tensor-core path
    _, lp_tc = model.estimate(r, 'all', 'tc', want_logp=True)
    lp_64 = torch.cat([model.estimate(r[i:i + chunk64], 'all', 'fp64', want_logp=True)[1] for i in range(0, B, chunk64)])
    d = lp_tc - lp_64
    top = (lp_64 - lp_64.max(1, keepdim=True).values) > -15
    out['logp_err_max'] = float(d[top].abs().max())
    out['logp_err_rms'] = float(d[top].pow(2).mean().sqrt())
    # error of the DIFFERENCE to the best component: what a selection actually depends on
    dd = d - d.gather(1, lp_64.argmax(1)[:, None])
    out['logp_gap_err_max'] = float(dd[top].abs().max())
    del d, dd, top
    for mtag, mode in MODES.items():
        ref = torch.cat([model.estimate(r[i:i + chunk64], mode, 'fp64') for i in range(0, B, chunk64)])
        rn = ref.norm(dim=1).clamp(min=1e-300)
        os.environ['QCE_TC_TIE_EPS'] = '0'
        e0, ms0 = timed(lambda: model.estimate(r, mode, 'tc'))
        del os.environ['QCE_TC_TIE_EPS']
        e1, ms1 = timed(lambda: model.estimate(r, mode, 'tc'))
        nfix = fix_count()
        p0 = (e0 - ref).norm(dim=1) / rn
        p1 = (e1 - ref).norm(dim=1) / rn
        out[mtag] = dict(flips_no_fix=int((p0 > 1e-4).sum()), flip_rate_no_fix=float((p0 > 1e-4).float().mean()),
                         flips=int((p1 > 1e-4).sum()), worst=float(p1.max()), fixed=nfix, fixed_share=nfix / B,
                         ms=ms1, ms_no_fix=ms0)
        if int((p1 > 1e-4).sum()) and os.environ.get('FLIP_DEBUG'):
            for row in torch.nonzero(p1 > 1e-4)[:3, 0].tolist():
                l64, ltc = lp_64[row], lp_tc[row]
                order = torch.argsort(l64, descending=True)[:40]
                p64 = torch.softmax(l64, 0)[order]
                ptc = torch.softmax(ltc, 0)[order]
                print('DEBUG', tag, mtag, 'row', row, 'err', float(p1[row]), file=sys.stderr)
                print('  order', order.tolist(), file=sys.stderr)
                print('  p64  ', ['%.6e' % v for v in p64.tolist()], file=sys.stderr)
                print('  cum64', ['%.9f' % v for v in torch.cumsum(p64, 0).tolist()], file=sys.stderr)
                print('  cumtc', ['%.9f' % v for v in torch.cumsum(torch.sort(torch.softmax(ltc, 0), descending=True).values, 0)[:40].tolist()], file=sys.stderr)
                print('  dl   ', ['%.2e' % v for v in (ltc - l64)[order].tolist()], file=sys.stderr)
        del ref, e0, e1
    del lp_tc, lp_64
    print(json.dumps(out), flush=True)


def main():
    B = int(os.environ.get('FLIP_B', 1 << 18))
    only = os.environ.get('FLIP_CASES', '')
    dev = torch.device('cuda')
    for tag, K, N, snr, nb, qt, b in (('C2 GMM full N=64 K=64 1-bit 10 dB', 64, 64, 10, 1, 'uniform', B),
                                      ('C2 -10 dB', 64, 64, -10, 1, 'uniform', B), ('C2 30 dB', 64, 64, 30, 1, 'uniform', B),
                                      ('C1 GMM full N=32 K=16 1-bit 10 dB (top-1: fused launch with a running argmax)', 16, 32, 10, 1, 'uniform', B),
                                      ('C1 -10 dB', 16, 32, -10, 1, 'uniform', B),
                                      ('C5 shape N=64 K=256 1-bit 10 dB', 256, 64, 10, 1, 'uniform', B // 4),
                                      ('N=128 K=64 2-bit uniform (split path)', 64, 128, 10, 2, 'uniform', B // 4),
                                      ('N=64 K=32 3-bit Lloyd (off-grid, three passes)', 32, 64, 10, 3, 'lloyd', B // 2),
                                      ('N=256 K=64 1-bit 10 dB (n_obs = 256 split path)', 64, 256, 10, 1, 'uniform', B // 4),
                                      ('N=256 K=64 2-bit uniform 10 dB (n_obs = 256 split path)', 64, 256, 10, 2, 'uniform', B // 4)):
        if only not in tag:
            continue
        means, covs, w = synthetic.random_psd_gmm(K, N, seed=0)
        h, noise, _ = synthetic.sample_gmm_channels(means, covs, w, b, seed=1)
        qz = qce.get_quantizer([snr], nb, qt)[snr]
        r = qce.get_observation_nbit(torch.from_numpy(h).to(dev), snr, n_bits=nb, thresholds=qz[0], cluster=qz[1], noise=torch.from_numpy(noise).to(dev))
        model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, nb, qt, qz))
        run_case(tag, model, r)
        del model, r
    # config 3: block-circulant 16 x 16, 3-bit Lloyd-Max, K = 128
    for tag, blocks in (('C3 block-circulant 16x16 K=128 3-bit Lloyd', (16, 16)), ('C3 plain circulant 256 K=128 3-bit Lloyd', (1, 256))):
        if only not in tag:
            continue
        K, N, snr, nb, qt = 128, 256, 8, 3, 'lloyd'
        c, _, w, _ = synthetic.circulant_gmm(K, *blocks, seed=K, dense=False)
        qz = qce.get_quantizer([snr], nb, qt)[snr]
        g = torch.Generator(device=dev).manual_seed(3)
        b = B // 2
        # pilots: quantised CN(0, C_k + s2 I) draws in the DFT domain of a random component
        lab = torch.randint(0, K, (b,), generator=g, device=dev)
        ct = torch.as_tensor(c, device=dev)[lab] + 10 ** (-snr / 10)
        z = torch.view_as_complex(torch.randn((b, N, 2), generator=g, device=dev, dtype=torch.float64)) * (0.5 * ct).sqrt()
        y = torch.fft.ifft2(z.reshape(b, *blocks), norm='ortho').reshape(b, N)
        r = qce.quant(y.contiguous(), nb, qz[0], qz[1])
        model = engine.CircModel(precompute.prepare_circulant(c, w, blocks, snr, nb, qt, qz))
        run_case(tag, model, r, chunk64=1 << 15)
        del model, r


if __name__ == '__main__':
    main()
