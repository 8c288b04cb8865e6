"""The library's per-(device, stream) scratch store: calls on different streams never share a buffer, the scratch of the host path's
private streams goes when they do, and qce_estimate_formatted only runs on pilots formatted for its model on its stream."""
import ctypes as C
import threading
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from oracle import qce_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def qce():
    import quantized_channel_estimation_b200 as q
    from quantized_channel_estimation_b200 import _lib
    _lib.require_device()
    return q


@contextmanager
def raw_stream():
    """A stream created with the CUDA runtime itself (not from torch's pool): its handle is new to the library, or the handle of a
    stream that has been destroyed."""
    from quantized_channel_estimation_b200 import _lib
    _lib.load()
    rt = C.CDLL('libcudart.so.12')          # the runtime libqce_b200.so is linked against, already loaded
    s = C.c_void_p()
    assert rt.cudaStreamCreateWithFlags(C.byref(s), 1) == 0          # cudaStreamNonBlocking
    try:
        yield s
    finally:
        rt.cudaStreamSynchronize(s)
        rt.cudaStreamDestroy(s)


def _channels(N, B, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    h = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float64)).contiguous()
    noise = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float64)).contiguous()
    return h, noise


@pytest.mark.parametrize('precision', ['fp64', 'tc'])
def test_concurrent_pipeline_on_a_shared_model(qce, precision):
    """Four host threads, each on its own stream, run the fused observe -> quantise -> estimate step on ONE model: each gets what
    it gets alone.  Every stream first runs its call once serially, so no buffer grows while the threads run."""
    from quantized_channel_estimation_b200 import engine, precompute
    K, N, B, snr, nthr = 16, 64, 1 << 15, 5, 4
    means, covs, w = orc.random_psd_gmm(K, N, seed=21)
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1))
    quant = engine.Quantizer.get(1)
    scale = 10 ** (-snr / 20)
    data = [_channels(N, B, seed=100 + i) for i in range(nthr)]
    streams = [torch.cuda.Stream() for _ in range(nthr)]
    torch.cuda.synchronize()
    serial = []
    for st, (h, noise) in zip(streams, data):
        with torch.cuda.stream(st):
            serial.append(model.pipeline(quant, h, noise, scale, 'all', precision, want_est=True))
        st.synchronize()
    results = [[] for _ in range(nthr)]
    errors = []

    def worker(i):
        try:
            h, noise = data[i]
            with torch.cuda.stream(streams[i]):
                for _ in range(4):
                    results[i].append(model.pipeline(quant, h, noise, scale, 'all', precision, want_est=True))
                streams[i].synchronize()
        except Exception as exc:                                  # noqa: BLE001 -- reported by the main thread
            errors.append((i, repr(exc)))

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(nthr)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i in range(nthr):
        ref_est, ref_acc = serial[i]
        assert ref_acc[2].item() == B
        for rep, (est, acc) in enumerate(results[i]):
            if precision == 'fp64':
                assert torch.equal(est, ref_est), (i, rep)
                np.testing.assert_allclose(acc.cpu().numpy(), ref_acc.cpu().numpy(), rtol=1e-12, err_msg=f'thread {i} rep {rep}')
            else:
                e = float((est - ref_est).norm() / ref_est.norm())
                assert e < 1e-6, (i, rep, e)
                np.testing.assert_allclose(acc.cpu().numpy(), ref_acc.cpu().numpy(), rtol=1e-6, err_msg=f'thread {i} rep {rep}')


def test_fix_count_after_host_staging_release(qce):
    """Fix lists of the host path's private streams are released with them: a new stream that has made no tensor-core call reports -1,
    and a device call on a stream of the caller's still reports its own count."""
    from quantized_channel_estimation_b200 import _lib
    lib = _lib.load()
    K, N, B, snr = 4, 32, 300, 10
    means, covs, w = orc.random_psd_gmm(K, N, seed=2, mean_scale=0.0)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=3)
    qz = orc.get_quantizer([snr], 1, 'uniform')[snr]
    r = orc.get_observation_nbit(h, snr, noise, None, 1, qz[0], qz[1])
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    bad = r.copy()
    bad[[3, 77, 200], 0] = 0.123
    est = m.estimate_from_y(bad, snr, N, n_summands_or_proba='all')          # host arrays: the private staging streams
    assert isinstance(est, np.ndarray) and est.shape == (B, N)
    # circulant tensor-core kernel, top-n: its own fix list, also on the private streams
    Kc, n1, n2, snr_c = 64, 16, 16, 8
    c, covs_c, w_c, _ = orc.circulant_gmm(Kc, n1, n2, seed=Kc)
    hc, noise_c, _ = orc.sample_gmm_channels(np.zeros((Kc, n1 * n2), complex), covs_c, w_c, 400, seed=5)
    qz_c = orc.get_quantizer([snr_c], 1, 'uniform')[snr_c]
    rc = orc.get_observation_nbit(hc, snr_c, noise_c, None, 1, qz_c[0], qz_c[1])
    mc = qce.Gmm_nbit(n_components=Kc, covariance_type='block-circulant')
    mc.set_circulant_parameters(c, w_c, (n1, n2))
    circ = mc._prepared(np.eye(n1 * n2), snr_c, 1, 'uniform', qz_c)
    assert type(circ).__name__ == 'CircModel'
    assert circ.estimate_host(rc, 3, 'tc').shape == (400, n1 * n2)
    lib.qce_host_staging_release()
    with raw_stream() as s0, raw_stream() as s1, raw_stream() as s2, raw_stream() as s3:
        for s in (s0, s1, s2, s3):
            assert lib.qce_last_fix_count(s) == -1
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        m.estimate_from_y(torch.from_numpy(bad).cuda(), snr, N, n_summands_or_proba='all')
        assert lib.qce_last_fix_count(C.c_void_p(st.cuda_stream)) == 3


def test_estimate_formatted_preconditions(qce):
    """qce_estimate_formatted refuses a stream with nothing formatted, another model's pilots and more rows than were formatted;
    on the pilots formatted for its model it gives the estimates of qce_estimate on the tensor cores."""
    from quantized_channel_estimation_b200 import _lib, engine, precompute
    lib = _lib.load()
    INVALID = -1                             # QCE_ERR_INVALID
    K, N, B, snr = 16, 64, 1000, 10
    means, covs, w = orc.random_psd_gmm(K, N, seed=7)
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1))
    other = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1))
    h, noise = _channels(N, B, seed=8)
    r = qce.get_observation_nbit(h, snr, n_bits=1, noise=noise)
    out = torch.zeros((B, N), dtype=torch.complex128, device='cuda')
    ref = torch.zeros_like(out)
    p = lambda t: C.c_void_p(t.data_ptr())
    torch.cuda.synchronize()                 # the raw streams do not wait for torch's
    with raw_stream() as fresh, raw_stream() as s:
        assert lib.qce_estimate_formatted(model.handle, fresh, B, p(out), None, None) == INVALID
        assert lib.qce_format_pilots(model.handle, s, p(r), B) == 0
        assert lib.qce_estimate_formatted(other.handle, s, B, p(out), None, None) == INVALID
        assert lib.qce_estimate_formatted(model.handle, s, B + 1, p(out), None, None) == INVALID
        assert lib.qce_estimate_formatted(model.handle, s, B, p(out), None, None) == 0
        assert lib.qce_estimate(model.handle, fresh, p(r), B, _lib.MODE_ALL, 0, 0.0, _lib.PREC_TC, p(ref), None, None, None) == 0
    torch.cuda.synchronize()
    assert bool(torch.isfinite(torch.view_as_real(ref)).all())
    assert torch.equal(out, ref)
