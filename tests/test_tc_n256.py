"""Dense models with n_obs = 256 on the tensor cores: one pilot per antenna on 256 antennas, and two pilots on 128 antennas.  The
whitening launch has 512 columns (two MMAs per K-step where the triangular skip leaves more than 256), the operand ring stages K-slices
of 4 K-steps, and one 128 KB pilot tile is resident per CTA.  Pilots off the integer grid keep the complex128 kernel at this shape.
GPU tests check every estimate against the complex128 oracle (1e-5 overall, 1e-4 per estimate, no tolerated flips)."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import relerr
from oracle import qce_oracle as orc

TOL_TC = 1e-5
MODES = ('all', 1, 3, 0.9)


@pytest.fixture(scope='module')
def qce():
    import quantized_channel_estimation_b200 as q
    from quantized_channel_estimation_b200 import _lib
    _lib.require_device()
    return q


def _case(K, N, B, snr, nb, qt, mean_scale, seed, A=None):
    means, covs, w = orc.random_psd_gmm(K, N, seed=seed, mean_scale=mean_scale)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=seed + 1)
    if A is not None:
        noise = orc.crandn(B, A.shape[0], rng=np.random.default_rng(seed + 2))
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    r = orc.get_observation_nbit(h, snr, noise, A, nb, qz[0], qz[1])
    return means, covs, w, h, noise, qz, r


def _check(est, ref, what):
    assert np.isfinite(est.view(np.float64)).all(), what
    per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert relerr(est, ref) < TOL_TC and per.max() < 1e-4, (what, relerr(est, ref), np.sort(per)[-5:])


def _fix_count():
    from quantized_channel_estimation_b200 import _lib
    return int(_lib.load().qce_last_fix_count(C.c_void_p(torch.cuda.current_stream().cuda_stream)))


# ----------------------------------------------------------------------------- CPU: shape and route predicates

def test_tc_shape_predicates_n256():
    from quantized_channel_estimation_b200.engine import tc_padded_shape, tc_shape_ok
    for shape in ((256, 256), (256, 128)):
        assert tc_shape_ok(*shape, on_grid=True)
        assert not tc_shape_ok(*shape) and not tc_shape_ok(*shape, on_grid=False)
    assert not tc_shape_ok(256, 64, on_grid=True) and not tc_shape_ok(512, 256, on_grid=True)
    assert tc_shape_ok(128, 128) and tc_shape_ok(128, 128, on_grid=True)
    # on-grid models with 128 < N <= 256 pad up to 256; off-grid ones have no tensor-core shape there
    assert tc_padded_shape(200, 200, on_grid=True) == (256, 256)
    assert tc_padded_shape(256, 100, on_grid=True) == (256, 128)
    assert tc_padded_shape(200, 200) is None and tc_padded_shape(200, 200, on_grid=False) is None
    assert tc_padded_shape(256, 256) is None
    assert tc_padded_shape(300, 300, on_grid=True) is None
    # shapes up to 128 pad as before, whatever the grid
    for on_grid in (False, True):
        assert tc_padded_shape(100, 100, on_grid) == (128, 128)
        assert tc_padded_shape(20, 20, on_grid) == (32, 32)


def test_estep_route_stays_on_torch_beyond_128(monkeypatch):
    """The E-step feeds unquantised data (off the grid): at N > 128 it keeps the torch E-step."""
    from quantized_channel_estimation_b200 import em

    class _X:                      # a CUDA tensor as far as the route decision looks at it
        is_cuda = True

        def __init__(self, n):
            self.shape = (10, n)

        def contiguous(self):
            return self
    assert em._KernelEStep(_X(128)).ok and em._KernelEStep(_X(100)).ok
    assert not em._KernelEStep(_X(200)).ok and not em._KernelEStep(_X(256)).ok


@pytest.mark.parametrize('nb,qt,dense', [(2, 'uniform', True), (3, 'lloyd', False), ('inf', 'uniform', False)])
def test_mofa_route_at_256_antennas(monkeypatch, nb, qt, dense):
    """Mofa at D = 256: on-grid pilots (uniform b bit) switch to the dense tensor-core model, Lloyd-Max and unquantised pilots keep
    the Woodbury kernel."""
    import quantized_channel_estimation_b200 as q
    from quantized_channel_estimation_b200 import engine
    made = []
    monkeypatch.setattr(engine, 'MfaModel', lambda prep, flags=0: made.append('mfa') or 'mfa')
    monkeypatch.setattr(engine, 'DenseModel', lambda prep, flags=0, pad=False: made.append('dense') or 'dense')
    K, D, M, snr = 2, 256, 4, 10
    means, lam, psi, amps = orc.random_mfa(K, D, M, seed=3, mean_scale=0.0)
    m = q.Mofa(K, M, verbose=False).set_parameters(means, lam, psi, amps)
    qz = (None, None, None) if nb == 'inf' else orc.get_quantizer([snr], nb, qt)[snr]
    m._prepared(np.eye(D), snr, nb, qt, qz)
    assert made == ['dense' if dense else 'mfa']


# ----------------------------------------------------------------------------- GPU: estimates against the oracle

@pytest.mark.gpu
def test_n256_one_bit_zero_means_all_modes(qce):
    """N = 256, 1 bit, zero means, a ragged batch (700 pilots: two work units of 256 and a partial third); 'auto' takes the split
    tensor-core launches."""
    from quantized_channel_estimation_b200 import _lib
    K, N, B, snr = 6, 256, 700, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.0, seed=40)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    rt = torch.from_numpy(r).cuda()
    m.precision = 'auto'
    m.estimate_from_y(rt, snr, N, n_summands_or_proba='all')
    n0 = _lib.launch_count()
    m.estimate_from_y(rt, snr, N, n_summands_or_proba='all')
    # formatter, whitening, selection, four row blocks, fix-up: not the one complex128 launch
    assert _lib.launch_count() - n0 >= 7
    assert _fix_count() < B // 100
    m.precision = 'tc'
    for mode in MODES:
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=1)
        _check(m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode).cpu().numpy(), ref, mode)


@pytest.mark.gpu
def test_n256_two_bit_offsets_pair_and_bucketed_paths(qce, monkeypatch):
    """2-bit uniform, non-zero means (offset epilogues), a batch large enough for the pair-bucketed combination (top-n, cumulative,
    'all') and the bucketed top-1 combination (at least four work units of 256 pilots); the same pilots through the dense weighted
    launch (pair and bucket routes off) give the same estimates."""
    K, N, B, snr = 8, 256, 8300, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 2, 'uniform', 0.2, seed=41)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    for mode in MODES:
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=2, quantizer=qz)
        est = m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, n_bits=2, quantizer=qz).cpu().numpy()
        _check(est, ref, mode)
        monkeypatch.setenv('QCE_TC_PAIRS', '0')
        monkeypatch.setenv('QCE_TC_BUCKET', '0')
        est_w = m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, n_bits=2, quantizer=qz).cpu().numpy()
        monkeypatch.delenv('QCE_TC_PAIRS')
        monkeypatch.delenv('QCE_TC_BUCKET')
        _check(est_w, ref, (mode, 'weighted launch'))


@pytest.mark.gpu
@pytest.mark.parametrize('nb', [1, 2])
def test_n256_two_pilots_on_128_antennas(qce, nb):
    """A = kron([1, j], I): n_obs = 256 observations of 128 antennas (two row blocks), all four modes."""
    K, N, B, snr = 5, 128, 600, 5
    A = np.kron(np.array([[1.0], [1j]]), np.eye(N))
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, 'uniform', 0.1, seed=42, A=A)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    for mode in MODES:
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, A=A, n_summands_or_proba=mode, n_bits=nb, quantizer=qz)
        _check(m.estimate_from_y(rt, snr, N, A=A, n_summands_or_proba=mode, n_bits=nb, quantizer=qz).cpu().numpy(), ref, mode)


@pytest.mark.gpu
def test_n256_zero_padding_from_200_antennas(qce):
    """N = 200 on-grid pads to 256: the surplus estimate columns are cut off again."""
    from quantized_channel_estimation_b200.engine import DenseModel
    K, N, B, snr = 5, 200, 500, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.1, seed=43)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    model = m._prepared(np.eye(N), snr, 1, 'uniform', qz)
    assert isinstance(model, DenseModel) and (model.pad_obs, model.pad_ant) == (256, 256)
    rt = torch.from_numpy(r).cuda()
    for mode in MODES:
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=1)
        est = m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode).cpu().numpy()
        assert est.shape == (B, N)
        _check(est, ref, mode)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['all', 1])
def test_n256_pipeline_nmse_accumulators(qce, mode):
    """Fused observe -> quantise -> estimate -> NMSE at N = 256: the accumulators against a recomputation from the returned estimates;
    the row count is added once across the four row blocks."""
    from quantized_channel_estimation_b200 import engine, precompute
    K, N, B, snr = 6, 256, 1500, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.1, seed=44)
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1, 'uniform', qz))
    q = engine.Quantizer.get(1)
    ht = torch.from_numpy(h).cuda()
    est, acc = model.pipeline(q, ht, torch.from_numpy(noise).cuda(), 10 ** (-snr / 20), mode, 'tc', want_est=True)
    acc = acc.cpu().numpy()
    est = est.cpu().numpy()
    _check(est, orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=1), mode)
    assert acc[2] == B
    np.testing.assert_allclose(acc[0], np.sum(np.abs(est - h) ** 2), rtol=1e-5)
    np.testing.assert_allclose(acc[1], np.sum(np.abs(h) ** 2), rtol=1e-5)


@pytest.mark.gpu
def test_n256_log_prob_and_responsibilities(qce):
    """Weighted log-probabilities of the whitening launch against the oracle's, and the responsibilities.  Over 512 reduction
    elements the FP32 accumulation error of l_k reaches ~4e-4 nats at |l| ~ 700 (5.5e-7 relative); it is nearly the same for all
    components of a pilot, so the differences l_k - l_best -- what responsibilities and selections depend on -- stay within 2e-4."""
    from quantized_channel_estimation_b200 import engine, precompute
    K, N, B, snr = 7, 256, 600, 0
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 2, 'uniform', 0.1, seed=45)
    _, aux = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=2, quantizer=qz, return_aux=True)
    ref = aux['wlp']
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 2, 'uniform', qz))
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    for lp in (model.log_prob(torch.from_numpy(r).cuda(), 'tc').cpu().numpy(), m.weighted_log_prob(r, snr, np.eye(N), 2, 'uniform', qz)):
        d = lp - ref
        assert (np.abs(d) <= 1e-6 * np.abs(ref) + 1e-5).all(), np.abs(d).max()
        dd = d - d[np.arange(B), ref.argmax(1)][:, None]
        assert np.abs(dd).max() < 2e-4, np.abs(dd).max()
    np.testing.assert_allclose(m.predict_proba_cplx(r, snr, np.eye(N), 2, 'uniform', qz), aux['proba'], atol=2e-4)


@pytest.mark.gpu
def test_n256_host_and_level_code_entry_points(qce):
    """Host arrays in and out, and uint8 level codes in: the same estimates as the device entry point."""
    from quantized_channel_estimation_b200 import engine
    K, N, B, snr, nb = 4, 256, 900, 10, 2
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, 'uniform', 0.1, seed=46)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    q = engine.Quantizer.get(nb, qz[0], qz[1])
    _, codes = q.quantize(torch.from_numpy(h + 10 ** (-snr / 20) * noise).cuda(), want_codes=True)
    codes = codes.cpu().numpy()
    for mode in ('all', 1, 0.9):
        dev = m.estimate_from_y(torch.from_numpy(r).cuda(), snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer=qz).cpu().numpy()
        _check(dev, orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer=qz), mode)
        host = m.estimate_from_y(r, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer=qz)
        assert isinstance(host, np.ndarray)
        _check(host, dev, (mode, 'host'))
        e128 = m.estimate_from_codes(codes, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer=qz, out_dtype=np.complex128)
        assert np.array_equal(e128, host)


@pytest.mark.gpu
def test_n256_statistical_zero_flips_and_nmse(qce):
    """2000 pilots per SNR over -10 .. 30 dB at N = 256, K = 16, 1 bit: every estimate within 1e-4 of the oracle's in all four
    modes and the NMSE within 0.01 dB."""
    K, N, B = 16, 256, 2000
    means, covs, w = orc.random_psd_gmm(K, N, seed=47)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    for i, snr in enumerate(range(-10, 31, 10)):
        h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=200 + i)
        r = orc.get_observation_nbit(h, snr, noise, None, 1)
        rt = torch.from_numpy(r).cuda()
        for mode in MODES:
            ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=1)
            est = m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode).cpu().numpy()
            per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
            assert per.max() < 1e-4, (snr, mode, int((per > 1e-4).sum()), np.sort(per)[-3:])
            d_db = 10 * np.log10(orc.mse(est, h) / orc.mse(ref, h))
            assert abs(d_db) < 0.01, (snr, mode, d_db)


@pytest.mark.gpu
def test_n256_off_grid_keeps_the_complex128_kernel(qce):
    """3-bit Lloyd-Max at N = 256: 'tc' is refused with a reason, 'auto' gives the complex128 result, Mofa keeps the Woodbury kernel,
    and DenseModel(pad=True) does not pad an off-grid N = 200 model to 256."""
    from quantized_channel_estimation_b200 import _lib, engine, precompute
    K, N, B, snr, nb, qt = 4, 256, 300, 10, 3, 'lloyd'
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, qt, 0.1, seed=48)
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, nb, qt, qz), pad=True)
    rt = torch.from_numpy(r).cuda()
    with pytest.raises(_lib.QceError) as e:
        model.estimate(rt, 'all', 'tc')
    assert e.value.status == _lib.ERR_UNSUPPORTED and 'grid' in str(e.value)
    for mode in ('all', 1):
        assert torch.equal(model.estimate(rt, mode, 'auto'), model.estimate(rt, mode, 'fp64'))
    means2, covs2, w2 = orc.random_psd_gmm(K, 200, seed=49)
    m200 = engine.DenseModel(precompute.prepare(means2, covs2, w2, np.eye(200), snr, nb, qt, qz), pad=True)
    assert not m200.padded
    lam_means, lam, psi, amps = orc.random_mfa(2, N, 4, seed=50, mean_scale=0.0)
    mf = qce.Mofa(2, 4, verbose=False).set_parameters(lam_means, lam, psi, amps)
    assert isinstance(mf._prepared(np.eye(N), snr, nb, qt, qz), engine.MfaModel)
