"""GPU parity tests (run on the B200 box with ``-m gpu``): the CUDA path, called through the C ABI,
against (a) the golden vectors produced by the unmodified reference and (b) the numpy oracle on seeded
inputs.  Tolerances: quantised pilots bit-exact; estimates 1e-4 relative (north_star) -- the complex128
kernel is held to 1e-10, the tensor-core kernel to 1e-5."""
import os

import numpy as np
import pytest
import torch

from conftest import BASELINE_TAGS, GMM_MODES, GMM_TAGS, GMM_TC_TAGS, MFA_MODES, MFA_TAGS, baseline_case, golden_quantizer_tuple, relerr
from oracle import qce_oracle as orc

pytestmark = pytest.mark.gpu

TOL_FP64 = 1e-10
TOL_TC = 1e-5          # FP16 hi/lo split operands, FP32 accumulation (north_star bound: 1e-4)


@pytest.fixture(scope='module')
def qce():
    import quantized_channel_estimation_b200 as q
    from quantized_channel_estimation_b200 import _lib
    _lib.require_device()
    return q


def _bits_equal(a, b):
    a = np.ascontiguousarray(a).view(np.uint64)
    b = np.ascontiguousarray(b).view(np.uint64)
    return np.array_equal(a, b)


def _nb(g, tag):
    nb = float(g[f'{tag}_nbits'])
    return int(nb) if np.isfinite(nb) else np.inf


# ----------------------------------------------------------------------------- quantiser: bit-exact

def test_quant_golden_bit_exact(qce, golden_quant):
    g = golden_quant
    y = g['y']
    ok = ~(np.isnan(y.real) | np.isnan(y.imag))
    out = qce.quant(y, 1)
    assert _bits_equal(out[ok], g['q1'][ok])
    assert np.isnan(out[~ok].real).all() and np.isnan(out[~ok].imag).all()      # NaN spreads like numpy's complex product
    qu = qce.get_quantizer([10], 2, 'uniform')[10]
    assert _bits_equal(qce.quant(g['yu'], 2, qu[0], qu[1]), g['q2u'])
    assert _bits_equal(qce.quant(y, 3, g['q3l_thr'], g['q3l_lab']), g['q3l'])


def test_observation_golden_bit_exact(qce, golden_quant):
    g = golden_quant
    for snr in (-5, 10):
        assert _bits_equal(qce.get_observation_nbit(g['obs_h'], snr, n_bits=1, noise=g['obs_noise']), g[f'obs1_s{snr}'])
        qs = qce.get_quantizer([snr], 2, 'uniform')[snr]
        assert _bits_equal(qce.get_observation_nbit(g['obs_h'], snr, n_bits=2, thresholds=qs[0], cluster=qs[1],
                                                    noise=g['obs_noise']), g[f'obs2u_s{snr}'])
        assert _bits_equal(qce.get_observation_nbit(g['obs_h'], snr, n_bits=np.inf, noise=g['obs_noise']), g[f'obsinf_s{snr}'])


@pytest.mark.parametrize('nb,qt', [(1, 'uniform'), (2, 'uniform'), (3, 'lloyd'), (4, 'uniform'), (8, 'uniform')])
def test_quant_large_vs_oracle(qce, nb, qt):
    rng = np.random.default_rng(nb)
    h = orc.crandn(40000, 64, rng=rng).astype(np.complex64)
    n = orc.crandn(40000, 64, rng=rng)
    snr = 5
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    ref = orc.get_observation_nbit(h, snr, n, None, nb, qz[0], qz[1])
    out = qce.get_observation_nbit(h, snr, n_bits=nb, thresholds=qz[0], cluster=qz[1], noise=n)
    assert _bits_equal(out, ref)
    # codes reproduce the labels; torch CUDA in -> torch CUDA out
    from quantized_channel_estimation_b200 import engine
    q = engine.Quantizer.get(nb, qz[0], qz[1])
    y = torch.from_numpy(orc.observe(h, snr, n)).cuda()
    r, codes = q.quantize(y, want_codes=True)
    assert r.is_cuda and _bits_equal(r.cpu().numpy(), ref)
    assert np.array_equal(codes.cpu().numpy(), orc.quant_codes(orc.observe(h, snr, n), nb, qz[0]))


def test_quant_empty_and_ragged(qce):
    assert qce.quant(np.zeros((0, 8), complex), 1).shape == (0, 8)
    y = orc.crandn(7, 3, rng=np.random.default_rng(0))
    assert _bits_equal(qce.quant(y, 1), orc.quant(y, 1))


# ----------------------------------------------------------------------------- estimates vs golden

def _gmm(qce, g, tag, precision):
    m = qce.Gmm_nbit(n_components=g[f'{tag}_means'].shape[0], covariance_type='full')
    m.set_parameters(g[f'{tag}_means'], g[f'{tag}_covs'], g[f'{tag}_w'])
    m.precision = precision
    return m


@pytest.mark.parametrize('tag', GMM_TAGS)
def test_gmm_golden_fp64(qce, golden_gmm, tag):
    g = golden_gmm
    qz = golden_quantizer_tuple(g, tag)
    m = _gmm(qce, g, tag, 'fp64')
    N = g[f'{tag}_means'].shape[1]
    for mtag, mode in GMM_MODES.items():
        if f'{tag}_est_{mtag}' not in g:
            continue
        est = m.estimate_from_y(g[f'{tag}_r'], float(g[f'{tag}_snr']), N, A=g[f'{tag}_A'], n_summands_or_proba=mode,
                                n_bits=_nb(g, tag), quantizer_type=str(g[f'{tag}_qtype']), quantizer=qz)
        assert isinstance(est, np.ndarray) and est.dtype == np.complex128
        assert relerr(est, g[f'{tag}_est_{mtag}']) < TOL_FP64, (tag, mtag)
    lp = m.weighted_log_prob(g[f'{tag}_r'], float(g[f'{tag}_snr']), g[f'{tag}_A'], _nb(g, tag), str(g[f'{tag}_qtype']), qz)
    np.testing.assert_allclose(lp, g[f'{tag}_wlp'], rtol=1e-11)
    np.testing.assert_allclose(m.predict_proba_cplx(g[f'{tag}_r'], float(g[f'{tag}_snr']), g[f'{tag}_A'], _nb(g, tag),
                                                    str(g[f'{tag}_qtype']), qz), g[f'{tag}_proba'], rtol=1e-9, atol=1e-300)
    # the reference's calling convention: predict_proba_cplx(X) / _predict_cplx(X) use the setting of the last estimate_from_y
    np.testing.assert_allclose(m.predict_proba_cplx(g[f'{tag}_r']), g[f'{tag}_proba'], rtol=1e-9, atol=1e-300)
    assert np.array_equal(m._predict_cplx(g[f'{tag}_r']), np.argmax(g[f'{tag}_proba'], axis=1))


@pytest.mark.parametrize('tag', MFA_TAGS)
def test_mfa_golden_fp64(qce, golden_mfa, tag):
    g = golden_mfa
    qz = golden_quantizer_tuple(g, tag)
    m = qce.Mofa(g[f'{tag}_means'].shape[0], g[f'{tag}_lambdas'].shape[-1], verbose=False)
    m.set_parameters(g[f'{tag}_means'], g[f'{tag}_lambdas'], g[f'{tag}_psis'], g[f'{tag}_amps'])
    m.precision = 'fp64'
    np.testing.assert_allclose(m.covs, g[f'{tag}_covs'], rtol=1e-13)
    for mtag, mode in MFA_MODES.items():
        est = m.estimate_from_y(g[f'{tag}_r'], float(g[f'{tag}_snr']), n_summands_or_proba=mode, n_bits=_nb(g, tag),
                                quantizer_type=str(g[f'{tag}_qtype']), quantizer=qz)
        assert relerr(est, g[f'{tag}_est_{mtag}']) < TOL_FP64, (tag, mtag)
    np.testing.assert_allclose(m.predict_proba(g[f'{tag}_r']), g[f'{tag}_proba'], rtol=1e-9, atol=1e-300)
    assert np.array_equal(m.predict_proba_max(g[f'{tag}_r']), g[f'{tag}_labels'])


# ----------------------------------------------------------------------------- K = 1 baselines (BLMMSE / LS)

@pytest.mark.parametrize('tag', BASELINE_TAGS)
def test_baselines_golden(qce, golden_baselines, tag):
    """estimators.BLMMSE / LS: the global variants run on the dense estimate kernels (K = 1), the genie variants as batched
    complex128 solves; both against the outputs of the reference's estimators/blmmse.py and estimators/LS.py."""
    from quantized_channel_estimation_b200 import estimators
    g = golden_baselines
    r, A, nb, qt, qz = baseline_case(g, tag)
    snr = float(g['snr'])
    for prec, tol in (('fp64', TOL_FP64), ('auto', TOL_TC)):
        bl, ls = estimators.BLMMSE(snr), estimators.LS(snr)
        bl.precision = ls.precision = prec
        assert relerr(bl.estimate_global(r, g['C_glob'], A, nb, qt, qz), g[tag + '_blmmse_global']) < tol
        assert relerr(ls.estimate_global(r, g['C_glob'], A, nb, qt, qz), g[tag + '_ls_global']) < tol
    # per-pilot solves with the arcsine-law C_r (condition numbers ~1e6): cuSOLVER vs LAPACK round differently
    assert relerr(estimators.BLMMSE(snr).estimate_genie(r, g['t'], A, nb, qt, qz), g[tag + '_blmmse_genie']) < 1e-7
    if tag + '_ls_genie' in g:
        assert relerr(estimators.LS(snr).estimate_genie(r, g['t'], A, nb, qt, qz), g[tag + '_ls_genie']) < 1e-7
    # CUDA tensors in -> CUDA tensor out; mp_eval dispatch like the scripts
    out = estimators.mp_eval(estimators.BLMMSE(snr), torch.from_numpy(r).cuda(), torch.from_numpy(g['C_glob']).cuda(), None, False, A, nb, qt, qz)
    assert out.is_cuda and relerr(out.cpu().numpy(), g[tag + '_blmmse_global']) < TOL_TC


def test_rate_lower_bound_vs_oracle(qce):
    """utils.rate_lower_bound (the scripts' post-processing, Bussgang_GMM.py:291-309) against its loop-form restatement."""
    from quantized_channel_estimation_b200 import uniform_quantizer as uq, utils
    K, N, B, snr, nb = 4, 16, 500, 10, 2
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, 'uniform', 0.0, seed=31)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    est = m.estimate_from_y(r, snr, N, n_summands_or_proba='all', n_bits=nb, quantizer=qz)
    cov = np.einsum('k,kij->ij', w, covs)
    cy = cov + 10 ** (-snr / 10) * np.eye(N)
    buss = uq.get_Bussgang_matrix(snr, nb, cy)
    cq = uq.get_Cr(cy, nb, snr, qz) - buss @ cov @ buss.conj().T
    ref = orc.rate_lower_bound(est, h, buss, cq)
    assert abs(utils.rate_lower_bound(est, h, buss, cq) - ref) < 1e-9 * max(1.0, abs(ref))
    assert abs(utils.rate_lower_bound(torch.from_numpy(est).cuda(), torch.from_numpy(h).cuda(), buss, cq) - ref) < 1e-9 * max(1.0, abs(ref))


# ----------------------------------------------------------------------------- estimates vs oracle, larger shapes

def _case(K, N, B, snr, nb, qt, mean_scale, seed):
    means, covs, w = orc.random_psd_gmm(K, N, seed=seed, mean_scale=mean_scale)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=seed + 1)
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    return means, covs, w, h, noise, qz, r


@pytest.mark.parametrize('K,N,B,snr,nb,qt,ms', [
    (16, 32, 500, 0, 1, 'uniform', 0.0),        # config 1 shape (N=32, K=16, 1-bit)
    (64, 64, 300, 10, 1, 'uniform', 0.0),       # config 2 shape (N=64, K=64, 1-bit)
    (64, 64, 200, -10, 1, 'uniform', 0.1),
    (8, 64, 200, 30, 1, 'uniform', 0.0),
    (12, 64, 200, 10, 2, 'uniform', 0.1),
    (12, 48, 200, 10, 3, 'lloyd', 0.0),
    (5, 20, 77, 5, 4, 'uniform', 0.2),          # ragged: N not a multiple of anything nice, B not a tile multiple
])
@pytest.mark.parametrize('precision', ['fp64', 'tc'])
def test_gmm_vs_oracle(qce, K, N, B, snr, nb, qt, ms, precision):
    from quantized_channel_estimation_b200 import _lib
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, qt, ms, seed=K + N)
    m = qce.Gmm_nbit(n_components=K, covariance_type='full').set_parameters(means, covs, w)
    m.precision = precision
    tol = TOL_FP64 if precision == 'fp64' else TOL_TC
    for mode in ('all', 1, 3, 0.95):
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt,
                                      quantizer=qz)
        try:
            est = m.estimate_from_y(torch.from_numpy(r).cuda(), snr, N, n_summands_or_proba=mode, n_bits=nb,
                                    quantizer_type=qt, quantizer=qz)
        except _lib.QceError as e:
            if precision == 'tc' and e.status == _lib.ERR_UNSUPPORTED:
                pytest.skip(f'tensor-core kernel does not cover this shape/mode: {e}')
            raise
        assert est.is_cuda and est.dtype == torch.complex128
        est = est.cpu().numpy()
        assert relerr(est, ref) < tol, (mode, relerr(est, ref))
        # north_star: every estimate within 1e-4 -- no exemption for the hard selections (near-ties are re-evaluated in complex128)
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert per.max() < 1e-4, (mode, np.sort(per)[-5:])
    # NMSE within 0.01 dB of the oracle's (north_star)
    ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
    est = m.estimate_from_y(r, snr, N, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
    d_db = 10 * np.log10(orc.mse(est, h) / orc.mse(ref, h))
    assert abs(d_db) < 0.01


@pytest.mark.parametrize('tag', GMM_TC_TAGS)
def test_tc_golden_reference(qce, golden_gmm_tc, tag):
    """The tensor-core path directly against outputs of the UNMODIFIED reference at shapes it is instantiated for
    (tests/golden/make_golden_tc.py): every estimate within 1e-4 (north_star), all four combination modes, log-probabilities."""
    g = golden_gmm_tc
    qz = golden_quantizer_tuple(g, tag)
    m = _gmm(qce, g, tag, 'tc')
    N = g[f'{tag}_means'].shape[1]
    for mtag, mode in GMM_MODES.items():
        est = m.estimate_from_y(torch.from_numpy(g[f'{tag}_r']).cuda(), float(g[f'{tag}_snr']), N, A=g[f'{tag}_A'], n_summands_or_proba=mode,
                                n_bits=_nb(g, tag), quantizer_type=str(g[f'{tag}_qtype']), quantizer=qz).cpu().numpy()
        ref = g[f'{tag}_est_{mtag}']
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert relerr(est, ref) < TOL_TC and per.max() < 1e-4, (tag, mtag, relerr(est, ref), per.max())
    model = m._prepared(g[f'{tag}_A'], float(g[f'{tag}_snr']), _nb(g, tag), str(g[f'{tag}_qtype']), qz)
    _, lp = model.estimate(torch.from_numpy(g[f'{tag}_r']).cuda(), 'all', 'tc', want_logp=True)
    assert np.abs(lp.cpu().numpy() - g[f'{tag}_wlp']).max() < 2e-4


def test_tc_statistical_size_zero_flips_and_nmse(qce):
    """SURVEY section 4(iv): 10 000 pilots per SNR over the -10 .. 30 dB sweep at the config-2 shape (N = 64, K = 64, 1 bit).  Every
    estimate of the tensor-core path within 1e-4 of the oracle's in all four combination modes -- zero flipped selections -- and the
    NMSE (Bussgang_GMM.py:289) within 0.01 dB."""
    K, N, B = 64, 64, 10000
    means, covs, w = orc.random_psd_gmm(K, N, seed=0)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    for i, snr in enumerate(range(-10, 31, 5)):
        h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=100 + i)
        r = orc.get_observation_nbit(h, snr, noise, None, 1)
        rt = torch.from_numpy(r).cuda()
        for mode in ('all', 1, 4, 0.9):
            ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=1)
            est = m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode).cpu().numpy()
            per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
            assert per.max() < 1e-4, (snr, mode, int((per > 1e-4).sum()), np.sort(per)[-3:])
            d_db = 10 * np.log10(orc.mse(est, h) / orc.mse(ref, h))
            assert abs(d_db) < 0.01, (snr, mode, d_db)


def test_pipeline_matches_stepwise(qce):
    """Fused observe->quantise->estimate->NMSE equals the three reference-API calls and the oracle."""
    from quantized_channel_estimation_b200 import engine
    K, N, B, snr = 16, 32, 3000, 5
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.0, seed=3)
    m = qce.Gmm_nbit(n_components=K, covariance_type='full').set_parameters(means, covs, w)
    model = m._prepared(np.eye(N, dtype=complex), snr, 1, 'uniform', None)
    q = engine.Quantizer.get(1)
    h64 = h.astype(np.complex64)
    r64 = orc.get_observation_nbit(h64, snr, noise, None, 1)
    ref = orc.gmm_estimate_from_y(means, covs, w, r64, snr, n_summands_or_proba='all', n_bits=1)
    for prec in ('fp64', 'auto'):
        est, acc = model.pipeline(q, torch.from_numpy(h64).cuda(), torch.from_numpy(noise).cuda(), 10 ** (-snr / 20), 'all',
                                  prec, want_est=True)
        acc = acc.cpu().numpy()
        assert relerr(est.cpu().numpy(), ref) < (TOL_FP64 if prec == 'fp64' else TOL_TC)
        assert acc[2] == B
        np.testing.assert_allclose(acc[0] / (B * N), orc.mse(ref, h64.astype(complex)), rtol=1e-6)
        np.testing.assert_allclose(acc[1], np.sum(np.abs(h64.astype(complex)) ** 2), rtol=1e-6 if prec == 'auto' else 1e-12)


def test_linearity_and_batch_invariance_full_size(qce):
    """Size-independent properties at the BASELINE shape (N=64, K=64, 1-bit, 2^17 pilots): estimates do not
    depend on how the batch is tiled or ordered, and with a single component the estimator is linear in r."""
    K, N, B, snr = 64, 64, 1 << 17, 10
    means, covs, w = orc.random_psd_gmm(K, N, seed=0)
    m = qce.Gmm_nbit(n_components=K, covariance_type='full').set_parameters(means, covs, w)
    g = torch.Generator(device='cuda').manual_seed(0)
    bits = torch.randint(0, 2, (B, N, 2), generator=g, device='cuda', dtype=torch.int8)
    r = torch.view_as_complex(((bits.double() * 2 - 1) / np.sqrt(2)).contiguous())
    full = m.estimate_from_y(r, snr, N, n_summands_or_proba='all')
    perm = torch.randperm(B, generator=g, device='cuda')
    part = m.estimate_from_y(r[perm][:50001].contiguous(), snr, N, n_summands_or_proba='all')
    assert torch.equal(part, full[perm][:50001])
    # spot-check 64 rows of the full batch against the oracle
    idx = np.arange(0, B, B // 64)
    ref = orc.gmm_estimate_from_y(means, covs, w, r[idx].cpu().numpy(), snr, n_summands_or_proba='all', n_bits=1)
    assert relerr(full[idx].cpu().numpy(), ref) < TOL_TC
    m1 = qce.Gmm_nbit(n_components=1, covariance_type='full').set_parameters(means[:1], covs[:1], [1.0])
    a = m1.estimate_from_y(r[:4096].contiguous(), snr, N, n_summands_or_proba='all')
    b = m1.estimate_from_y((-r[:4096]).contiguous(), snr, N, n_summands_or_proba='all')
    assert float((a + b).abs().max()) < 1e-5 * float(a.abs().max())


def _grid_pilots(B, N, levels, scale, seed):
    """Random pilots on the grid {+-1, +-3, ...} * scale (what a uniform quantiser emits), on the GPU."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    idx = torch.randint(0, levels, (B, N, 2), generator=g, device='cuda', dtype=torch.int8)
    return torch.view_as_complex(((idx.double() * 2 - (levels - 1)) * scale).contiguous()), g


def test_full_size_config4_mfa_split_path(qce):
    """BASELINE config 4 at full size (MFA, N=128, K=64, latent 16, 2-bit uniform; 2^16 pilots): tiling / order invariance of the
    split tensor-core path, oracle spot check, agreement with the complex128 Woodbury kernel."""
    K, N, M, B, snr = 64, 128, 16, 1 << 16, 10
    means, lambdas, psis, amps = orc.random_mfa(K, N, M, seed=0)
    covs = orc.mofa_covs(lambdas, psis)
    qz = orc.get_quantizer([snr], 2, 'uniform')[snr]
    mf = qce.Mofa(K, M, verbose=False).set_parameters(means, lambdas, psis, amps)
    r, g = _grid_pilots(B, N, 4, qz[1][-1] / 3, seed=4)
    full = mf.estimate_from_y(r, snr, n_summands_or_proba='all', n_bits=2, quantizer=qz)
    perm = torch.randperm(B, generator=g, device='cuda')
    part = mf.estimate_from_y(r[perm][:20001].contiguous(), snr, n_summands_or_proba='all', n_bits=2, quantizer=qz)
    assert torch.equal(part, full[perm][:20001])
    idx = np.arange(0, B, B // 48)
    ref = orc.mofa_estimate_from_y(means, covs, amps, r[idx].cpu().numpy(), snr, n_summands_or_proba='all', n_bits=2, quantizer=qz)
    assert relerr(full[idx].cpu().numpy(), ref) < TOL_TC
    mf.precision = 'fp64'                                       # Woodbury kernel
    w64 = mf.estimate_from_y(r[:4096].contiguous(), snr, n_summands_or_proba='all', n_bits=2, quantizer=qz)
    assert relerr(full[:4096].cpu().numpy(), w64.cpu().numpy()) < TOL_TC


def test_full_size_config3_block_circulant(qce):
    """BASELINE config 3 at full size (block-circulant 16x16, N=256, K=128, 3-bit Lloyd-Max; 2^16 pilots): tiling / order
    invariance of the FP32-FFT + tensor-core kernel, agreement with the complex128 kernel, dense-oracle spot check."""
    K, N, B, snr = 128, 256, 1 << 16, 10
    c, covs, w, F = orc.circulant_gmm(K, 16, 16, seed=0)
    qz = orc.get_quantizer([snr], 3, 'lloyd')[snr]
    m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant')
    m.set_circulant_parameters(c, w, (16, 16))
    g = torch.Generator(device='cuda').manual_seed(3)
    y = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float64)) * 0.8
    r = qce.quant(y, 3, qz[0], qz[1])
    full = m.estimate_from_y(r, snr, N, n_summands_or_proba='all', n_bits=3, quantizer_type='lloyd', quantizer=qz)
    perm = torch.randperm(B, generator=g, device='cuda')
    part = m.estimate_from_y(r[perm][:10007].contiguous(), snr, N, n_summands_or_proba='all', n_bits=3, quantizer_type='lloyd', quantizer=qz)
    assert torch.equal(part, full[perm][:10007])
    m.precision = 'fp64'
    f64 = m.estimate_from_y(r[:8192].contiguous(), snr, N, n_summands_or_proba='all', n_bits=3, quantizer_type='lloyd', quantizer=qz)
    assert relerr(full[:8192].cpu().numpy(), f64.cpu().numpy()) < TOL_TC
    idx = np.arange(0, B, B // 16)
    ref = orc.gmm_estimate_from_y(np.zeros((K, N)), covs, w, r[idx].cpu().numpy(), snr, n_summands_or_proba='all', n_bits=3,
                                  quantizer_type='lloyd', quantizer=qz)
    assert relerr(full[idx].cpu().numpy(), ref) < TOL_TC


def test_full_size_config5_shape(qce):
    """BASELINE config 5 shape (N=64, K=256, 1 bit; 2^17 pilots): NMSE accumulators of the fused pipeline do not depend on how the
    observations are split (the sample-sharded run adds them across ranks), oracle spot check."""
    from quantized_channel_estimation_b200 import engine, precompute
    K, N, B, snr = 256, 64, 1 << 17, 5
    means, covs, w = orc.random_psd_gmm(K, N, seed=0)
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1))
    quant = engine.Quantizer.get(1)
    g = torch.Generator(device='cuda').manual_seed(5)
    h = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float32)).contiguous()
    noise = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float64)).contiguous()
    est, acc = model.pipeline(quant, h, noise, 10 ** (-snr / 20), 'all', 'auto', want_est=True)
    parts = torch.zeros(3, dtype=torch.float64, device='cuda')
    for lo, hi in ((0, 40000), (40000, 40001), (40001, B)):
        model.pipeline(quant, h[lo:hi].contiguous(), noise[lo:hi].contiguous(), 10 ** (-snr / 20), 'all', 'auto', acc=parts)
    assert parts[2].item() == acc[2].item() == B
    np.testing.assert_allclose(parts.cpu().numpy(), acc.cpu().numpy(), rtol=1e-9)
    idx = np.arange(0, B, B // 32)
    r = orc.get_observation_nbit(h[idx].cpu().numpy(), snr, noise[idx].cpu().numpy(), None, 1)
    ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=1)
    assert relerr(est[idx].cpu().numpy(), ref) < TOL_TC


def test_host_and_device_entry_points_agree(qce):
    K, N, B, snr = 8, 32, 300000, 0         # > two staging chunks -> exercises the double-buffered host path
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.0, seed=9)
    m = qce.Gmm_nbit(n_components=K, covariance_type='full').set_parameters(means, covs, w)
    a = m.estimate_from_y(r, snr, N, n_summands_or_proba='all')
    b = m.estimate_from_y(torch.from_numpy(r).cuda(), snr, N, n_summands_or_proba='all').cpu().numpy()
    assert np.array_equal(a, b)
    assert m.estimate_from_y(np.zeros((0, N), complex), snr, N, n_summands_or_proba='all').shape == (0, N)


# ----------------------------------------------------------------------------- circulant / block-circulant kernel

@pytest.mark.parametrize('n1,n2,K,nb,qt,tol', [
    (1, 64, 8, 1, 'uniform', 1e-7),          # plain circulant, 1 bit (arcsine-law diagonal: the reference's C_r diag is 1 - O(1e-8))
    (8, 8, 16, 1, 'uniform', 1e-7),
    (16, 16, 12, 3, 'lloyd', 1e-10),         # config 3 shape: 256 antennas, 16x16 blocks, 3-bit Lloyd-Max
    (4, 8, 6, 2, 'uniform', 1e-10),
    (3, 5, 4, 2, 'uniform', 1e-10),          # odd sizes
])
def test_circulant_kernel_vs_dense_oracle(qce, n1, n2, K, nb, qt, tol):
    """The DFT-domain kernel (new algorithm) against the oracle's DENSE path, which is what the reference computes
    for circulant / block-circulant models after it densifies them (gmm:104-136)."""
    N, B, snr = n1 * n2, 150, 8
    c, covs, w, F = orc.circulant_gmm(K, n1, n2, seed=n1 + n2)
    h, noise, _ = orc.sample_gmm_channels(np.zeros((K, N), complex), covs, w, B, seed=5)
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant')
    m.set_parameters(np.zeros((K, N)), covs, w, zero_mean=True)           # structure is detected from the dense covariances
    assert m.blocks is not None and m.blocks[0] * m.blocks[1] == N
    np.testing.assert_allclose(m.fft_covs, c, rtol=1e-8, atol=1e-12)
    from quantized_channel_estimation_b200.engine import CircModel
    assert isinstance(m._prepared(np.eye(N), snr, nb, qt, qz), CircModel)
    for mode in ('all', 1, 3, 0.9):
        ref = orc.gmm_estimate_from_y(np.zeros((K, N)), covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt,
                                      quantizer=qz)
        est = m.estimate_from_y(r, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz)
        assert relerr(est, ref) < tol, (mode, relerr(est, ref))
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert per.max() < 100 * tol, (mode, np.sort(per)[-5:])      # no flipped selection
    # and the structured path agrees with our own dense kernels
    m.use_structure = False
    m._cache.clear()
    dense = m.estimate_from_y(r, snr, N, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
    m.use_structure = True
    m._cache.clear()
    assert relerr(m.estimate_from_y(r, snr, N, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz), dense) < max(tol, 1e-5)


@pytest.mark.parametrize('K,nb,qt,B,n1,n2', [
    (128, 3, 'lloyd', 150, 16, 16),          # config 3: 256 antennas, 16x16 blocks, 3-bit Lloyd-Max, K = 128 (ragged batch)
    (64, 1, 'uniform', 97, 16, 16),
    (64, np.inf, 'uniform', 33, 16, 16),     # unquantised pilots: no grid assumption in this kernel
    (128, 3, 'lloyd', 140, 1, 256),          # config 3, plain circulant: one 256-point DFT as a two-stage 16 x 16 FFT with twiddles
    (64, 2, 'uniform', 70, 1, 256),
])
def test_circulant_tc_kernel_vs_dense_oracle(qce, K, nb, qt, B, n1, n2):
    """FP32-FFT + split-FP16 tensor-core version of the DFT-domain kernel against the oracle's dense path."""
    from quantized_channel_estimation_b200.engine import CircModel
    N, snr = 256, 8
    c, covs, w, F = orc.circulant_gmm(K, n1, n2, seed=K)
    h, noise, _ = orc.sample_gmm_channels(np.zeros((K, N), complex), covs, w, B, seed=5)
    qz = orc.get_quantizer([snr], nb, qt)[snr] if np.isfinite(nb) else (None, None, None)
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant')
    m.set_circulant_parameters(c, w, (n1, n2))
    model = m._prepared(np.eye(N), snr, nb, qt, qz)
    assert isinstance(model, CircModel)
    rt = torch.from_numpy(r).cuda()
    for mode in ('all', 1, 3, 0.9):
        ref = orc.gmm_estimate_from_y(np.zeros((K, N)), covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt,
                                      quantizer=qz)
        est = model.estimate(rt, mode, 'tc').cpu().numpy()
        assert est.shape == (B, N) and np.isfinite(est.view(np.float64)).all()
        assert relerr(est, ref) < TOL_TC, (mode, relerr(est, ref))
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert per.max() < 1e-4, (mode, np.sort(per)[-5:])
    # log-probabilities, NMSE accumulators, agreement with the complex128 kernel; 'auto' picks the fast kernel
    est64, lp64 = model.estimate(rt, 'all', 'fp64', want_logp=True)
    est_tc, lp_tc, acc = model.estimate(rt, 'all', 'auto', want_logp=True, h_true=torch.from_numpy(h).cuda())
    assert relerr(est_tc.cpu().numpy(), est64.cpu().numpy()) < TOL_TC
    assert float((lp_tc - lp64).abs().max()) < 2e-3 * max(1.0, float(lp64.abs().max()) / 300)
    acc = acc.cpu().numpy()
    assert acc[2] == B
    np.testing.assert_allclose(acc[0], np.sum(np.abs(est_tc.cpu().numpy() - h) ** 2), rtol=1e-4)
    np.testing.assert_allclose(acc[1], np.sum(np.abs(h) ** 2), rtol=1e-4)


@pytest.mark.parametrize('scale,snr,nb,qt', [(1e3, 10, 3, 'lloyd'), (1e-3, 0, 2, 'uniform'), (1.0, 35, 1, 'uniform'), (1.0, -20, 3, 'lloyd')])
def test_circulant_tc_kernel_scales_and_extreme_snr(qce, scale, snr, nb, qt):
    """Per-pilot scaling of |rt|^2, global scaling of the parameter fragments and the compensated log-likelihood accumulation under
    channel powers far from one and extreme SNRs; against the complex128 kernel on the same pilots."""
    K, N, B = 64, 256, 200
    c, _, w, _ = orc.circulant_gmm(K, 16, 16, seed=17)
    c = c * scale
    m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant')
    m.set_circulant_parameters(c, w, (16, 16))
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    g = torch.Generator(device='cuda').manual_seed(18)
    y = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float64)) * float(np.sqrt(scale + 10 ** (-snr / 10)))
    r = qce.quant(y, nb, qz[0], qz[1])
    model = m._prepared(np.eye(N), snr, nb, qt, qz)
    e_tc, lp_tc = model.estimate(r, 'all', 'tc', want_logp=True)
    e_64, lp_64 = model.estimate(r, 'all', 'fp64', want_logp=True)
    assert torch.isfinite(torch.view_as_real(e_tc)).all()
    per = (e_tc - e_64).norm(dim=1) / e_64.norm(dim=1).clamp(min=1e-300)
    assert float((e_tc - e_64).norm() / e_64.norm()) < TOL_TC and float(per.max()) < 1e-4, (float(per.max()),)
    assert float((lp_tc - lp_64).abs().max()) < 5e-3 * max(1.0, float(lp_64.abs().max()) / 300)


# ----------------------------------------------------------------------------- MFA Woodbury kernel

@pytest.mark.parametrize('K,N,M,nb,qt,ms', [
    (6, 48, 8, 2, 'uniform', 0.3),
    (8, 64, 16, 3, 'lloyd', 0.0),
    (4, 128, 16, 2, 'uniform', 0.1),          # config 4 shape: 128 antennas, latent rank 16, 2-bit uniform
    (3, 20, 3, np.inf, 'uniform', 0.2),
])
def test_mfa_woodbury_vs_dense_oracle(qce, K, N, M, nb, qt, ms):
    """Low-rank + diagonal kernel against the oracle's dense MFA path (what the reference computes, mofa:162-216)."""
    from quantized_channel_estimation_b200.engine import MfaModel, DenseModel
    B, snr = 120, 9
    means, lam, psi, amps = orc.random_mfa(K, N, M, seed=K + N, mean_scale=ms)
    covs = orc.mofa_covs(lam, psi)
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    h, noise, _ = orc.sample_gmm_channels(means, covs, amps, B, seed=4)
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    m = qce.Mofa(K, M, verbose=False).set_parameters(means, lam, psi, amps)
    m.precision = 'fp64'              # complex128 path: the Woodbury kernel ('auto' prefers the tensor-core kernels on grid data)
    assert isinstance(m._prepared(np.eye(N), snr, nb, qt, qz), MfaModel)
    for mode in ('all', 1, 2, 0.9):
        ref, aux = orc.mofa_estimate_from_y(means, covs, amps, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt,
                                            quantizer=qz, return_aux=True)
        est = m.estimate_from_y(r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz)
        assert relerr(est, ref) < 1e-10, (mode, relerr(est, ref))
    np.testing.assert_allclose(m.predict_proba(r), aux['proba'], rtol=1e-8, atol=1e-300)
    # 1 bit destroys the low-rank structure: dense path
    assert isinstance(m._prepared(np.eye(N), snr, 1, 'uniform', (None, None, None)), DenseModel)
    # 'auto': pilots on a uniform grid and a tensor-core shape go to the dense tcgen05 kernels, everything else stays Woodbury
    m.precision = 'auto'
    from quantized_channel_estimation_b200.engine import tc_padded_shape
    # every shape that fits a tensor-core shape after zero padding (off-grid pilots -- Lloyd-Max labels, unquantised data -- as FP16
    # (hi, lo) tile pairs)
    assert isinstance(m._prepared(np.eye(N), snr, nb, qt, qz), DenseModel if tc_padded_shape(N, N) is not None else MfaModel)
    if tc_padded_shape(N, N) is not None:
        ref = orc.mofa_estimate_from_y(means, covs, amps, r, snr, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
        est = m.estimate_from_y(r, snr, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
        assert relerr(est, ref) < TOL_TC


# ----------------------------------------------------------------------------- fit -> estimate end to end

def test_fit_then_estimate_matches_true_model_nmse(qce):
    """EM on the GPU, then the hot path: the fitted model's NMSE is within 0.1 dB of the data-generating model's."""
    import warnings
    K, N, snr = 4, 16, 10
    means, covs, w = orc.random_psd_gmm(K, N, seed=5)
    htrain, _, _ = orc.sample_gmm_channels(means, covs, w, 20000, seed=6)
    hval, noise, _ = orc.sample_gmm_channels(means, covs, w, 4000, seed=7)
    r = orc.get_observation_nbit(hval, snr, noise, None, 1)
    g = qce.Gmm_nbit(n_components=K, covariance_type='full', random_state=0, max_iter=200, tol=1e-5)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        g.fit(htrain, zero_mean=True)
    est_fit = g.estimate_from_y(r, snr, N, n_summands_or_proba='all')
    true = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w)
    est_true = true.estimate_from_y(r, snr, N, n_summands_or_proba='all')
    d_db = 10 * np.log10(orc.mse(est_fit, hval) / orc.mse(est_true, hval))
    assert abs(d_db) < 0.1, d_db


# ----------------------------------------------------------------------------- tensor-core path: edges and variants

@pytest.mark.parametrize('B', [1, 127, 129, 511, 513, 1025])
def test_tc_ragged_batches(qce, B):
    """Unit / tile boundaries of the persistent SM-pair kernel (512 pilots per work unit, 128 per tile)."""
    K, N, snr = 3, 32, 5
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.1, seed=B)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    for mode in ('all', 2):
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=1)
        est = m.estimate_from_y(torch.from_numpy(r).cuda(), snr, N, n_summands_or_proba=mode).cpu().numpy()
        assert est.shape == (B, N) and np.isfinite(est.view(np.float64)).all()
        assert relerr(est, ref) < TOL_TC
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert per.max() < 1e-4, (mode, np.sort(per)[-5:])


def _check_modes(est_fn, ref_fn, B):
    for mode in ('all', 1, 3, 0.95):
        est, ref = est_fn(mode), ref_fn(mode)
        assert np.isfinite(est.view(np.float64)).all()
        assert relerr(est, ref) < TOL_TC, (mode, relerr(est, ref))
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert per.max() < 1e-4, (mode, np.sort(per)[-5:])


@pytest.mark.parametrize('K,N,B,snr,nb,ms', [
    (6, 128, 700, 10, 1, 0.0),      # two row blocks of 128 estimate columns, zero means
    (5, 128, 300, 5, 2, 0.1),       # 2-bit uniform, non-zero means (offset epilogues)
    (4, 96, 515, 0, 1, 0.1),        # 96 antennas: 192-column whitening launch, two row blocks of 96
    (70, 128, 130, 20, 3, 0.0),     # more components than the config-4 shape, 3-bit uniform grid (odd integers up to 7)
])
def test_tc_split_path_large_antenna_counts(qce, K, N, B, snr, nb, ms):
    """64 < N <= 128: whitening-only launch -> selection -> LMMSE row-block launches (all four modes)."""
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, 'uniform', ms, seed=K + N)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    _check_modes(lambda mode: m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer=qz).cpu().numpy(),
                 lambda mode: orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer=qz), B)
    # NMSE accumulators of the fused pipeline: each row block adds its columns, the row count is added once
    from quantized_channel_estimation_b200 import engine, precompute
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, nb, 'uniform', qz))
    est, acc = model.estimate(rt, 'all', 'tc', h_true=torch.from_numpy(h).cuda())
    acc = acc.cpu().numpy()
    assert acc[2] == B
    np.testing.assert_allclose(acc[0], np.sum(np.abs(est.cpu().numpy() - h) ** 2), rtol=1e-5)
    np.testing.assert_allclose(acc[1], np.sum(np.abs(h) ** 2), rtol=1e-5)


@pytest.mark.parametrize('N,nb,qt', [(64, 1, 'uniform'), (32, 1, 'uniform'), (16, 2, 'uniform'), (32, 3, 'lloyd'), (64, 2, 'lloyd')])
def test_tc_two_pilots(qce, N, nb, qt):
    """A = kron(x, I): n_obs = 2 N observations of N antennas.  N = 64: split path (one row block of 128 columns); N = 32 / 16: the
    fused kernel with Z twice as wide as H; Lloyd-Max rows: off-grid pilots as (hi, lo) tile pairs on both."""
    K, B, snr = 5, 400, 5
    means, covs, w = orc.random_psd_gmm(K, N, seed=21 + N, mean_scale=0.1)
    h, _, _ = orc.sample_gmm_channels(means, covs, w, B, seed=22)
    A = np.kron(np.array([[1.0], [1j]]), np.eye(N))
    noise = orc.crandn(B, 2 * N, rng=np.random.default_rng(23))
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    r = orc.get_observation_nbit(h, snr, noise, A, nb, qz[0], qz[1])
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    _check_modes(lambda mode: m.estimate_from_y(rt, snr, N, A=A, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz).cpu().numpy(),
                 lambda mode: orc.gmm_estimate_from_y(means, covs, w, r, snr, A=A, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt,
                                                      quantizer=qz), B)


def test_tc_split_path_mfa_config4_shape(qce):
    """MFA, N = 128, latent 16, 2-bit uniform (BASELINE config 4 with fewer components) through the dense tensor-core path."""
    K, N, M, B, snr = 8, 128, 16, 300, 10
    means, lambdas, psis, amps = orc.random_mfa(K, N, M, seed=5, mean_scale=0.1)
    covs = orc.mofa_covs(lambdas, psis)
    qz = orc.get_quantizer([snr], 2, 'uniform')[snr]
    h, noise, _ = orc.sample_gmm_channels(means, covs, amps, B, seed=6)
    r = orc.get_observation_nbit(h, snr, noise, None, 2, qz[0], qz[1])
    mf = qce.Mofa(K, M, verbose=False).set_parameters(means, lambdas, psis, amps)
    mf.use_structure = False
    mf.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    _check_modes(lambda mode: mf.estimate_from_y(rt, snr, n_summands_or_proba=mode, n_bits=2, quantizer=qz).cpu().numpy(),
                 lambda mode: orc.mofa_estimate_from_y(means, covs, amps, r, snr, n_summands_or_proba=mode, n_bits=2, quantizer=qz), B)


@pytest.mark.parametrize('K,N,B,snr,nb,qt,ms', [
    (10, 64, 400, 10, 3, 'lloyd', 0.1),          # Lloyd-Max labels are not on an integer grid
    (7, 32, 300, 0, 2, 'lloyd', 0.0),
    (6, 64, 260, 15, np.inf, 'uniform', 0.2),    # unquantised pilots
    (5, 128, 390, 10, 3, 'lloyd', 0.1),          # large shape: one resident (hi, lo) tile pair per CTA, split launches
    (4, 96, 131, 5, np.inf, 'uniform', 0.0),
])
def test_tc_off_grid_pilots_three_pass(qce, K, N, B, snr, nb, qt, ms):
    """Pilots that are not integer multiples of a step are staged as FP16 (hi, lo) tile pairs: three tensor passes."""
    means, covs, w = orc.random_psd_gmm(K, N, seed=K + N, mean_scale=ms)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=K)
    qz = orc.get_quantizer([snr], nb, qt)[snr] if np.isfinite(nb) else (None, None, None)
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    _check_modes(lambda mode: m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz).cpu().numpy(),
                 lambda mode: orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt,
                                                      quantizer=qz), B)
    if np.isfinite(nb):     # fused observe -> quantise -> estimate pipeline with Lloyd-Max tables
        from quantized_channel_estimation_b200 import engine, precompute
        model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, nb, qt, qz))
        quant = engine.Quantizer.get(nb, qz[0], qz[1])
        est, acc = model.pipeline(quant, torch.from_numpy(h).cuda(), torch.from_numpy(noise).cuda(), 10 ** (-snr / 20), 'all', 'tc', want_est=True)
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
        assert relerr(est.cpu().numpy(), ref) < TOL_TC
        assert acc.cpu().numpy()[2] == B


def test_tc_mode_path_is_chunked(qce):
    """The log-probability / weight scratch of the three-launch path is bounded: large batches are walked in chunks of whole work
    units (QCE_TC_MODE_CHUNK shrinks the chunk for this test); results must not depend on the chunking."""
    import os
    K, N, B, snr = 5, 32, 1700, 5
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.1, seed=77)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    model = m._prepared(np.eye(N), snr, 1, 'uniform', None)
    ref = {mode: model.estimate(rt, mode, 'tc', want_logp=True, h_true=torch.from_numpy(h).cuda()) for mode in (1, 3, 0.9)}
    os.environ['QCE_TC_MODE_CHUNK'] = '512'
    try:
        for mode, (e0, l0, a0) in ref.items():
            e1, l1, a1 = model.estimate(rt, mode, 'tc', want_logp=True, h_true=torch.from_numpy(h).cuda())
            assert torch.equal(e0, e1) and torch.equal(l0, l1)
            np.testing.assert_allclose(a0.cpu().numpy(), a1.cpu().numpy(), rtol=1e-12)
    finally:
        del os.environ['QCE_TC_MODE_CHUNK']


@pytest.mark.parametrize('scale,snr,nb', [(1e4, 0, 1), (1e-4, 0, 1), (1.0, 40, 1), (1e3, 20, 2), (1.0, -30, 2)])
def test_tc_parameter_scales_and_extreme_snr(qce, scale, snr, nb):
    """Channel power far from one and extreme SNRs: the power-of-two normalisation of the FP16 operand images and the FP32 (hi, lo)
    log-probabilities must hold the tensor-core path on the oracle."""
    K, N, B = 7, 32, 300
    means, covs, w = orc.random_psd_gmm(K, N, seed=91, mean_scale=0.1)
    means, covs = means * np.sqrt(scale), covs * scale
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=92)
    qz = orc.get_quantizer([snr], nb, 'uniform')[snr]
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    _check_modes(lambda mode: m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer=qz).cpu().numpy(),
                 lambda mode: orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer=qz), B)


@pytest.mark.parametrize('K,N,c64', [(64, 64, True), (128, 64, False), (32, 32, True)])
def test_tc_pipeline_nan_zero_and_ragged_tail(qce, K, N, c64):
    """The fused Monte-Carlo step (observe + 1-bit quantise + estimate) on the tensor-core path against the complex128 path on the same
    inputs: a NaN noise entry (its row is NaN, like numpy), an element with y = 0 exactly, complex64 and complex128 channels, and a
    ragged tail over several work units per CTA."""
    from quantized_channel_estimation_b200 import engine, precompute
    B, snr = 148 * 512 * 2 + 777, 5
    means, covs, w = orc.random_psd_gmm(K, N, seed=K + N, mean_scale=0.1)
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1))
    quant = engine.Quantizer.get(1)
    g = torch.Generator(device='cuda').manual_seed(12)
    h = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float32 if c64 else torch.float64)).contiguous()
    noise = torch.view_as_complex(torch.randn((B, N, 2), generator=g, device='cuda', dtype=torch.float64)).contiguous()
    noise[5, 3] = complex(float('nan'), 0.0)
    h[B - 2, 0] = 0.0
    noise[B - 2, 0] = 0.0                          # y = 0 exactly: np.sign gives 0, both paths must carry the value 0
    est, acc = model.pipeline(quant, h, noise, 10 ** (-snr / 20), 'all', 'tc', want_est=True)
    est64, _ = model.pipeline(quant, h, noise, 10 ** (-snr / 20), 'all', 'fp64', want_est=True)
    assert bool(torch.isnan(est[5].real).all()) and bool(torch.isfinite(est[B - 2]).all())
    assert torch.equal(torch.isnan(est.real), torch.isnan(est64.real))
    ok = ~torch.isnan(est64.real).any(dim=1)
    per = (est[ok] - est64[ok]).norm(dim=1) / est64[ok].norm(dim=1).clamp(min=1e-300)
    assert float((est[ok] - est64[ok]).norm() / est64[ok].norm()) < TOL_TC and float(per.max()) < 1e-4
    assert acc[2].item() == B


def test_tc_single_component_and_many_components(qce):
    """K = 1, and K = 130 / 300: the selection kernel holds 2, 8 or 32 entries per lane depending on K."""
    for K, N in ((1, 64), (130, 16), (300, 16)):
        B = 300
        means, covs, w, h, noise, qz, r = _case(K, N, B, 10, 1, 'uniform', 0.0, seed=K)
        m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
        m.precision = 'tc'
        rt = torch.from_numpy(r).cuda()
        _check_modes(lambda mode: m.estimate_from_y(rt, 10, N, n_summands_or_proba=mode).cpu().numpy(),
                     lambda mode: orc.gmm_estimate_from_y(means, covs, w, r, 10, n_summands_or_proba=mode, n_bits=1), B)


@pytest.mark.parametrize('mode', ['all', 1, 3, 0.9])
def test_tc_off_grid_pilots_are_reevaluated_in_complex128(qce, mode):
    """Data that is not on the declared quantiser grid cannot be represented exactly in the FP16 pilot tiles: those rows are answered
    by the complex128 kernel (the reference gives a finite estimate for ANY y), NaN data gives NaN like numpy, and the NMSE
    accumulators count every row once."""
    K, N, B, snr = 4, 32, 700, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.0, seed=2)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    bad = r.copy()
    bad[7, 3] = 0.3 + 0.1j
    bad[600, :] = 0.25 * r[600]
    bad[150, 0] = complex(np.nan, 0.0)
    est = m.estimate_from_y(torch.from_numpy(bad).cuda(), snr, N, n_summands_or_proba=mode).cpu().numpy()
    finite = np.ones(B, bool)
    finite[150] = False
    ref = orc.gmm_estimate_from_y(means, covs, w, bad[finite], snr, n_summands_or_proba=mode, n_bits=1)
    assert np.isnan(est[150].view(np.float64)).all()
    per = np.linalg.norm(est[finite] - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert per.max() < 1e-4 and relerr(est[finite], ref) < TOL_TC
    assert relerr(est[[7, 600]], ref[[7, 599]]) < TOL_FP64          # the two off-grid rows: complex128 arithmetic
    # accumulators: every (finite) row exactly once
    model = m._prepared(np.eye(N), snr, 1, 'uniform', None)
    _, acc = model.estimate(torch.from_numpy(bad[finite]).cuda(), mode, 'tc', h_true=torch.from_numpy(h[finite]).cuda())
    acc = acc.cpu().numpy()
    assert acc[2] == B - 1
    np.testing.assert_allclose(acc[0], np.sum(np.abs(ref - h[finite]) ** 2), rtol=1e-5)


def test_tc_whole_batch_off_grid_falls_to_complex128(qce):
    """Uniform 2-bit pilots quantised with the step of ANOTHER SNR than the one passed to estimate_from_y (ADVICE r1): no row is on the
    expected grid; the answer is still the reference's."""
    K, N, B = 5, 32, 300
    means, covs, w, h, noise, qz, r = _case(K, N, B, 0, 2, 'uniform', 0.1, seed=4)      # quantised for 0 dB
    qz10 = orc.get_quantizer([10], 2, 'uniform')[10]
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    for mode in ('all', 1):
        ref = orc.gmm_estimate_from_y(means, covs, w, r, 10, n_summands_or_proba=mode, n_bits=2, quantizer_type='uniform', quantizer=qz10)
        est = m.estimate_from_y(torch.from_numpy(r).cuda(), 10, N, n_summands_or_proba=mode, n_bits=2, quantizer_type='uniform', quantizer=qz10)
        assert relerr(est.cpu().numpy(), ref) < TOL_FP64


def test_tc_non_triangular_whitening_uses_single_cta_variant(qce):
    """A whitening factor that is not lower triangular (Q L^-1 with Q unitary gives the same quadratic form) takes the
    cta_group::1 variant without column skipping; results must not change."""
    from quantized_channel_estimation_b200 import precompute, engine
    K, N, B, snr = 6, 64, 700, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.2, seed=11)
    prep = precompute.prepare(means, covs, w, np.eye(N), snr, 1)
    rng = np.random.default_rng(0)
    Q = torch.as_tensor(np.linalg.qr(orc.crandn(N, N, rng=rng))[0]).to(prep['Linv'].device)
    prep2 = dict(prep)
    prep2['Linv'] = (Q[None] @ prep['Linv']).contiguous()
    prep2['zoff'] = (Q[None] @ prep['zoff'][:, :, None])[:, :, 0].contiguous()
    ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=1)
    rt = torch.from_numpy(r).cuda()
    for p in (prep, prep2):
        model = engine.DenseModel(p)
        est = model.estimate(rt, 'all', 'tc').cpu().numpy()
        assert relerr(est, ref) < TOL_TC
        est64 = model.estimate(rt, 'all', 'fp64').cpu().numpy()
        assert relerr(est64, ref) < 1e-9


@pytest.mark.gpu
def test_c_abi_error_behaviour(qce):
    """The C ABI reports misuse through its status codes and ``qce_last_error_string`` (include/qce_b200.h:34-40) instead of
    crashing, and an empty batch is a valid no-op -- the reference's numpy code returns an empty array for it."""
    import ctypes as C
    from quantized_channel_estimation_b200 import _lib
    lib = _lib.require_device()
    INVALID, UNSUPPORTED = -1, -3
    err = lambda: lib.qce_last_error_string().decode()
    h = C.c_void_p()
    assert lib.qce_model_create(0, 8, 4, 0, C.byref(h)) == INVALID and 'shape' in err()
    assert lib.qce_model_create(8, 8, 4, 0, None) == INVALID
    assert lib.qce_quantizer_create(0, None, None, C.byref(h)) == INVALID and 'n_bits' in err()
    assert lib.qce_quantizer_create(2, None, None, C.byref(h)) == INVALID and 'tables' in err()
    thr = (C.c_double * 3)(0.5, -0.5, 1.0)                   # not ascending
    lab = (C.c_double * 4)(-1.5, -0.5, 0.5, 1.5)
    assert lib.qce_quantizer_create(2, thr, lab, C.byref(h)) == INVALID and 'ascend' in err()

    m = C.c_void_p()
    assert lib.qce_model_create(20, 20, 5, 0, C.byref(m)) == 0
    try:
        r = torch.zeros((4, 20), dtype=torch.complex128, device='cuda')
        out = torch.empty_like(r)
        # a model without parameters refuses to estimate
        assert lib.qce_estimate(m, None, r.data_ptr(), 4, 0, 0, 0.0, 0, out.data_ptr(), None, None, None) == INVALID
        assert 'no parameters' in err()
        assert lib.qce_model_set_params(m, None, None, None, None, None, None, 0.0) == INVALID
        K, N = 5, 20
        eye = torch.eye(N, dtype=torch.complex128, device='cuda').repeat(K, 1, 1).contiguous()
        z = torch.zeros((K, N), dtype=torch.complex128, device='cuda')
        lc = torch.zeros(K, dtype=torch.float64, device='cuda')
        assert lib.qce_model_set_params(m, None, eye.data_ptr(), eye.data_ptr(), z.data_ptr(), z.data_ptr(), lc.data_ptr(),
                                        -1.0) == INVALID
        assert lib.qce_model_set_params(m, None, eye.data_ptr(), eye.data_ptr(), z.data_ptr(), z.data_ptr(), lc.data_ptr(),
                                        0.0) == 0
        args = lambda B, mode, ntop, rho, prec, rp=r.data_ptr(): (m, None, rp, B, mode, ntop, rho, prec, out.data_ptr(), None,
                                                                   None, None)
        assert lib.qce_estimate(*args(-1, 0, 0, 0.0, 0)) == INVALID
        assert lib.qce_estimate(*args(4, 0, 0, 0.0, 0, rp=None)) == INVALID
        assert lib.qce_estimate(*args(4, 7, 0, 0.0, 0)) == INVALID and 'unknown mode' in err()
        assert lib.qce_estimate(*args(4, _lib.MODE_TOPN, 0, 0.0, 0)) == INVALID and 'n_top' in err()
        assert lib.qce_estimate(*args(4, _lib.MODE_CUMPROB, 0, float('nan'), 0)) == INVALID and 'NaN' in err()
        assert lib.qce_estimate(*args(4, 0, 0, 0.0, 9)) == INVALID and 'precision' in err()
        # N = 20 is not a tensor-core shape: asking for that kernel explicitly is refused, never silently rerouted
        assert lib.qce_estimate(*args(4, 0, 0, 0.0, _lib.PREC_TC)) == UNSUPPORTED and 'tensor-core' in err()
        assert lib.qce_format_pilots(m, None, r.data_ptr(), 4) == UNSUPPORTED
        # empty batch: OK, nothing written
        out.fill_(7.0)
        assert lib.qce_estimate(*args(0, 0, 0, 0.0, 0, rp=None)) == 0
        torch.cuda.synchronize()
        assert bool((out == 7.0).all())
        # and a valid call still works afterwards (identity filters, equal weights -> h = r)
        r2 = torch.randn((4, 20), dtype=torch.complex128, device='cuda')
        assert lib.qce_estimate(*args(4, 0, 0, 0.0, 0, rp=r2.data_ptr())) == 0
        torch.cuda.synchronize()
        assert torch.allclose(out, r2, rtol=1e-12, atol=1e-12)
        host_in = np.zeros((4, 20), dtype=np.complex128)
        assert lib.qce_estimate_host(m, None, 4, 0, 0, 0.0, 0, host_in.ctypes.data) == INVALID
        assert lib.qce_estimate_host(m, host_in.ctypes.data, 0, 0, 0, 0.0, 0, None) == 0
    finally:
        lib.qce_model_destroy(m)
    # pipeline needs a square pilot matrix (A = I)
    m2 = C.c_void_p()
    assert lib.qce_model_create(8, 16, 2, 0, C.byref(m2)) == 0
    try:
        q = C.c_void_p()
        assert lib.qce_quantizer_create(1, None, None, C.byref(q)) == 0
        x = torch.zeros((2, 16), dtype=torch.complex128, device='cuda')
        assert lib.qce_pipeline(m2, q, None, x.data_ptr(), 0, x.data_ptr(), 1.0, 2, 0, 0, 0.0, 0, None, None) == INVALID
        assert 'n_obs == n_ant' in err()
        lib.qce_quantizer_destroy(q)
    finally:
        lib.qce_model_destroy(m2)


@pytest.mark.gpu
@pytest.mark.parametrize('K,N,B,snr,nb,qt,ms,kind', [
    (64, 64, 6000, 10, 1, 'uniform', 0.0, 'gmm'),       # config-2 shape, fused-shape model on the per-purpose launches
    (5, 32, 2500, 0, 2, 'uniform', 0.1, 'gmm'),         # means: offsets in the combine epilogue; some buckets nearly empty
    (9, 128, 4200, 10, 2, 'uniform', 0.0, 'gmm'),       # split shape: two LMMSE row blocks per pilot
    (6, 128, 2100, 5, 3, 'lloyd', 0.1, 'gmm'),          # off-grid pilots: (hi, lo) tile pairs, one tile per CTA
    (8, 64, 3000, 10, 1, 'uniform', 0.0, 'mfa'),        # MFA: argmax of exp(l) (label 0 on underflow)
])
def test_tc_top1_bucketed_combination(qce, K, N, B, snr, nb, qt, ms, kind):
    """Top-1 on large batches regroups the pilots by selected component and runs ONE component per work unit (1/K of the combine
    work).  Must equal the weighted three-launch path bit for bit (QCE_TC_BUCKET=0), NaN rows and NMSE accumulators included, and
    match the oracle."""
    import os
    if kind == 'gmm':
        means, covs, w = orc.random_psd_gmm(K, N, seed=K + N, mean_scale=ms)
        h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=K)
        m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
        oracle = lambda r, qz: orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=1, n_bits=nb, quantizer_type=qt,
                                                       quantizer=qz)
    else:
        means, lam, psi, w = orc.random_mfa(K, N, 4, seed=K + N)
        covs = orc.mofa_covs(lam, psi)
        h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=K)
        m = qce.Mofa(K, 4, verbose=False).set_parameters(means, lam, psi, w)
        oracle = lambda r, qz: orc.mofa_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=1, n_bits=nb, quantizer_type=qt,
                                                        quantizer=qz)
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    r[17, 3] = np.nan                                     # a row the tensor path cannot represent: NaN estimate, still counted
    m.precision = 'tc'
    model = m._prepared(np.eye(N), snr, nb, qt, qz)
    rt, ht = torch.from_numpy(r).cuda(), torch.from_numpy(h).cuda()
    e1, l1, a1 = model.estimate(rt, 1, 'tc', want_logp=True, h_true=ht)
    e2, a2 = model.estimate(rt, 1, 'tc', h_true=ht)       # no log-probability export: the whitening launch keeps the argmax itself
    os.environ['QCE_TC_BUCKET'] = '0'
    try:
        e0, l0, a0 = model.estimate(rt, 1, 'tc', want_logp=True, h_true=ht)
    finally:
        del os.environ['QCE_TC_BUCKET']
    ok = torch.ones(B, dtype=torch.bool, device='cuda'); ok[17] = False
    assert torch.equal(e0[ok], e1[ok]) and torch.equal(l0[ok], l1[ok])
    assert torch.equal(e1[ok], e2[ok])
    assert bool(torch.isnan(e1[17]).all()) and bool(torch.isnan(e0[17]).all()) and bool(torch.isnan(e2[17]).all())
    assert a1.cpu().numpy()[2] == B and a2.cpu().numpy()[2] == B
    good = np.ones(B, dtype=bool); good[17] = False
    ref = oracle(r[good], qz)
    per = np.linalg.norm(e1.cpu().numpy()[good] - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert np.mean(per > TOL_TC) < 0.01, np.mean(per > TOL_TC)          # near-ties may pick the other component under FP32


@pytest.mark.gpu
def test_tc_top1_bucketed_full_size_chunks(qce):
    """Config-2 size (2^19 pilots, K = 64, N = 64, 1 bit): the bucketed top-1 path over several chunks (bucket scratch reused, ragged
    last chunk) equals the weighted three-launch path bit for bit, and every pilot is written exactly once."""
    import os
    from quantized_channel_estimation_b200 import synthetic
    K, N, B, snr = 64, 64, (1 << 19) - 77, 10
    means, covs, w = synthetic.random_psd_gmm(K, N, seed=0)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    model = m._prepared(np.eye(N), snr, 1, 'uniform', None)
    gen = torch.Generator(device='cuda').manual_seed(5)
    bits = torch.randint(0, 2, (B, N, 2), generator=gen, device='cuda', dtype=torch.int8)
    r = torch.view_as_complex(((bits.to(torch.float64) * 2 - 1) * np.sqrt(0.5)).contiguous())
    h_true = torch.view_as_complex(torch.randn((B, N, 2), generator=gen, device='cuda', dtype=torch.float64))
    os.environ['QCE_TC_BUCKET'] = '0'
    try:
        e0, a0 = model.estimate(r, 1, 'tc', h_true=h_true)
    finally:
        del os.environ['QCE_TC_BUCKET']
    e1, a1 = model.estimate(r, 1, 'tc', h_true=h_true)
    assert torch.equal(e0, e1)
    os.environ['QCE_TC_MODE_CHUNK'] = '150000'
    try:
        e2, a2 = model.estimate(r, 1, 'tc', h_true=h_true)
    finally:
        del os.environ['QCE_TC_MODE_CHUNK']
    assert torch.equal(e0, e2) and not bool(torch.isnan(e2.real).any())
    for a in (a1, a2):
        np.testing.assert_allclose(a.cpu().numpy(), a0.cpu().numpy(), rtol=1e-9)
        assert a.cpu().numpy()[2] == B


@pytest.mark.gpu
def test_circulant_model_beyond_structured_limits_takes_the_dense_path(qce):
    """ADVICE r1: a zero-mean plain-circulant model with 256 < N <= 1024 is detected as structured, but the DFT-domain kernels stop at
    256 bins per axis -- estimate_from_y must fall back to the dense path (what the reference computes), not raise."""
    K, N, B, snr = 3, 512, 40, 5
    c, covs, w, F = orc.circulant_gmm(K, 1, N, seed=9)
    h, noise, _ = orc.sample_gmm_channels(np.zeros((K, N), complex), covs, w, B, seed=5)
    r = orc.get_observation_nbit(h, snr, noise, None, 1)
    m = qce.Gmm_nbit(n_components=K, covariance_type='circulant').set_parameters(np.zeros((K, N)), covs, w, zero_mean=True)
    assert m.blocks == (1, N)
    from quantized_channel_estimation_b200.engine import DenseModel
    assert isinstance(m._prepared(np.eye(N), snr, 1, 'uniform', None), DenseModel)
    est = m.estimate_from_y(r, snr, N, n_summands_or_proba='all', n_bits=1)
    ref = orc.gmm_estimate_from_y(np.zeros((K, N)), covs, w, r, snr, n_summands_or_proba='all', n_bits=1)
    assert relerr(est, ref) < 1e-8


@pytest.mark.gpu
def test_prepared_cache_follows_in_place_parameter_edits(qce):
    """The prepared-model cache is keyed by the CONTENT of the parameter arrays: an in-place edit must not serve a stale GPU handle."""
    K, N, B, snr = 4, 16, 64, 5
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.2, seed=11)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'fp64'
    e0 = m.estimate_from_y(r, snr, N, n_summands_or_proba='all')
    with pytest.raises(ValueError):           # set_parameters froze the arrays: an in-place edit cannot go unnoticed
        m.means_cplx *= 0.5
    buf = np.array(means)                     # a caller-owned, writable array assigned directly ...
    m.means_cplx = buf
    assert relerr(m.estimate_from_y(r, snr, N, n_summands_or_proba='all'), e0) < 1e-14
    buf *= 0.5                                # ... and edited in place: same identity, the strided content sample follows the edit
    e1 = m.estimate_from_y(r, snr, N, n_summands_or_proba='all')
    ref = orc.gmm_estimate_from_y(0.5 * means, covs, w, r, snr, n_summands_or_proba='all', n_bits=1)
    assert relerr(e1, ref) < TOL_FP64 and relerr(e0, ref) > 1e-3


@pytest.mark.gpu
def test_last_fix_count_reports_reevaluated_rows(qce):
    import ctypes as C
    from quantized_channel_estimation_b200 import _lib
    K, N, B, snr = 4, 32, 300, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.0, seed=2)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    bad = r.copy()
    bad[[3, 77, 200], 0] = 0.123
    m.estimate_from_y(torch.from_numpy(bad).cuda(), snr, N, n_summands_or_proba='all')
    assert _lib.load().qce_last_fix_count(C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 3


@pytest.mark.gpu
@pytest.mark.parametrize('tag,ctype,blocks,zm', [('full_zm', 'full', None, True), ('full_mean', 'full', None, False),
                                                 ('toep', 'toeplitz', None, True)])
def test_fit_on_gpu_reaches_reference_likelihood(qce, tag, ctype, blocks, zm):
    """fit() on the GPU -- E-step on the inference path's whitening launch (tensor cores, N = 4 / 8 zero-padded to 16), batched M-step
    -- against the likelihood the UNMODIFIED reference EM reaches on the same seeded data (tests/golden/fit.npz)."""
    import warnings
    from conftest import load_golden
    from fit_common import avg_loglik, make_data
    from quantized_channel_estimation_b200 import _lib
    gold = load_golden('fit')
    h, true = make_data(tag)
    g = qce.Gmm_nbit(n_components=3, covariance_type=ctype, random_state=0, max_iter=200, tol=1e-5, n_init=2 if ctype == 'full' else 1)
    l0 = _lib.launch_count()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        g.fit(h, blocks=blocks, zero_mean=zm)
    assert _lib.launch_count() - l0 > 10, 'the E-step did not run on the library kernels'
    ll = avg_loglik(h, g.gm.weights_, g.means_cplx, g.covs_cplx)
    if ctype == 'full':
        assert ll > float(gold[f'{tag}_ref_ll']) - 0.02, (ll, float(gold[f'{tag}_ref_ll']))
        assert ll > float(gold[f'{tag}_true_ll']) - 0.02
    else:
        assert abs(ll - float(gold[f'{tag}_ref_ll'])) < 0.02, (ll, float(gold[f'{tag}_ref_ll']))


@pytest.mark.gpu
def test_kernel_estep_matches_torch_log_prob(qce):
    """The E-step's log-densities from the whitening launch (three-pass tensor-core path, padded shape) against the torch formula."""
    from quantized_channel_estimation_b200 import em
    from fit_common import make_data
    h, (w, means, covs) = make_data('full_mean')
    X = torch.as_tensor(h, dtype=torch.complex128, device='cuda')
    wt, mt, ct = (torch.as_tensor(a, device='cuda') for a in (w, means, covs))
    ks = em._KernelEStep(X)
    assert ks.ok
    lp_k = ks.log_prob(wt, mt.to(torch.complex128), ct.to(torch.complex128))
    lp_t = em._log_prob(X, wt, mt.to(torch.complex128), ct.to(torch.complex128), False)
    assert float((lp_k - lp_t).abs().max()) < 2e-4 * max(1.0, float(lp_t.abs().max()) / 50)


@pytest.mark.gpu
@pytest.mark.parametrize('N,K,nb,qt', [(20, 5, 1, 'uniform'), (8, 4, 2, 'uniform'), (40, 6, 3, 'lloyd')])
def test_tc_zero_padded_shapes(qce, N, K, nb, qt):
    """Antenna counts that are not multiples of 16 run on the tensor cores zero-padded to the next instantiated shape."""
    from quantized_channel_estimation_b200.engine import DenseModel
    B, snr = 300, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, qt, 0.2, seed=N)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    model = m._prepared(np.eye(N), snr, nb, qt, qz)
    assert isinstance(model, DenseModel) and model.padded
    for mode in ('all', 1, 2, 0.9):
        ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz)
        est = m.estimate_from_y(torch.from_numpy(r).cuda(), snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz).cpu().numpy()
        assert est.shape == (B, N)
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert relerr(est, ref) < TOL_TC and per.max() < 1e-4, (mode, relerr(est, ref), per.max())
    # host arrays, responsibilities and the NMSE accumulators go through the padded handle too
    est_h = m.estimate_from_y(r, snr, N, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
    ref = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz)
    assert relerr(est_h, ref) < TOL_TC
    _, aux = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=nb, quantizer_type=qt, quantizer=qz, return_aux=True)
    np.testing.assert_allclose(m.predict_proba_cplx(r), aux['proba'], atol=2e-4)
    _, acc = model.estimate(torch.from_numpy(r).cuda(), 'all', 'tc', h_true=torch.from_numpy(h).cuda())
    np.testing.assert_allclose(acc.cpu().numpy()[0], np.sum(np.abs(ref - h) ** 2), rtol=1e-5)


@pytest.mark.gpu
def test_predict_proba_runs_on_the_whitening_launch(qce):
    """predict_proba_cplx / _predict_cplx with the default precision use the tensor-core whitening launch (log-probabilities only, no
    combination launches) and agree with the complex128 kernel."""
    from quantized_channel_estimation_b200 import _lib
    K, N, B, snr = 16, 64, 4000, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.0, seed=3)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    rt = torch.from_numpy(r).cuda()
    m.estimate_from_y(rt[:8], snr, N, n_summands_or_proba='all')
    l0 = _lib.launch_count()
    p_tc = m.predict_proba_cplx(rt)
    n_launch = _lib.launch_count() - l0
    m.precision = 'fp64'
    m.estimate_from_y(rt[:8], snr, N, n_summands_or_proba='all')
    p_64 = m.predict_proba_cplx(rt)
    assert n_launch <= 4                       # format, whitening, selection / export, (empty) complex128 fix-up
    assert float((p_tc - p_64).abs().max()) < 1e-4
    m.precision = 'auto'
    m.estimate_from_y(rt[:8], snr, N, n_summands_or_proba='all')
    lab = m._predict_cplx(rt)
    assert float((lab != p_64.argmax(1)).float().mean()) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize('K,N,nb,qt,snr', [(64, 64, 1, 'uniform', 10), (16, 128, 2, 'uniform', 10), (64, 64, 1, 'uniform', -10)])
def test_tc_pair_bucketed_combination(qce, K, N, nb, qt, snr):
    """Top-n / cumulative-rho (and 'all' on the large shapes) through the pair-bucketed combination -- only the (pilot, component)
    pairs with a weight that matters, regrouped by component -- against the dense weighted launch (QCE_TC_PAIRS=0) and the oracle.
    -10 dB: the posterior is flat, the device-side decision falls back to the weighted launch; results must not change."""
    import os
    B = 20000
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, qt, 0.1, seed=K + N)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    m.precision = 'tc'
    rt, ht = torch.from_numpy(r).cuda(), torch.from_numpy(h).cuda()
    model = m._prepared(np.eye(N), snr, nb, qt, qz)
    for mode in ((2, 4, 0.9) if N <= 64 else ('all', 3, 0.95)):
        try:
            os.environ['QCE_TC_PAIRS'] = '1'       # (the default is on for n_obs > 64 only)
            est, acc = model.estimate(rt, mode, 'tc', h_true=ht)
            os.environ['QCE_TC_PAIRS'] = '0'
            est0, acc0 = model.estimate(rt, mode, 'tc', h_true=ht)
        finally:
            del os.environ['QCE_TC_PAIRS']
        per = ((est - est0).norm(dim=1) / est0.norm(dim=1)).max()
        assert float(per) < 2e-6, (mode, float(per))
        acc, acc0 = acc.cpu().numpy(), acc0.cpu().numpy()
        assert acc[2] == acc0[2] == B
        np.testing.assert_allclose(acc[:2], acc0[:2], rtol=1e-5)
        nref = 3000
        ref = orc.gmm_estimate_from_y(means, covs, w, r[:nref], snr, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz)
        e = est[:nref].cpu().numpy()
        pr = np.linalg.norm(e - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert pr.max() < 1e-4 and relerr(e, ref) < TOL_TC, (mode, pr.max())
    # NMSE accumulators only (no estimate buffer from the caller): the fused pipeline entry point
    from quantized_channel_estimation_b200 import engine
    if nb == 1:
        quant = engine.Quantizer.get(1)
        os.environ['QCE_TC_PAIRS'] = '1'
        try:
            accp = model.pipeline(quant, ht, torch.from_numpy(noise).cuda(), 10 ** (-snr / 20), 4, 'tc')
        finally:
            del os.environ['QCE_TC_PAIRS']
        est4 = model.estimate(rt, 4, 'tc')
        np.testing.assert_allclose(accp.cpu().numpy()[0], float(((est4 - ht).abs() ** 2).sum()), rtol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize('nb,qt', [(1, 'uniform'), (2, 'uniform'), (3, 'lloyd')])
def test_estimate_from_codes_host_path(qce, nb, qt):
    """qce_estimate_host_codes: uint8 level codes in, complex64 / complex128 estimates out -- the same estimates as estimate_from_y on the
    complex128 pilots the codes stand for (bit-identical for complex128 output, narrowed for complex64)."""
    from quantized_channel_estimation_b200 import engine
    K, N, B, snr = 8, 32, 5000, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, qt, 0.1, seed=nb)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    q = engine.Quantizer.get(1) if nb == 1 else engine.Quantizer.get(nb, qz[0], qz[1])
    y = torch.from_numpy(h + 10 ** (-snr / 20) * noise).cuda()
    r_dev, codes = q.quantize(y, want_codes=True)
    assert _bits_equal(r_dev.cpu().numpy(), r)
    codes = codes.cpu().numpy()
    for mode in ('all', 1, 3):
        ref = m.estimate_from_y(r, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz)
        e128 = m.estimate_from_codes(codes, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz, out_dtype=np.complex128)
        e64 = m.estimate_from_codes(codes, snr, N, n_summands_or_proba=mode, n_bits=nb, quantizer_type=qt, quantizer=qz)
        assert e128.dtype == np.complex128 and e64.dtype == np.complex64
        assert np.array_equal(e128, ref)
        assert np.array_equal(e64, ref.astype(np.complex64))


@pytest.mark.gpu
def test_predict_proba_right_after_set_parameters_uses_the_trained_mixture(qce):
    """ADVICE r1: with no observation setting prepared yet, predict_proba / predict_proba_cplx are the responsibilities under the
    trained (channel-domain) mixture -- what the reference computes right after fit() -- instead of an error."""
    from fit_common import make_data
    h, (w, means, covs) = make_data('full_mean')

    def resp(x):
        lp = np.empty((x.shape[0], len(w)))
        for k in range(len(w)):
            d = x - means[k]
            lp[:, k] = np.log(w[k]) - x.shape[1] * np.log(np.pi) - np.linalg.slogdet(covs[k])[1] - np.real(np.sum(d.conj() * np.linalg.solve(covs[k], d.T).T, axis=1))
        lp -= lp.max(1, keepdims=True)
        return np.exp(lp) / np.exp(lp).sum(1, keepdims=True)
    ref = resp(h[:500])
    g = qce.Gmm_nbit(n_components=3).set_parameters(means, covs, w, detect_structure=False)
    np.testing.assert_allclose(g.predict_proba_cplx(h[:500]), ref, atol=2e-4)
    g.precision = 'fp64'
    g._cache.clear(); g._last = None
    np.testing.assert_allclose(g.predict_proba_cplx(h[:500]), ref, atol=1e-10)
    hm, (wm, mm, cm) = make_data('mfa')
    m = qce.Mofa(3, 2, verbose=False)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m.fit(hm[:1500], zero_mean=False)
    p = m.predict_proba(hm[:200])
    assert p.shape == (200, 3) and np.allclose(p.sum(1), 1.0, atol=1e-6)


@pytest.mark.gpu
def test_two_gpus_in_one_process(qce):
    """ADVICE r1: scratch, fix lists, shared-memory attributes and host staging are per device -- a process may drive several GPUs.
    (Skipped where fewer than two GPUs are visible.)"""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    K, N, B, snr = 8, 32, 3000, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.1, seed=5)
    ref = {mode: orc.gmm_estimate_from_y(means, covs, w, r[:500], snr, n_summands_or_proba=mode, n_bits=1) for mode in ('all', 1, 3)}
    models = []
    for d in (0, 1):
        with torch.cuda.device(d):
            m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
            models.append((m, torch.from_numpy(r).to(f'cuda:{d}')))
    for rep in range(2):                      # interleaved: both devices use the default stream (handle 0 on each)
        for d, (m, rt) in enumerate(models):
            with torch.cuda.device(d):
                for mode in ('all', 1, 3):
                    for prec in ('tc', 'fp64'):
                        m.precision = prec
                        est = m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode)
                        assert est.device.index == d
                        assert relerr(est[:500].cpu().numpy(), ref[mode]) < TOL_TC
                m.precision = 'tc'
                assert relerr(m.estimate_from_y(r[:500], snr, N, n_summands_or_proba='all'), ref['all']) < TOL_TC      # host path on device d


@pytest.mark.gpu
@pytest.mark.parametrize('K,N,nb,qt,B', [(8, 64, 1, 'uniform', 900), (6, 128, 2, 'uniform', 700), (5, 48, 3, 'lloyd', 500), (4, 40, 1, 'uniform', 300)])
def test_tc_launch_time_knobs_do_not_change_results(qce, K, N, nb, qt, B, monkeypatch):
    """Every launch-time knob of the tensor-core path (DESIGN.md knobs table) selects another route to the SAME estimates: all pilots sent
    through the complex128 re-selection (QCE_TC_TIE_EPS=0.5), pair-bucketed / weighted combination, bucketed top-1 off -- on the
    fused shape, the split path, the three-pass path and a zero-padded shape, all four modes, with some pilots off the grid."""
    snr = 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, qt, 0.1, seed=K)
    r = r.copy()
    r[::7] *= 1.37                                              # off the declared grid: re-evaluated in complex128 inside the call
    rt = torch.from_numpy(r).cuda()
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    kw = dict(n_bits=nb, quantizer_type=qt, quantizer=qz)
    modes = ('all', 1, 3, 0.9)
    m.precision = 'fp64'
    ref = {mode: m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, **kw) for mode in modes}
    m.precision = 'tc'
    base = {mode: m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, **kw) for mode in modes}
    for mode in modes:
        assert relerr(base[mode].cpu().numpy(), ref[mode].cpu().numpy()) < TOL_TC
    for knob, val in (('QCE_TC_TIE_EPS', '0.5'), ('QCE_TC_PAIRS', '1'), ('QCE_TC_PAIRS', '0'), ('QCE_TC_BUCKET', '0')):
        monkeypatch.setenv(knob, val)
        for mode in modes:
            got = m.estimate_from_y(rt, snr, N, n_summands_or_proba=mode, **kw)
            assert relerr(got.cpu().numpy(), ref[mode].cpu().numpy()) < TOL_TC, (knob, val, mode)
            # hard selections are the same selections, whatever the route
            if mode != 'all':
                rows = (got - base[mode]).norm(dim=1) / base[mode].norm(dim=1).clamp(min=1e-300)
                assert float(rows.max()) < 1e-4, (knob, val, mode, float(rows.max()))
        monkeypatch.delenv(knob)


@pytest.mark.gpu
def test_concurrent_host_threads_on_their_own_streams(qce):
    """SURVEY 8b threading contract: a model handle is immutable after set_params and qce_estimate is stream-ordered and re-entrant across
    streams and handles.  Four host threads, each on its own stream, share one model and own another; all modes, tensor-core and complex128
    paths, device tensors and host arrays; results equal the serial ones."""
    import threading
    K, N, B, snr = 16, 64, 6000, 10
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, 1, 'uniform', 0.1, seed=11)
    shared = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    shared.precision = 'tc'
    rt = torch.from_numpy(r).cuda()
    modes = ('all', 1, 3, 0.9)
    serial = {mode: shared.estimate_from_y(rt, snr, N, n_summands_or_proba=mode) for mode in modes}
    torch.cuda.synchronize()
    errors = []

    def worker(i):
        try:
            st = torch.cuda.Stream()
            own = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
            own.precision = 'tc' if i % 2 else 'fp64'
            sl = slice(i * 1000, i * 1000 + 1500)
            with torch.cuda.stream(st):
                mine = rt[sl].clone()
                for rep in range(6):
                    for mode in modes:
                        a = shared.estimate_from_y(mine, snr, N, n_summands_or_proba=mode)
                        b = own.estimate_from_y(mine, snr, N, n_summands_or_proba=mode)
                        c = shared.estimate_from_y(r[sl], snr, N, n_summands_or_proba=mode)        # host arrays: the library's copies
                        st.synchronize()
                        ref = serial[mode][sl]
                        for got, tol in ((a, 1e-6), (b, TOL_TC), (torch.from_numpy(c).cuda(), 1e-6)):
                            e = float((got - ref).norm() / ref.norm())
                            if not e < tol:
                                errors.append((i, rep, mode, e))
        except Exception as exc:                                  # noqa: BLE001 -- reported by the main thread
            errors.append((i, repr(exc)))

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:5]


def _tail_invariance(m, r, snr, N, modes, kw, tail=6000):
    """Estimates of rows at the start, across rows 2^20 and 2^21 and at the very end of one big call == the same rows in small calls."""
    B = r.shape[0]
    spots = [p for p in (0, (1 << 20) - tail // 2, (1 << 21) - tail // 2, (1 << 22) - tail // 2, B // 2 + 1, B - tail) if 0 <= p and p + tail <= B]
    for mode in modes:
        full = m.estimate_from_y(r, snr, N, n_summands_or_proba=mode, **kw)
        assert full.shape == (B, N)
        for p in spots:
            part = m.estimate_from_y(r[p:p + tail].contiguous(), snr, N, n_summands_or_proba=mode, **kw)
            err = float((full[p:p + tail] - part).norm() / part.norm())
            assert err < 1e-6, (mode, p, err)                  # FP32 atomics of the pair path: order-dependent in the last bits
        del full


@pytest.mark.gpu
def test_batches_beyond_4_gib_dense(qce):
    """Maximum sizes: one call whose pilot and estimate arrays exceed 4 GiB each (32-bit byte offsets would wrap at row 2^22 for
    N = 64, 2^21 for N = 128): the fused kernel, the chunked mode paths, the split path and the complex128 kernel index in 64 bits."""
    snr = 10
    # N = 64: 1 KiB per row -> 2^22 rows = 4 GiB; 5.2 M pilots
    K, N, B = 8, 64, (1 << 22) + (1 << 20) + 77
    means, covs, w = orc.random_psd_gmm(K, N, seed=3)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    r, _ = _grid_pilots(B, N, 2, 1 / np.sqrt(2), seed=1)
    assert r.numel() * 16 > (1 << 32)
    m.precision = 'tc'
    _tail_invariance(m, r, snr, N, ('all', 1, 3, 0.9), {})
    m.precision = 'fp64'
    _tail_invariance(m, r, snr, N, ('all',), {}, tail=2000)
    del r, m
    torch.cuda.empty_cache()
    # N = 128 split path, 2-bit uniform: 2 KiB per row
    K, N, B = 4, 128, (1 << 21) + 333
    means, covs, w = orc.random_psd_gmm(K, N, seed=4)
    qz = orc.get_quantizer([snr], 2, 'uniform')[snr]
    step = float(qz[1][1] - qz[1][0])
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    r, _ = _grid_pilots(B, N, 4, step / 2, seed=2)
    m.precision = 'tc'
    _tail_invariance(m, r, snr, N, ('all', 1, 2), dict(n_bits=2, quantizer_type='uniform', quantizer=qz))


@pytest.mark.gpu
def test_batches_beyond_4_gib_circulant(qce):
    """The same for the DFT-domain kernels (N = 256: 4 KiB per row -> 2^20 rows = 4 GiB)."""
    from quantized_channel_estimation_b200 import synthetic
    K, N, B, snr = 64, 256, (1 << 20) + (1 << 18) + 5, 10
    c, _, w, _ = synthetic.circulant_gmm(K, 16, 16, seed=2, dense=False)
    qz = orc.get_quantizer([snr], 3, 'lloyd')[snr]
    m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant').set_circulant_parameters(c, w, (16, 16))
    g = torch.Generator(device='cuda').manual_seed(3)
    r = torch.empty((B, N), dtype=torch.complex128, device='cuda')
    for i in range(0, B, 1 << 18):
        y = torch.view_as_complex(torch.randn((min(1 << 18, B - i), N, 2), generator=g, device='cuda', dtype=torch.float64)) * 0.8
        r[i:i + (1 << 18)] = qce.quant(y, 3, qz[0], qz[1])
    del y
    kw = dict(n_bits=3, quantizer_type='lloyd', quantizer=qz)
    _tail_invariance(m, r, snr, N, ('all', 1, 0.9), kw, tail=3000)


@pytest.mark.gpu
def test_host_arrays_beyond_4_gib(qce):
    """qce_estimate_host / qce_estimate_host_codes with host arrays past 4 GiB: chunk offsets are 64-bit, head / middle / tail rows equal
    the device path."""
    from quantized_channel_estimation_b200 import engine
    K, N, B, snr = 4, 64, (1 << 22) + 333, 10
    means, covs, w = orc.random_psd_gmm(K, N, seed=5)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    r, _ = _grid_pilots(B, N, 2, 1 / np.sqrt(2), seed=9)
    _, codes = engine.Quantizer.get(1).quantize(r, want_codes=True)
    r_host, codes_host = r.cpu().numpy(), codes.cpu().numpy()
    assert r_host.nbytes > (1 << 32)
    tail = 5000
    spots = (0, (1 << 21) - tail // 2, (1 << 22) - tail // 2, B - tail)
    for mode in ('all', 1):
        est = m.estimate_from_y(r_host, snr, N, n_summands_or_proba=mode)
        e64 = m.estimate_from_codes(codes_host, snr, N, n_summands_or_proba=mode)
        assert est.shape == (B, N) and e64.shape == (B, N)
        for p in spots:
            ref = m.estimate_from_y(r[p:p + tail].contiguous(), snr, N, n_summands_or_proba=mode).cpu().numpy()
            assert np.array_equal(est[p:p + tail], ref), (mode, p)
            assert np.array_equal(e64[p:p + tail], ref.astype(np.complex64)), (mode, p)
        del est, e64


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [torch.complex64, torch.complex128])
def test_pipeline_with_buffers_that_are_not_32_byte_aligned(qce, dtype):
    """Estimate rows and true-channel rows move with 256-bit accesses when the caller's buffers are 32-byte aligned; buffers that are
    not (a view one element into an allocation) take the 128-bit form: same NMSE accumulators."""
    from quantized_channel_estimation_b200 import engine, precompute
    K, N, B, snr = 8, 64, 5000, 10
    means, covs, w = orc.random_psd_gmm(K, N, seed=2)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=3)
    model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1, 'uniform', (None, None, None)))
    quant = engine.Quantizer.get(1)
    noise_t = torch.from_numpy(noise).cuda()
    h_al = torch.from_numpy(h).cuda().to(dtype).contiguous()
    buf = torch.empty(B * N + 1, dtype=dtype, device='cuda')
    h_off = buf[1:].view(B, N)
    h_off.copy_(h_al)
    assert h_al.data_ptr() % 32 == 0 and h_off.data_ptr() % 32 != 0
    accs = []
    for hh in (h_al, h_off):
        for mode in ('all', 1, 3):
            accs.append(model.pipeline(quant, hh, noise_t, 10 ** (-snr / 20), mode, 'tc').cpu().numpy())
    half = len(accs) // 2
    for a, b in zip(accs[:half], accs[half:]):
        assert a[2] == B and b[2] == B
        assert np.allclose(a, b, rtol=1e-6, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize('K,N,nb,qt,ms', [(16, 32, 1, 'uniform', 0.0), (64, 32, 1, 'uniform', 0.1), (8, 64, 1, 'uniform', 0.1), (16, 16, 2, 'uniform', 0.0),
                                         (12, 48, 1, 'uniform', 0.1), (16, 64, 3, 'uniform', 0.0)])
def test_tc_fused_hard_top1(qce, K, N, nb, qt, ms, monkeypatch):
    """Small shapes (N <= 32, or K <= 8; forced here for the others): top-1 runs as ONE fused launch with a running argmax in place of the online softmax; pilots
    whose two best components are too close to call are answered by the exact path (complex128 log-likelihoods, exact label, complex128
    estimate).  Same estimates as the complex128 kernel (no flipped selection), as the three-launch path (QCE_TC_HARD=0), with every
    pilot sent through the exact path (QCE_TC_TIE_EPS large), and the same NMSE accumulators in the fused pipeline."""
    from quantized_channel_estimation_b200 import _lib, engine, precompute
    import ctypes as C
    snr, B = 5, 40000 + 77
    means, covs, w, h, noise, qz, r = _case(K, N, B, snr, nb, qt, ms, seed=K + N)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    kw = dict(n_bits=nb, quantizer_type=qt, quantizer=qz)
    rt = torch.from_numpy(r).cuda()
    m.precision = 'fp64'
    ref = m.estimate_from_y(rt, snr, N, n_summands_or_proba=1, **kw)
    m.precision = 'tc'
    monkeypatch.setenv('QCE_TC_HARD', '1')
    got = m.estimate_from_y(rt, snr, N, n_summands_or_proba=1, **kw)
    rows = (got - ref).norm(dim=1) / ref.norm(dim=1).clamp(min=1e-300)
    assert float(rows.max()) < 1e-4, float(rows.max())                 # no flipped selection
    assert relerr(got.cpu().numpy(), ref.cpu().numpy()) < TOL_TC
    monkeypatch.setenv('QCE_TC_HARD', '0')
    three = m.estimate_from_y(rt, snr, N, n_summands_or_proba=1, **kw)
    monkeypatch.setenv('QCE_TC_HARD', '1')
    rows = (got - three).norm(dim=1) / three.norm(dim=1).clamp(min=1e-300)
    assert float(rows.max()) < 1e-5
    monkeypatch.setenv('QCE_TC_TIE_EPS', '1e6')                       # everybody is too close to call: the exact path answers the batch
    exact = m.estimate_from_y(rt[:3000].contiguous(), snr, N, n_summands_or_proba=1, **kw)
    monkeypatch.delenv('QCE_TC_TIE_EPS')
    assert relerr(exact.cpu().numpy(), ref[:3000].cpu().numpy()) < 1e-10
    # fused pipeline: NMSE accumulators of the hard launch + exact rows == those of the complex128 kernel
    if nb == 1:
        model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 1, 'uniform', (None, None, None)))
        quant = engine.Quantizer.get(1)
        ht, nt = torch.from_numpy(h).cuda(), torch.from_numpy(noise).cuda()
        a_tc = model.pipeline(quant, ht, nt, 10 ** (-snr / 20), 1, 'tc').cpu().numpy()
        a_64 = model.pipeline(quant, ht, nt, 10 ** (-snr / 20), 1, 'fp64').cpu().numpy()
        assert a_tc[2] == B and a_64[2] == B
        assert np.allclose(a_tc, a_64, rtol=1e-6)
