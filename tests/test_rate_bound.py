"""The achievable-rate lower bound in summable form: ``engine.RateModel.accumulate`` (qce_rate.cu) adds five sums per batch,
``utils.rate_from_accumulators`` turns them into the bound of ``utils.rate_lower_bound`` / ``orc.rate_lower_bound``
(Bussgang_GMM.py:291-309), ``utils.rate_params`` builds the scripts' ``(buss, Cq)`` and ``montecarlo.nmse_rate_sweep`` all-reduces
NMSE and rate sums together.  CPU tests use the numpy oracle; the kernel tests carry the ``gpu`` marker."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT
from oracle import qce_oracle as orc
from quantized_channel_estimation_b200 import utils
from quantized_channel_estimation_b200.montecarlo import nmse_rate_sweep, nmse_sweep

QUANTS = [(1, 'uniform'), (2, 'uniform'), (3, 'lloyd'), (np.inf, 'uniform')]


def moments(h_est, h, buss, cq):
    """The five sums in complex128 numpy, in the scripts' arithmetic (g = h_est / clip(|h_est|^2, 0.1))."""
    g = h_est / np.clip(np.sum(np.abs(h_est) ** 2, axis=1), 1e-1, np.inf)[:, None]
    inner = np.einsum('bi,ij,bj->b', g.conj(), buss, h)
    q = np.real(np.einsum('bi,ij,bj->b', g.conj(), cq, g))
    return np.array([inner.real.sum(), inner.imag.sum(), np.sum(np.abs(inner) ** 2), q.sum(), h.shape[0]]), g, inner


def oracle_params(C, snr, nb, qt, qz):
    """The construction test_gpu_parity.test_rate_lower_bound_vs_oracle restates, from the oracle's functions."""
    cy = C + 10 ** (-snr / 10) * np.eye(C.shape[0])
    if qt == 'lloyd':
        buss = orc.lloyd_get_bussgang_matrix(nb, cy, qz)
    else:
        buss = orc.uniform_get_bussgang_matrix(snr, nb, cy)
    return buss, orc.get_Cr(cy, nb, snr, qz) - buss @ C @ buss.conj().T


def case(N, B, snr, nb, qt, seed):
    """Global covariance of a random mixture, channels drawn from it, estimates = a shrunk noisy copy with a few rows scaled
    below the clip (|h_est|^2 < 0.1)."""
    means, covs, w = orc.random_psd_gmm(3, N, seed=seed)
    C = np.einsum('k,kij->ij', w, covs)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    h_est = 0.8 * h + 0.3 * orc.crandn(B, N, rng=rng)
    h_est[::7] *= 0.01
    qz = orc.get_quantizer([snr], nb, qt)[snr] if np.isfinite(nb) and nb > 1 else (None, None, None)
    return C, h, h_est, qz


# ----------------------------------------------------------------------------- CPU: host-side maths

def test_rate_from_accumulators_matches_oracle():
    rows = []
    for seed, (nb, qt), snr in zip(range(4), QUANTS, (-10, 0, 10, 30)):
        C, h, h_est, qz = case(16, 300, snr, nb, qt, seed)
        buss, cq = oracle_params(C, snr, nb, qt, qz)
        acc, _, _ = moments(h_est, h, buss, cq)
        ref = orc.rate_lower_bound(h_est, h, buss, cq)
        assert abs(utils.rate_from_accumulators(acc) - ref) < 1e-12 * max(1.0, abs(ref))
        assert abs(utils.rate_from_accumulators(torch.from_numpy(acc)) - ref) < 1e-12 * max(1.0, abs(ref))
        rows.append((acc, ref))
    rates = utils.rate_from_accumulators(np.stack([a for a, _ in rows]))        # [n_snr, 5] -> [n_snr]
    assert rates.shape == (4,)
    np.testing.assert_allclose(rates, [r for _, r in rows], rtol=1e-12)


@pytest.mark.parametrize('nb,qt', QUANTS)
def test_rate_params_reproduces_the_scripts_construction(nb, qt):
    N, snr = 12, 5
    C, _, _, qz = case(N, 10, snr, nb, qt, seed=7)
    buss, cq = utils.rate_params(C, snr, nb, qt, qz)
    rb, rq = oracle_params(C, snr, nb, qt, qz)
    assert buss.shape == cq.shape == (N, N)
    assert np.count_nonzero(buss - np.diag(np.diag(buss))) == 0
    np.testing.assert_allclose(buss, rb, rtol=1e-12, atol=0)
    np.testing.assert_allclose(cq, rq, rtol=1e-12, atol=1e-14)
    if np.isfinite(nb) and nb > 1:       # the table is looked up when omitted
        b2, q2 = utils.rate_params(C, snr, nb, qt)
        np.testing.assert_allclose(b2, rb, rtol=1e-8)
        np.testing.assert_allclose(q2, rq, rtol=1e-8, atol=1e-10)


SW_SNRS = [-5, 10]
SW_K, SW_N, SW_B = 4, 8, 101


def _sweep_step():
    means, covs, w = orc.random_psd_gmm(SW_K, SW_N, seed=2)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, SW_B, seed=3)
    C = np.einsum('k,kij->ij', w, covs)

    def step(i, snr, lo, hi):
        r = orc.get_observation_nbit(h[lo:hi], snr, noise[lo:hi], None, 1)
        est = orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=1)
        buss, cq = oracle_params(C, snr, 1, 'uniform', None)
        acc, _, _ = moments(est, h[lo:hi], buss, cq)
        return (np.sum(np.abs(est - h[lo:hi]) ** 2), np.sum(np.abs(h[lo:hi]) ** 2), hi - lo) + tuple(acc)
    return step


def _sweep_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    nmse, rate, acc = nmse_rate_sweep(_sweep_step(), SW_B, SW_SNRS, SW_N)
    q.put((rank, nmse, rate, acc.numpy()))
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_rate_sweep_matches_single_process():
    nmse1, rate1, acc1 = nmse_rate_sweep(_sweep_step(), SW_B, SW_SNRS, SW_N)
    assert acc1.shape == (len(SW_SNRS), 8) and np.all(acc1[:, 7].numpy() == SW_B)
    nmse0, _ = nmse_sweep(lambda *a: _sweep_step()(*a)[:3], SW_B, SW_SNRS, SW_N)
    np.testing.assert_allclose(nmse1, nmse0, rtol=1e-12)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 1000) % 2000
    procs = [ctx.Process(target=_sweep_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, nmse, rate, acc in res:
        np.testing.assert_allclose(nmse, nmse1, rtol=1e-12)
        np.testing.assert_allclose(rate, rate1, rtol=1e-12)
        np.testing.assert_allclose(acc, acc1.numpy(), rtol=1e-12)


# ----------------------------------------------------------------------------- GPU: the kernel

@pytest.fixture(scope='module')
def qce():
    import quantized_channel_estimation_b200 as q
    from quantized_channel_estimation_b200 import _lib
    _lib.require_device()
    return q


def _check_acc(acc, ref, g, cq, n):
    acc = acc.cpu().numpy() if isinstance(acc, torch.Tensor) else acc
    sc1 = max(abs(ref[0]) + abs(ref[1]), 1e-300)
    assert abs(acc[0] - ref[0]) <= 1e-12 * sc1 and abs(acc[1] - ref[1]) <= 1e-12 * sc1
    assert abs(acc[2] - ref[2]) <= 1e-12 * abs(ref[2])
    assert acc[4] == n
    qtol = 1e-5 * np.sum(np.abs(g) ** 2) * np.linalg.norm(cq, 2)
    assert abs(acc[3] - ref[3]) <= qtol, (acc[3], ref[3], qtol)


@pytest.mark.gpu
@pytest.mark.parametrize('N', [8, 16, 50, 64, 128, 200, 256])
@pytest.mark.parametrize('nb,qt', QUANTS)
@pytest.mark.parametrize('snr', [-10, 10, 30])
def test_accumulate_vs_complex128_moments(qce, N, nb, qt, snr):
    from quantized_channel_estimation_b200 import engine
    C, h, h_est, qz = case(N, 4097, snr, nb, qt, seed=100 + N + int(snr))
    buss, cq = utils.rate_params(C, snr, nb, qt, qz)
    model = engine.RateModel(buss, cq)
    for B in (1, 31, 4097):
        for dt in (torch.complex64, torch.complex128):
            ht = torch.from_numpy(h[:B]).to(dt).cuda()
            hr = ht.cpu().numpy().astype(np.complex128)     # the values the kernel reads (c64 channels rounded)
            ref, g, _ = moments(h_est[:B], hr, buss, cq)
            acc = model.accumulate(torch.from_numpy(h_est[:B]).cuda(), ht)
            _check_acc(acc, ref, g, cq, B)
            if B > 1:                                       # (one row has no variance; the oracle's squeeze needs B > 1)
                assert abs(utils.rate_from_accumulators(acc) - orc.rate_lower_bound(h_est[:B], hr, buss, cq)) < 2e-5, (B, dt)


@pytest.mark.gpu
def test_end_to_end_gmm_tensor_core_estimates(qce):
    """Config-2 shape: GMM 'full', N = K = 64, 1 bit, 2^16 pilots, tensor-core estimates."""
    from quantized_channel_estimation_b200 import engine
    K, N, B, snr = 64, 64, 1 << 16, 10
    means, covs, w = orc.random_psd_gmm(K, N, seed=5)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=6)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, detect_structure=False)
    r = qce.get_observation_nbit(torch.from_numpy(h).cuda(), snr, n_bits=1, noise=torch.from_numpy(noise).cuda())
    est = m.estimate_from_y(r, snr, N, n_summands_or_proba='all')
    buss, cq = utils.rate_params(np.einsum('k,kij->ij', w, covs), snr, 1)
    acc = engine.RateModel(buss, cq).accumulate(est, torch.from_numpy(h).cuda())
    assert abs(utils.rate_from_accumulators(acc) - utils.rate_lower_bound(est, h, buss, cq)) < 2e-5


@pytest.mark.gpu
def test_end_to_end_circulant_n256(qce):
    """Block-circulant 16 x 16 (N = 256), 3-bit Lloyd-Max, CircModel estimates."""
    from quantized_channel_estimation_b200 import engine, synthetic
    K, B, snr = 64, 4096, 10
    c, covs, w, _ = synthetic.circulant_gmm(K, 16, 16, seed=1)
    h, noise, _ = orc.sample_gmm_channels(np.zeros((K, 256), complex), covs, w, B, seed=2)
    qz = qce.get_quantizer([snr], 3, 'lloyd')[snr]
    m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant')
    m.set_circulant_parameters(c, w, (16, 16))
    r = qce.get_observation_nbit(torch.from_numpy(h).cuda(), snr, n_bits=3, thresholds=qz[0], cluster=qz[1],
                                 noise=torch.from_numpy(noise).cuda())
    est = m.estimate_from_y(r, snr, 256, n_summands_or_proba='all', n_bits=3, quantizer_type='lloyd', quantizer=qz)
    assert isinstance(m._last, engine.CircModel)
    buss, cq = utils.rate_params(np.einsum('k,kij->ij', w, covs), snr, 3, 'lloyd', qz)
    acc = engine.RateModel(buss, cq).accumulate(est, torch.from_numpy(h).cuda())
    assert abs(utils.rate_from_accumulators(acc) - utils.rate_lower_bound(est, h, buss, cq)) < 2e-5


@pytest.mark.gpu
def test_in_process_pipeline_sweep(qce):
    """pipeline(want_est=True) + accumulate per chunk and SNR through nmse_rate_sweep equals the torch bound of the concatenated
    estimates, and the NMSE the sweep reports."""
    from quantized_channel_estimation_b200 import engine
    K, N, B, chunk, snrs = 16, 64, 3000, 1024, [-5, 10]
    means, covs, w = orc.random_psd_gmm(K, N, seed=11)
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, B, seed=12)
    m = qce.Gmm_nbit(n_components=K).set_parameters(means, covs, w, zero_mean=True, detect_structure=False)
    C = np.einsum('k,kij->ij', w, covs)
    ht, nt = torch.from_numpy(h).to(torch.complex64).cuda(), torch.from_numpy(noise).cuda()
    quant = engine.Quantizer.get(1)
    ests = {}

    def step(i, snr, lo, hi):
        dm = m._prepared(np.eye(N, dtype=complex), snr, 1, 'uniform', None)
        rm = engine.RateModel(*utils.rate_params(C, snr, 1))
        acc = torch.zeros(8, dtype=torch.float64, device='cuda')
        parts = []
        for a in range(lo, hi, chunk):
            b = min(hi, a + chunk)
            est, _ = dm.pipeline(quant, ht[a:b], nt[a:b], 10 ** (-snr / 20), 'all', 'auto', want_est=True, acc=acc[:3])
            rm.accumulate(est, ht[a:b], acc=acc[3:])
            parts.append(est)
        ests[i] = torch.cat(parts)
        return acc
    nmse, rate, acc = nmse_rate_sweep(step, B, snrs, N, device='cuda')
    for i, snr in enumerate(snrs):
        buss, cq = utils.rate_params(C, snr, 1)
        assert abs(rate[i] - utils.rate_lower_bound(ests[i], ht, buss, cq)) < 2e-5
        assert abs(nmse[i] - utils.mse(ests[i], ht)) < 1e-6 * nmse[i]
        assert acc[i, 7].item() == B


@pytest.mark.gpu
def test_chunks_add_up(qce):
    from quantized_channel_estimation_b200 import engine
    C, h, h_est, qz = case(64, 3000, 10, 2, 'uniform', seed=21)
    model = engine.RateModel(*utils.rate_params(C, 10, 2, 'uniform', qz))
    he, ht = torch.from_numpy(h_est).cuda(), torch.from_numpy(h).cuda()
    one = model.accumulate(he, ht).cpu().numpy()
    acc = torch.zeros(5, dtype=torch.float64, device='cuda')
    for a, b in ((0, 1000), (1000, 1001), (1001, 3000)):
        out = model.accumulate(he[a:b], ht[a:b], acc=acc)
        assert out is acc
    three = acc.cpu().numpy()
    np.testing.assert_allclose(three[:3], one[:3], rtol=1e-12)
    assert abs(three[3] - one[3]) <= 1e-6 * abs(one[3])
    assert three[4] == one[4] == 3000


@pytest.mark.gpu
def test_edge_cases(qce):
    from quantized_channel_estimation_b200 import _lib, engine
    N = 50
    C, h, h_est, qz = case(N, 200, 0, 1, 'uniform', seed=3)
    buss, cq = utils.rate_params(C, 0, 1)
    model = engine.RateModel(buss, cq)
    ht = torch.from_numpy(h).cuda()
    # B = 0: nothing enqueued, acc untouched
    acc = torch.arange(5, dtype=torch.float64, device='cuda')
    n0 = _lib.launch_count()
    model.accumulate(torch.zeros((0, N), dtype=torch.complex128, device='cuda'), ht[:0], acc=acc)
    assert _lib.launch_count() == n0
    assert torch.equal(acc, torch.arange(5, dtype=torch.float64, device='cuda'))
    # all-zero estimate rows contribute nothing but their count
    z = model.accumulate(torch.zeros((77, N), dtype=torch.complex128, device='cuda'), ht[:77]).cpu().numpy()
    assert np.array_equal(z, [0, 0, 0, 0, 77])
    # rows below the clip (|h_est|^2 < 0.1) are divided by 0.1, as the scripts do
    small = 0.02 * h_est / np.linalg.norm(h_est, axis=1, keepdims=True)
    ref, g, _ = moments(small, h, buss, cq)
    assert np.all(np.sum(np.abs(small) ** 2, axis=1) < 0.1)
    _check_acc(model.accumulate(torch.from_numpy(small).cuda(), ht), ref, g, cq, 200)
    # argument checks
    with pytest.raises(ValueError):
        engine.RateModel(buss + 1e-3 * np.eye(N, k=1), cq)
    big = np.eye(257, dtype=complex)
    with pytest.raises(_lib.QceError) as ei:
        engine.RateModel(big, big)
    assert ei.value.status == _lib.ERR_UNSUPPORTED
    with pytest.raises(TypeError):
        model.accumulate(torch.from_numpy(h_est), ht)
    with pytest.raises(TypeError):
        model.accumulate(torch.from_numpy(h_est).cuda(), torch.from_numpy(h))
    with pytest.raises(ValueError):
        model.accumulate(torch.from_numpy(h_est[:, :40]).cuda(), ht[:, :40])


@pytest.mark.gpu
def test_large_batch_64bit_indexing(qce):
    """B * N * 2 > 2^31 doubles in one call: exact count, S1 against chunked torch moments."""
    from quantized_channel_estimation_b200 import engine
    N, B = 64, (1 << 24) + 5
    C, _, _, _ = case(N, 2, 10, 1, 'uniform', seed=4)
    buss, cq = utils.rate_params(C, 10, 1)
    model = engine.RateModel(buss, cq)
    gen = torch.Generator(device='cuda').manual_seed(0)
    ht = torch.view_as_complex(torch.randn((B, N, 2), generator=gen, device='cuda', dtype=torch.float32)) * np.sqrt(0.5)
    he = (ht.to(torch.complex128) * 0.7 + torch.view_as_complex(torch.randn((B, N, 2), generator=gen, device='cuda',
                                                                             dtype=torch.float64)) * 0.2)
    acc = model.accumulate(he, ht).cpu().numpy()
    assert acc[4] == B
    bd = torch.from_numpy(np.diag(buss).copy()).cuda()
    s1 = torch.zeros((), dtype=torch.complex128, device='cuda')
    for a in range(0, B, 1 << 22):
        e, t = he[a:a + (1 << 22)], ht[a:a + (1 << 22)].to(torch.complex128)
        g = e / (e.abs() ** 2).sum(dim=1).clamp(min=0.1)[:, None]
        s1 += (g.conj() * t * bd).sum()
    s1 = complex(s1.item())
    assert abs(complex(acc[0], acc[1]) - s1) <= 1e-11 * abs(s1)
