"""Every estimate route over the whole combination-mode domain, and mixtures with zero-weight components.

The route table below names each kernel instantiation the library picks from the model shape, the precision, the batch size
and the launch-time knobs (``QCE_TC_PAIRS`` / ``QCE_TC_BUCKET`` / ``QCE_TC_HARD`` are read per call).  Every route runs in
every combination mode of ``mode_domain(K)`` -- 'all', top-1, top-n below, at and above K, cumulative rho below 0, at 0, inside
(0, 1), at 1, above 1 and infinite -- against the numpy oracle in complex128, evaluated on a strided subset of the batch plus every
row of the last (ragged) tile; the kernel always runs the whole batch.  Checked per route and mode: finite outputs, global and
per-row relative error (no per-row exemption: a flipped selection fails), the NMSE accumulators, and the log-probability export.

Zero-weight components (``w_k = 0``, ``logc_k = -inf``; the reference gives them responsibility 0 and finite estimates) run on
every route in every mode, and splitting one component into two identical halves must not change the 'all' estimate.

The CPU tests check the route predicates (mirrors of the dispatch thresholds in csrc/) and the row selection."""
import ctypes as C

import numpy as np
import pytest
from scipy.special import logsumexp

from conftest import relerr
from oracle import qce_oracle as orc

TOL = {'fp64': (1e-10, 1e-8), 'tc': (1e-5, 1e-4)}      # (global relative error, per-row relative error)

# dispatch constants of csrc/ that decide a route
TC_PAIR_CAP = 4              # qce_dense_tc.cu: top-n with n <= 4 is a pair mode
TC_TILE = 128                # TILE_M: pilots per tensor-core tile
TC_UNIT = 4 * TC_TILE        # work unit of the mode path
CIRC_TC_TILE = 32            # CT_P: pilots per CTA of circ_tc_kernel
N_SMS = 148


# ----------------------------------------------------------------------------------------------------- route predicates (CPU)

def fp64_dense_ts(B):
    """Tile size of dense_fp64_kernel and mfa_kernel (qce_dense_fp64.cu / qce_mfa.cu launch): 8 / 16 / 32."""
    return 32 if B >= 32 * N_SMS else 16 if B >= 16 * 64 else 8


def circ_ts(B):
    """Tile size of circ_kernel (qce_circ.cu launch): 4 / 8 / 16."""
    return 16 if B >= 16 * N_SMS else 8 if B >= 8 * 64 else 4


def tc_split(n_obs):
    """Dense tensor-core models with n_obs > 64 run whitening / selection / LMMSE row-block launches (the split path)."""
    return n_obs > 64


def tc_mode_chunk(B, K, pairs=False):
    chunk = max(((1 << 27) // K) // TC_UNIT * TC_UNIT, TC_UNIT)
    if pairs:
        chunk = min(chunk, 1 << 19)
    return min(chunk, B)


def tc_pairs(B, K, n_obs, mode, env=None):
    """tc_run_modes: the pair-bucketed combination (the device may still fall back to the dense weighted launch)."""
    pair_on = tc_split(n_obs) if env is None else bool(env)
    if isinstance(mode, str):
        ok = tc_split(n_obs)
    elif isinstance(mode, int):
        ok = mode != 1 and mode <= TC_PAIR_CAP
    else:
        ok = True
    return pair_on and ok and K >= 8 and B >= 16 * TC_UNIT


def tc_bucket_rows(n_obs, off_grid):
    tiles_per_unit = 2 * (1 if ((off_grid and 2 * n_obs > 128) or 2 * n_obs > 256) else 2)
    return tiles_per_unit * TC_TILE


def tc_bucketed_top1(B, K, n_obs, off_grid, env=None):
    """tc_run_modes: top-1 regrouped by label, one component per work unit (QCE_TC_BUCKET=0 turns it off)."""
    on = env is None or bool(env)
    return on and K >= 4 and tc_mode_chunk(B, K) >= 4 * tc_bucket_rows(n_obs, off_grid)


def tc_hard_top1(n_obs, K, off_grid):
    """tc_hard_top1_ok: the fused running-argmax launch (small shapes, on-grid, not split)."""
    return not tc_split(n_obs) and not off_grid and (n_obs <= 32 or K <= 8)


def mode_domain(K):
    """'all', top-1, top-n for n in {2, 4, 5, K-1, K, K+3}, cumulative rho in {-1, 0, 0.5, 0.999, 1, 1.5, inf}."""
    tops = []
    for n in (2, 4, 5, K - 1, K, K + 3):
        if n >= 2 and n not in tops:
            tops.append(int(n))
    return ['all', 1] + tops + [-1.0, 0.0, 0.5, 0.999, 1.0, 1.5, float('inf')]


def check_rows(B, tile, n_max=1500):
    """Rows the oracle evaluates: a strided subset of at most ~n_max rows before the last tile, plus every row of the last tile."""
    last0 = ((B - 1) // tile) * tile
    stride = max(1, -(-last0 // n_max))
    return np.union1d(np.arange(0, last0, stride), np.arange(last0, B)).astype(np.int64)


def zero_weight_variants(K):
    """Indices whose weight is set to exactly 0: the first, a middle and the last component, and two at once."""
    return {'first': [0], 'middle': [K // 2], 'last': [K - 1], 'two': [1, K - 2]}


# ----------------------------------------------------------------------------------------------------- route table

ROUTES = {
    # complex128 dense kernel: N = 48, K = 12, 2-bit uniform with means; TS = 8 / 16 / 32
    'dense_fp64_ts8': dict(kind='gmm', K=12, N=48, nb=2, qt='uniform', ms=0.1, snr=10, B=301, prec='fp64', ts=8),
    'dense_fp64_ts16': dict(kind='gmm', K=12, N=48, nb=2, qt='uniform', ms=0.1, snr=10, B=2003, prec='fp64', ts=16),
    'dense_fp64_ts32': dict(kind='gmm', K=12, N=48, nb=2, qt='uniform', ms=0.1, snr=10, B=6001, prec='fp64', ts=32),
    # tensor cores, fused shape (N = K = 64, 1 bit): fused 'all', bucketed top-1, weighted launches for the other modes
    'tc_fused': dict(kind='gmm', K=64, N=64, nb=1, qt='uniform', ms=0.0, snr=10, B=3001, prec='tc', tc='fused', n_max=600),
    'tc_fused_bucket_off': dict(kind='gmm', K=64, N=64, nb=1, qt='uniform', ms=0.0, snr=10, B=3001, prec='tc', tc='fused', n_max=600,
                                env={'QCE_TC_BUCKET': '0'}),
    # fused hard top-1 (N <= 32)
    'tc_hard_top1': dict(kind='gmm', K=16, N=32, nb=1, qt='uniform', ms=0.1, snr=5, B=1501, prec='tc', tc='hard'),
    # split path (N = 128, K = 16, 2-bit uniform): pairs on (B >= 8192), pairs off, flat posterior (device-side fallback)
    'tc_split_pairs': dict(kind='gmm', K=16, N=128, nb=2, qt='uniform', ms=0.0, snr=10, B=8300, prec='tc', tc='split',
                           n_max=1000),
    'tc_split_pairs_off': dict(kind='gmm', K=16, N=128, nb=2, qt='uniform', ms=0.0, snr=10, B=8300, prec='tc', tc='split',
                               env={'QCE_TC_PAIRS': '0'}, n_max=1000),
    'tc_split_flat': dict(kind='gmm', K=16, N=128, nb=2, qt='uniform', ms=0.0, snr=-10, B=8300, prec='tc', tc='split',
                          n_max=1000),
    # three-pass off-grid path (3-bit Lloyd-Max labels as FP16 (hi, lo) tile pairs)
    'tc_three_pass': dict(kind='gmm', K=12, N=48, nb=3, qt='lloyd', ms=0.1, snr=10, B=1101, prec='tc', tc='three_pass'),
    # complex128 circulant kernel, 8 x 8 blocks: TS = 4 / 8 / 16
    'circ_fp64_ts4': dict(kind='circ', K=16, blocks=(8, 8), nb=2, qt='uniform', snr=8, B=301, prec='fp64', ts=4),
    'circ_fp64_ts8': dict(kind='circ', K=16, blocks=(8, 8), nb=2, qt='uniform', snr=8, B=1001, prec='fp64', ts=8),
    'circ_fp64_ts16': dict(kind='circ', K=16, blocks=(8, 8), nb=2, qt='uniform', snr=8, B=2501, prec='fp64', ts=16),
    # circulant tensor-core kernel (16 x 16 blocks, K = 64)
    'circ_tc': dict(kind='circ', K=64, blocks=(16, 16), nb=3, qt='lloyd', snr=8, B=611, prec='tc', n_max=300),
    # MFA Woodbury kernel (N = 64, latent 8, 3-bit Lloyd-Max): TS = 8 / 16 / 32
    'mfa_ts8': dict(kind='mfa', K=8, N=64, M=8, nb=3, qt='lloyd', ms=0.1, snr=9, B=301, prec='fp64', ts=8),
    'mfa_ts16': dict(kind='mfa', K=8, N=64, M=8, nb=3, qt='lloyd', ms=0.1, snr=9, B=2003, prec='fp64', ts=16),
    'mfa_ts32': dict(kind='mfa', K=8, N=64, M=8, nb=3, qt='lloyd', ms=0.1, snr=9, B=6001, prec='fp64', ts=32),
}


def route_tile(rt):
    """The tile whose rows are all checked: the kernel's tile (complex128), the mode path's work unit (dense tensor cores)."""
    if rt['prec'] == 'fp64':
        return rt['ts']
    return CIRC_TC_TILE if rt['kind'] == 'circ' else TC_UNIT


def route_n_obs(rt):
    return rt['blocks'][0] * rt['blocks'][1] if rt['kind'] == 'circ' else rt['N']


def route_reaches(name):
    """The kernel instantiation a route reaches, from the dispatch predicates."""
    rt = ROUTES[name]
    B, K, n = rt['B'], rt['K'], route_n_obs(rt)
    if rt['kind'] == 'gmm' and rt['prec'] == 'fp64':
        return f'dense_fp64_kernel<{fp64_dense_ts(B)}>'
    if rt['kind'] == 'mfa':
        return f'mfa_kernel<{fp64_dense_ts(B)}>'
    if rt['kind'] == 'circ':
        return f'circ_kernel<{circ_ts(B)}>' if rt['prec'] == 'fp64' else 'circ_tc_kernel<K=64>'
    return f"dense_tc_kernel {rt['tc']} (n_obs={n}, K={K})"


# ----------------------------------------------------------------------------------------------------- oracle

def oracle_eval(kind, params, y, snr, nb, qt, qz):
    """The oracle's pieces on rows ``y``: weighted log-probabilities [B, K], responsibilities, per-component LMMSE estimates and
    the top-1 labels, composed exactly like ``orc.gmm_estimate_from_y`` / ``orc.mofa_estimate_from_y``."""
    means, covs, w = params['means'], params['covs'], params['w']
    A = np.eye(means.shape[1], dtype=complex)
    with np.errstate(divide='ignore'):
        if kind == 'mfa':
            prep = orc.mofa_prepare(means, covs, A, snr, nb, qt, qz)
            logrs = orc.mofa_log_resp_unnorm(y, prep, w)
            proba = np.exp(logrs - orc._log_sum(logrs)[None, :]).T
            wlp, labels = logrs.T, np.exp(logrs).argmax(axis=0)
        else:
            prep = orc.gmm_prepare(means, covs, A, snr, nb, qt, qz)
            wlp = orc.gmm_weighted_log_prob(y, prep, w)
            proba = np.exp(wlp - logsumexp(wlp, axis=1)[:, None])
            labels = wlp.argmax(axis=1)
    hk = orc._component_lmmse(y, means, covs, prep)
    return dict(wlp=wlp, proba=proba, hk=hk, labels=labels)


def oracle_mode(o, mode):
    return orc._combine(o['proba'], o['hk'], mode, lambda: o['labels'])


def pairs_per_pilot(o, mode):
    """Average number of (pilot, component) pairs with a renormalised weight above 1e-9 (the pair threshold) under ``mode``."""
    p = o['proba']
    if isinstance(mode, str):
        w = p
    else:
        w = np.zeros_like(p)
        for b in range(p.shape[0]):
            idx = np.argsort(p[b])[::-1]
            n = mode if isinstance(mode, int) else np.searchsorted(np.cumsum(p[b, idx]), mode) + 1
            idx = idx[:n]
            w[b, idx] = p[b, idx] / p[b, idx].sum()
    return float((w > 1e-9).sum(1).mean())


# ----------------------------------------------------------------------------------------------------- CPU tests

def test_mode_domain_covers_every_selection_edge():
    K = 16
    d = mode_domain(K)
    assert d[:2] == ['all', 1]
    tops = [m for m in d if isinstance(m, int) and m > 1]
    assert tops == [2, 4, 5, 15, 16, 19]
    assert any(n <= TC_PAIR_CAP for n in tops) and any(n == TC_PAIR_CAP + 1 for n in tops)      # both sides of the pair cap
    assert any(n > K for n in tops)                                                            # limit = min(n_top, K)
    rhos = [m for m in d if isinstance(m, float)]
    assert min(rhos) < 0 and 0.0 in rhos and 1.0 in rhos and max(rhos) == float('inf')
    from quantized_channel_estimation_b200 import _lib, engine
    assert [engine.parse_mode(m)[0] for m in d] == [_lib.MODE_ALL, _lib.MODE_TOP1] + [_lib.MODE_TOPN] * 6 + [_lib.MODE_CUMPROB] * 7
    assert mode_domain(4) == ['all', 1, 2, 4, 5, 3, 7, -1.0, 0.0, 0.5, 0.999, 1.0, 1.5, float('inf')]


@pytest.mark.parametrize('B,tile', [(301, 8), (2003, 16), (6001, 32), (3001, 512), (2048, 512), (611, 32), (7, 8)])
def test_check_rows_subset_and_tail(B, tile):
    rows = check_rows(B, tile)
    last0 = ((B - 1) // tile) * tile
    assert rows[0] == 0 and rows[-1] == B - 1
    assert np.all(np.diff(rows) > 0)
    assert set(range(last0, B)) <= set(rows.tolist())
    assert len(rows) <= 1500 + tile + 1
    assert 0 < B - last0 <= tile


def test_route_table_reaches_every_instantiation():
    """Each route of the table sits on the side of every dispatch threshold it claims."""
    reached = {name: route_reaches(name) for name in ROUTES}
    for ts in (8, 16, 32):
        assert f'dense_fp64_kernel<{ts}>' in reached.values() and f'mfa_kernel<{ts}>' in reached.values()
    for ts in (4, 8, 16):
        assert f'circ_kernel<{ts}>' in reached.values()
    assert fp64_dense_ts(1023) == 8 and fp64_dense_ts(1024) == 16 and fp64_dense_ts(4735) == 16 and fp64_dense_ts(4736) == 32
    assert circ_ts(511) == 4 and circ_ts(512) == 8 and circ_ts(2367) == 8 and circ_ts(2368) == 16
    for name, rt in ROUTES.items():
        if rt['prec'] == 'fp64':
            assert (circ_ts if rt['kind'] == 'circ' else fp64_dense_ts)(rt['B']) == rt['ts'], name
            assert rt['B'] % rt['ts'] != 0, name                                   # ragged last tile
        else:
            assert rt['B'] % route_tile(rt) != 0, name
    f = ROUTES['tc_fused']
    assert not tc_split(f['N']) and tc_bucketed_top1(f['B'], f['K'], f['N'], False)
    assert not tc_bucketed_top1(f['B'], f['K'], f['N'], False, env=0)
    assert not tc_hard_top1(f['N'], f['K'], False)
    assert not any(tc_pairs(f['B'], f['K'], f['N'], m) for m in mode_domain(f['K']))
    h = ROUTES['tc_hard_top1']
    assert tc_hard_top1(h['N'], h['K'], False) and not tc_bucketed_top1(h['B'], h['K'], h['N'], False)
    for name in ('tc_split_pairs', 'tc_split_flat'):
        s = ROUTES[name]
        assert tc_split(s['N']) and s['B'] >= 16 * TC_UNIT
        assert tc_pairs(s['B'], s['K'], s['N'], 'all') and tc_pairs(s['B'], s['K'], s['N'], 4) and tc_pairs(s['B'], s['K'], s['N'], 0.5)
        assert not tc_pairs(s['B'], s['K'], s['N'], 5) and not tc_pairs(s['B'], s['K'], s['N'], 1)
    s = ROUTES['tc_split_pairs_off']
    assert not any(tc_pairs(s['B'], s['K'], s['N'], m, env=0) for m in mode_domain(s['K']))
    t = ROUTES['tc_three_pass']
    assert t['qt'] == 'lloyd' and not tc_hard_top1(t['N'], t['K'], True)
    from quantized_channel_estimation_b200 import engine
    for name, rt in ROUTES.items():
        if rt['kind'] == 'gmm' and rt['prec'] == 'tc':
            assert engine.tc_shape_ok(rt['N'], rt['N'], on_grid=rt['qt'] == 'uniform'), name


def test_oracle_pieces_compose_to_the_oracle():
    """oracle_eval / oracle_mode reproduce orc.gmm_estimate_from_y and orc.mofa_estimate_from_y in every mode, with and without a
    zero-weight component (whose log-probability is -inf and whose responsibility is 0)."""
    K, N, snr = 5, 8, 5
    means, covs, w = orc.random_psd_gmm(K, N, seed=1, mean_scale=0.2)
    qz = orc.get_quantizer([snr], 2, 'uniform')[snr]
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, 40, seed=2)
    r = orc.get_observation_nbit(h, snr, noise, None, 2, qz[0], qz[1])
    mm, lam, psi, amps = orc.random_mfa(K, N, 2, seed=3, mean_scale=0.1)
    for kind, params in (('gmm', dict(means=means, covs=covs, w=w)), ('mfa', dict(means=mm, covs=orc.mofa_covs(lam, psi), w=amps))):
        for zero in ([], [2]):
            p = dict(params)
            p['w'] = params['w'].copy()
            p['w'][zero] = 0.0
            o = oracle_eval(kind, p, r, snr, 2, 'uniform', qz)
            fn = orc.mofa_estimate_from_y if kind == 'mfa' else orc.gmm_estimate_from_y
            for mode in mode_domain(K):
                with np.errstate(divide='ignore'):
                    ref = fn(p['means'], p['covs'], p['w'], r, snr, n_summands_or_proba=mode, n_bits=2, quantizer_type='uniform', quantizer=qz)
                got = oracle_mode(o, mode)
                assert np.isfinite(got).all() and np.array_equal(got, ref), (kind, zero, mode)
            if zero:
                assert np.isneginf(o['wlp'][:, zero]).all() and (o['proba'][:, zero] == 0).all()


def test_zero_weight_variants_and_pair_counts():
    assert zero_weight_variants(12) == {'first': [0], 'middle': [6], 'last': [11], 'two': [1, 10]}
    o = dict(proba=np.array([[0.7, 0.2, 0.1, 0.0], [0.25, 0.25, 0.25, 0.25]]))
    assert pairs_per_pilot(o, 'all') == 3.5
    assert pairs_per_pilot(o, 2) == 2.0
    assert pairs_per_pilot(o, 0.8) == (2 + 4) / 2


# ----------------------------------------------------------------------------------------------------- GPU side

@pytest.fixture(scope='module')
def qce():
    import quantized_channel_estimation_b200 as q
    from quantized_channel_estimation_b200 import _lib
    _lib.require_device()
    return q


_DATA = {}


def route_data(name):
    """Model parameters, pilots and channels of a route (seeded; built once per module)."""
    if name in _DATA:
        return _DATA[name]
    rt = ROUTES[name]
    K, snr, nb, qt, B = rt['K'], rt['snr'], rt['nb'], rt['qt'], rt['B']
    seed = sum(map(ord, name.split('_ts')[0].replace('_off', '').replace('_flat', '')))
    if rt['kind'] == 'gmm':
        means, covs, w = orc.random_psd_gmm(K, rt['N'], seed=seed, mean_scale=rt['ms'])
        params = dict(means=means, covs=covs, w=w)
    elif rt['kind'] == 'mfa':
        means, lam, psi, amps = orc.random_mfa(K, rt['N'], rt['M'], seed=seed, mean_scale=rt['ms'])
        params = dict(means=means, covs=orc.mofa_covs(lam, psi), w=amps, lam=lam, psi=psi)
    else:
        c, covs, w, _ = orc.circulant_gmm(K, *rt['blocks'], seed=seed)
        params = dict(means=np.zeros((K, c.shape[1]), dtype=complex), covs=covs, w=w, c=c)
    h, noise, _ = orc.sample_gmm_channels(params['means'], params['covs'], params['w'], B, seed=seed + 1)
    qz = orc.get_quantizer([snr], nb, qt)[snr]
    r = orc.get_observation_nbit(h, snr, noise, None, nb, qz[0], qz[1])
    rows = check_rows(B, route_tile(rt), rt.get('n_max', 1500))
    _DATA[name] = d = dict(params=params, h=h, r=r, qz=qz, rows=rows)
    return d


def with_weights(params, w):
    p = dict(params)
    p['w'] = np.asarray(w, dtype=float)
    return p


def split_component(kind, params, j):
    """The same mixture with component j split into two identical components of half its weight (appended last)."""
    p = dict(params)
    dup = lambda a: np.concatenate([a, a[j:j + 1]], axis=0)
    for key in ('means', 'covs', 'lam', 'psi', 'c'):
        if key in p:
            p[key] = dup(p[key])
    w = p['w'].copy()
    w[j] *= 0.5
    p['w'] = np.append(w, w[j])
    return p


def engine_model(qce, name, params):
    """The library model the high-level API prepares for this route and these parameters, and its expected type."""
    from quantized_channel_estimation_b200 import engine
    rt = ROUTES[name]
    d = route_data(name)
    K = len(params['w'])
    if rt['kind'] == 'gmm':
        m = qce.Gmm_nbit(n_components=K).set_parameters(params['means'], params['covs'], params['w'], detect_structure=False)
        want = engine.DenseModel
    elif rt['kind'] == 'mfa':
        m = qce.Mofa(K, rt['M'], verbose=False).set_parameters(params['means'], params['lam'], params['psi'], params['w'])
        want = engine.MfaModel
    else:
        m = qce.Gmm_nbit(n_components=K, covariance_type='block-circulant').set_circulant_parameters(params['c'], params['w'], rt['blocks'])
        want = engine.CircModel
    m.precision = rt['prec']
    N = params['means'].shape[1]
    with np.errstate(divide='ignore'):
        model = m._prepared(np.eye(N), rt['snr'], rt['nb'], rt['qt'], d['qz'])
    assert type(model) is want, (name, type(model))
    return model


def _launches():
    from quantized_channel_estimation_b200 import _lib
    return _lib.launch_count()


def _fix_count():
    import torch
    from quantized_channel_estimation_b200 import _lib
    return _lib.load().qce_last_fix_count(C.c_void_p(torch.cuda.current_stream().cuda_stream))


def check_route(qce, name, params, monkeypatch, modes=None):
    """Run the route's model over ``modes`` (default: the whole domain) and check it against the oracle."""
    import torch
    rt = ROUTES[name]
    for k, v in rt.get('env', {}).items():
        monkeypatch.setenv(k, v)
    d = route_data(name)
    rows, h, r = d['rows'], d['h'], d['r']
    B = r.shape[0]
    model = engine_model(qce, name, params)
    o = oracle_eval(rt['kind'], params, r[rows], rt['snr'], rt['nb'], rt['qt'], d['qz'])
    tg, tr = TOL[rt['prec']]
    rt_dev, ht = torch.from_numpy(r).cuda(), torch.from_numpy(h).cuda()
    zero = np.nonzero(params['w'] == 0)[0]
    for mode in (modes or mode_domain(len(params['w']))):
        est, acc = model.estimate(rt_dev, mode, rt['prec'], h_true=ht)
        est, acc = est.cpu().numpy(), acc.cpu().numpy()
        # the tensor cores answered the batch (at rho ~ 1 the prefix sums of most pilots end within the FP32 error of rho: those
        # selections are re-made in complex128 by design)
        if rt['prec'] == 'tc' and rt['kind'] == 'gmm' and not (isinstance(mode, float) and abs(mode - 1.0) < 2e-3):
            assert 0 <= _fix_count() <= B // 4, (name, mode, _fix_count())
        assert np.isfinite(est.view(np.float64)).all(), (name, mode, int((~np.isfinite(est)).any(1).sum()))
        ref = oracle_mode(o, mode)
        sub = est[rows]
        per = np.linalg.norm(sub - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert relerr(sub, ref) < tg and per.max() < tr, (name, mode, relerr(sub, ref), per.max(), rows[np.argmax(per)])
        # NMSE accumulators: every row once, the error sums of the whole batch and of the oracle's rows
        assert acc[2] == B, (name, mode, acc[2])
        np.testing.assert_allclose(acc[1], np.sum(np.abs(h) ** 2), rtol=1e-12 if rt['prec'] == 'fp64' else 1e-5)
        np.testing.assert_allclose(acc[0], np.sum(np.abs(est - h) ** 2), rtol=1e-9 if rt['prec'] == 'fp64' else 1e-5)
        np.testing.assert_allclose(np.sum(np.abs(sub - h[rows]) ** 2), np.sum(np.abs(ref - h[rows]) ** 2),
                                   rtol=1e-7 if rt['prec'] == 'fp64' else 1e-3)
    # log-probability export (for the dense tensor-core models this takes the mode path with the selection launch)
    est, lp = model.estimate(rt_dev, 'all', rt['prec'], want_logp=True)
    est, lp = est.cpu().numpy()[rows], lp.cpu().numpy()[rows]
    ref = oracle_mode(o, 'all')
    assert relerr(est, ref) < tg and (np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)).max() < tr
    wlp = o['wlp']
    assert np.array_equal(np.isneginf(lp), np.isneginf(wlp)) and np.isneginf(lp[:, zero]).all(), (name, zero)
    fin = np.isfinite(wlp)
    assert np.isfinite(lp[fin]).all()
    scale = np.abs(wlp[fin]).max()
    if rt['prec'] == 'fp64':
        bound = 1e-9 * max(1.0, scale)
    elif rt['kind'] == 'circ':
        bound = 2e-3 * max(1.0, scale / 300)
    else:
        bound = 2e-4 * max(1.0, scale / 50)
    assert np.abs(lp[fin] - wlp[fin]).max() < bound, (name, np.abs(lp[fin] - wlp[fin]).max(), bound)
    return model, o


def observe_route(qce, name, model, o, monkeypatch):
    """Where the route can be seen from the host: launch counts of the route against a neighbouring route, and the pair counts
    that decide the device-side fallback."""
    import torch
    rt = ROUTES[name]
    rt_dev = torch.from_numpy(route_data(name)['r']).cuda()

    def launches(mode, **kw):
        n0 = _launches()
        model.estimate(rt_dev, mode, rt['prec'], **kw)
        torch.cuda.synchronize()
        return _launches() - n0

    if rt.get('tc') == 'fused' and not rt.get('env'):
        # 'all' without export: the one fused launch; with export: whitening -> selection -> weighted launches
        assert launches('all') < launches('all', want_logp=True)
        # top-1 on this batch is bucketed: one regrouping launch more than the weighted top-1
        b = launches(1, want_logp=True)
        monkeypatch.setenv('QCE_TC_BUCKET', '0')
        assert b > launches(1, want_logp=True)
        monkeypatch.delenv('QCE_TC_BUCKET')
    if rt.get('tc') == 'hard':
        hard = launches(1)
        monkeypatch.setenv('QCE_TC_HARD', '0')
        assert hard > launches(1)
        monkeypatch.delenv('QCE_TC_HARD')
    if rt.get('tc') == 'split' and not rt.get('env'):
        on = launches(2)
        monkeypatch.setenv('QCE_TC_PAIRS', '0')
        assert on > launches(2)
        monkeypatch.delenv('QCE_TC_PAIRS')
        dense = [m for m in mode_domain(rt['K']) if tc_pairs(rt['B'], rt['K'], rt['N'], m) and pairs_per_pilot(o, m) > TC_PAIR_CAP]
        paired = [m for m in mode_domain(rt['K']) if tc_pairs(rt['B'], rt['K'], rt['N'], m) and pairs_per_pilot(o, m) <= TC_PAIR_CAP]
        if rt['snr'] < 0:
            assert 'all' in dense and 0.999 in dense, dense          # flat posterior: the device falls back to the weighted launch
        else:
            assert 2 in paired and -1.0 in paired, paired


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(ROUTES))
def test_route_over_mode_domain(qce, name, monkeypatch):
    model, o = check_route(qce, name, route_data(name)['params'], monkeypatch)
    observe_route(qce, name, model, o, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize('variant', list(zero_weight_variants(4)))
@pytest.mark.parametrize('name', list(ROUTES))
def test_zero_weight_components(qce, name, variant, monkeypatch):
    """A component of weight exactly 0 contributes nothing: responsibility 0, never selected with a non-zero weight, estimates
    equal to the oracle's, log-probability -inf."""
    p = route_data(name)['params']
    w = p['w'].copy()
    w[zero_weight_variants(len(w))[variant]] = 0.0
    check_route(qce, name, with_weights(p, w), monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(ROUTES))
def test_split_component_leaves_the_mixture_unchanged(qce, name, monkeypatch):
    """Component j split into two identical halves is the same mixture (exact log-likelihood ties on the FP32 paths): the same
    'all' estimates to the route's tolerance.  The circulant tensor-core kernel is instantiated for K = 64 and 128 only: there the
    split model has K = 64 and the unsplit one (63 components) runs on the complex128 circulant kernel."""
    import torch
    rt = ROUTES[name]
    for k, v in rt.get('env', {}).items():
        monkeypatch.setenv(k, v)
    d = route_data(name)
    p = d['params']
    prec_a = rt['prec']
    if rt['kind'] == 'circ' and rt['prec'] == 'tc':
        p = {k: (v[:-1] if k in ('means', 'covs', 'c', 'w') else v) for k, v in p.items()}
        prec_a = 'fp64'
    j = int(np.argmax(p['w']))
    r = torch.from_numpy(d['r']).cuda()
    a = engine_model(qce, name, p).estimate(r, 'all', prec_a).cpu().numpy()
    b = engine_model(qce, name, split_component(rt['kind'], p, j)).estimate(r, 'all', rt['prec']).cpu().numpy()
    assert np.isfinite(b.view(np.float64)).all()
    tg, tr = TOL[rt['prec']]
    per = np.linalg.norm(b - a, axis=1) / np.linalg.norm(a, axis=1)
    assert relerr(b, a) < tg and per.max() < tr, (name, relerr(b, a), per.max())


@pytest.mark.gpu
@pytest.mark.parametrize('prec', ['fp64', 'tc'])
def test_c_abi_topn_1_equals_top1(qce, prec):
    """QCE_MODE_TOPN with n_top = 1 selects the same component as QCE_MODE_TOP1 (weight p / p = 1)."""
    import torch
    from quantized_channel_estimation_b200 import _lib
    name = 'dense_fp64_ts16' if prec == 'fp64' else 'tc_fused'
    d = route_data(name)
    model = engine_model(qce, name, d['params'])
    lib = _lib.load()
    r = torch.from_numpy(d['r']).cuda()
    outs = []
    for mode in (_lib.MODE_TOP1, _lib.MODE_TOPN):
        out = torch.empty((r.shape[0], model.n_ant), dtype=torch.complex128, device='cuda')
        _lib.check(lib.qce_estimate(model.handle, C.c_void_p(torch.cuda.current_stream().cuda_stream), C.c_void_p(r.data_ptr()),
                                    r.shape[0], mode, 1, 0.0, _lib.PREC_FP64 if prec == 'fp64' else _lib.PREC_TC,
                                    C.c_void_p(out.data_ptr()), None, None, None))
        outs.append(out.cpu().numpy())
    per = np.linalg.norm(outs[1] - outs[0], axis=1) / np.linalg.norm(outs[0], axis=1)
    assert relerr(outs[1], outs[0]) < (1e-12 if prec == 'fp64' else TOL['tc'][0]) and per.max() < TOL[prec][1]
