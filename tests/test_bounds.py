"""Where the kernels read and write, and whether a result depends on what ran before it on the stream.

The parity suites allocate every output with exactly B rows through the high-level API, so a write one tile past the end lands in
allocator slack that nobody checks, and an out-of-range read sees whatever happens to lie there.  Here the C ABI is called through
ctypes with pointers into slabs the test owns:

  * every output lies between two guards of at least one 512-row work unit, filled with a sentinel byte (0xA5) that must survive
    the call; small accumulator arrays (f64[3], f64[5]) sit inside 16-element slabs;
  * every input is surrounded by "poison" -- zeros, NaN bytes, or 1e300 -- and the outputs (and the tensor-core fix count) must be
    the same bit for bit whatever the poison is; input slabs must come back unchanged, neighbours included;
  * batch sizes sit at 1, T - 1, T + 1, U - 1, U + 1 and 2U + T + 1 of each route's tile T and work unit U, and every row of them is
    checked against the numpy oracle;
  * each route also runs with every device array 16- but not 32-byte aligned, and with only some of its outputs requested;
  * a call on a stream that has run other work (a large batch with off-grid and NaN rows, a model with twice as wide tiles, a
    pair-bucketed top-4, another model's formatted pilots, the release of the host path's staging) gives what it gives on a fresh
    stream.

A stray access lands in memory the test owns, so nothing here can fault.  The route table is test_mode_domain's, plus the routes it
lacks (n_obs = 256, the plain length-256 circulant, a two-pilot shape, a zero-padded shape, K = 1)."""
import ctypes as C
from contextlib import contextmanager

import numpy as np
import pytest

from conftest import relerr
from oracle import qce_oracle as orc
from test_mode_domain import (CIRC_TC_TILE, N_SMS, ROUTES, TC_TILE, TC_UNIT, TOL, circ_ts, engine_model, fp64_dense_ts,
                              oracle_eval, oracle_mode, route_data, tc_bucketed_top1, tc_pairs)

SENTINEL = 0xA5
GUARD_ROWS = TC_UNIT                       # one work unit of guard on each side of every row array
POISON = {'zero': 0.0, 'nan': float('nan'), 'big': 1e300}
MODES = ['all', 1, 3, 0.9]
HOST_SLOT_BYTES = 32 << 20                 # qce_api.cu: staging slot of the host-buffer path (4 slots)
HOST_SLOTS = 4
QUANT_GRID_THREADS = N_SMS * 8 * 256       # qce_quantize.cu: the grid-stride loop's threads (8 CTAs of 256 per SM)

# ----------------------------------------------------------------------------------------------------- routes

# T: the route's tile; U: its work unit (dense tensor cores), or the batch size at which the next tile size takes over (complex128
# kernels, so that U - 1 and U + 1 run on different instantiations), or four tiles (circulant tensor cores).  `extra`: (batch size,
# modes) that reach the dispatches the sizes around T and U do not: top-1 regrouped by label (a chunk of at least four 512-row
# buckets, 4U + T + 1) and the pair-bucketed top-n / cumulative / 'all' of the split shapes (B >= 16 U, 16U + T + 1)
BUCKET_B = 4 * TC_UNIT + TC_TILE + 1
PAIR_B = 16 * TC_UNIT + TC_TILE + 1
BOUND_ROUTES = {
    'dense_fp64_ts8': dict(base='dense_fp64_ts8', T=8, U=16 * 64),
    'circ_fp64_ts4': dict(base='circ_fp64_ts4', T=4, U=8 * 64),
    'mfa_ts8': dict(base='mfa_ts8', T=8, U=16 * 64),
    'tc_fused': dict(base='tc_fused', T=TC_TILE, U=TC_UNIT, extra=[(BUCKET_B, [1])]),
    'tc_hard_top1': dict(base='tc_hard_top1', T=TC_TILE, U=TC_UNIT),
    'tc_split_pairs': dict(base='tc_split_pairs', T=TC_TILE, U=TC_UNIT, extra=[(PAIR_B, ['all', 1, 3, 0.9])]),
    'tc_three_pass': dict(base='tc_three_pass', T=TC_TILE, U=TC_UNIT, extra=[(BUCKET_B, [1])]),
    'circ_tc': dict(base='circ_tc', T=CIRC_TC_TILE, U=4 * CIRC_TC_TILE),
    # routes test_mode_domain's table lacks
    'tc_n256_split': dict(kind='gmm', K=8, N=256, nb=1, qt='uniform', ms=0.0, snr=10, prec='tc', T=TC_TILE, U=TC_UNIT,
                          extra=[(PAIR_B, ['all', 3])]),
    'circ_tc_plain256': dict(kind='circ', K=64, blocks=(1, 256), nb=1, qt='uniform', snr=8, prec='tc', T=CIRC_TC_TILE,
                             U=4 * CIRC_TC_TILE),
    'tc_two_pilot': dict(kind='gmm', K=16, N=32, pilots=2, nb=1, qt='uniform', ms=0.1, snr=5, prec='tc', T=TC_TILE, U=TC_UNIT),
    'tc_padded': dict(kind='gmm', K=8, N=40, nb=2, qt='uniform', ms=0.1, snr=10, prec='tc', pad=True, T=TC_TILE, U=TC_UNIT),
    'tc_k1': dict(kind='gmm', K=1, N=64, nb=1, qt='uniform', ms=0.0, snr=10, prec='tc', T=TC_TILE, U=TC_UNIT),
}


def route_spec(name):
    b = BOUND_ROUTES[name]
    spec = dict(ROUTES[b['base']]) if 'base' in b else dict(b)
    spec.update(T=b['T'], U=b['U'])
    return spec


def route_sizes(name):
    """(batch size, modes) of a route: every mode at the sizes around its tile and work unit, then its extra sizes."""
    rt = route_spec(name)
    return [(B, MODES) for B in batch_sizes(rt['T'], rt['U'])] + BOUND_ROUTES[name].get('extra', [])


def pair_call(rt, B, mode):
    """The call takes the pair-bucketed combination, whose FP32 atomics add the rows of a pilot in any order."""
    return rt['kind'] == 'gmm' and rt['prec'] == 'tc' and tc_pairs(B, rt['K'], rt['N'] * rt.get('pilots', 1), mode)


def bucketed_call(rt, B, mode):
    return (rt['kind'] == 'gmm' and rt['prec'] == 'tc' and mode == 1 and
            tc_bucketed_top1(B, rt['K'], rt['N'] * rt.get('pilots', 1), rt['qt'] == 'lloyd'))


TC_ROUTES = [n for n in BOUND_ROUTES if route_spec(n)['prec'] == 'tc']


def batch_sizes(T, U):
    """1, T - 1, T + 1, U - 1, U + 1 and 2U + T + 1 (ragged in both the tile and the work unit)."""
    return sorted({1, T - 1, T + 1, U - 1, U + 1, 2 * U + T + 1})


def host_chunk(max_row_bytes):
    """Rows per staging chunk of the host-buffer path (qce_api.cu estimate_host_impl)."""
    return max(HOST_SLOT_BYTES // max_row_bytes, 128)


def host_batch_sizes(max_row_bytes):
    c = host_chunk(max_row_bytes)
    return [c - 1, c + 1, HOST_SLOTS * c + 1]


QUANT_SIZES = [1, 3, 257, QUANT_GRID_THREADS + 1]

# ----------------------------------------------------------------------------------------------------- guarded slabs


def first_bad_guard(raw, lo, hi, row_bytes, sentinel=SENTINEL):
    """Guard bytes of ``raw`` (everything outside [lo, hi)) that are not ``sentinel``: None, or a message naming the side and the
    offset, in rows from the start of the data, of the first changed byte of each side (negative: before the data)."""
    msgs = []
    front = np.flatnonzero(raw[:lo] != sentinel)
    if front.size:
        msgs.append(f'front guard changed at row {(int(front[0]) - lo) // row_bytes} ({front.size} bytes)')
    back = np.flatnonzero(raw[hi:] != sentinel)
    if back.size:
        msgs.append(f'back guard changed at row {(int(back[0]) + hi - lo) // row_bytes} ({back.size} bytes)')
    return '; '.join(msgs) or None


def _pattern(value, n):
    return np.resize(np.frombuffer(np.float64(value).tobytes(), np.uint8), n)


class Slab:
    """``rows`` rows of ``row_bytes`` bytes between ``front`` and ``back`` guard rows, on the device ('cuda'), in pageable host memory
    ('host') or in page-locked host memory ('pinned').  ``offset`` shifts the data (and its back guard) by that many bytes."""

    def __init__(self, rows, row_bytes, where='cuda', front=GUARD_ROWS, back=GUARD_ROWS, offset=0):
        import torch
        self.rows, self.rb, self.where = rows, row_bytes, where
        self.lo = front * row_bytes + offset
        self.hi = self.lo + rows * row_bytes
        n = self.hi + back * row_bytes
        if where == 'cuda':
            self.buf = torch.full((n,), SENTINEL, dtype=torch.uint8, device='cuda')
        elif where == 'pinned':
            self.buf = torch.full((n,), SENTINEL, dtype=torch.uint8).pin_memory()
            assert self.buf.is_pinned()
        else:
            self.buf = np.full(n, SENTINEL, dtype=np.uint8)
        self.expect = None          # inputs: every byte must come back as written

    @property
    def addr(self):
        return (self.buf.ctypes.data if self.where == 'host' else self.buf.data_ptr()) + self.lo

    @property
    def ptr(self):
        return C.c_void_p(self.addr)

    def raw(self):
        if self.where == 'cuda':
            return self.buf.cpu().numpy()
        return (self.buf if self.where == 'host' else self.buf.numpy()).copy()

    def _store(self, raw):
        import torch
        if self.where == 'host':
            self.buf[:] = raw
        else:
            self.buf.copy_(torch.from_numpy(raw))

    def fill(self, data):
        """Set the data bytes of an output (accumulators that are added into)."""
        raw = self.raw()
        raw[self.lo:self.hi] = np.ascontiguousarray(data).view(np.uint8).ravel()
        self._store(raw)

    def write(self, data, poison=0.0):
        """An input: the data, and its neighbours (the guards) filled with float64 ``poison``."""
        raw = _pattern(poison, self.buf.shape[0])
        raw[self.lo:self.hi] = np.ascontiguousarray(data).view(np.uint8).ravel()
        self._store(raw)
        self.expect = raw
        return self

    def read(self, dtype):
        return self.raw()[self.lo:self.hi].view(dtype).copy()

    def check(self, what=''):
        raw = self.raw()
        if self.expect is not None:
            bad = np.flatnonzero(raw != self.expect)
            assert bad.size == 0, f'{what}: input slab changed at row {(int(bad[0]) - self.lo) // self.rb} ({bad.size} bytes)'
        else:
            msg = first_bad_guard(raw, self.lo, self.hi, self.rb)
            assert msg is None, f'{what}: {msg}'


def acc_slab(n=3, where='cuda', offset=0):
    """An f64[n] accumulator (zeros) inside a 16-element slab, 32-byte aligned plus ``offset`` bytes."""
    s = Slab(n, 8, where, front=4, back=16 - 4 - n - offset // 8, offset=offset)
    s.fill(np.zeros(n))
    return s


def _in(data, poison, offset=0, where='cuda'):
    data = np.ascontiguousarray(data)
    return Slab(data.shape[0], data[0].nbytes if data.ndim > 1 else data.itemsize, where, offset=offset).write(data, POISON[poison])


# ----------------------------------------------------------------------------------------------------- CPU tests

@pytest.mark.parametrize('where', ['front', 'back'])
def test_guard_checker_finds_one_planted_byte(where):
    rows, rb, front, back = 5, 48, 3, 4
    raw = np.full((front + rows + back) * rb, SENTINEL, dtype=np.uint8)
    lo, hi = front * rb, (front + rows) * rb
    raw[lo:hi] = 0
    assert first_bad_guard(raw, lo, hi, rb) is None
    for pos, row in ((0, -3), (lo - 1, -1), (hi, rows), (raw.size - 1, rows + back - 1)):
        if (pos < lo) != (where == 'front'):
            continue
        planted = raw.copy()
        planted[pos] ^= 0x01
        msg = first_bad_guard(planted, lo, hi, rb)
        assert msg is not None and f'{where} guard changed at row {row} (1 bytes)' == msg, msg


def test_batch_sizes_straddle_every_tile_and_unit():
    for name in BOUND_ROUTES:
        rt = route_spec(name)
        T, U = rt['T'], rt['U']
        sizes = batch_sizes(T, U)
        assert {1, T - 1, T + 1, U - 1, U + 1} <= set(sizes), name
        assert max(sizes) == 2 * U + T + 1 and max(sizes) % T == 1 and max(sizes) % U == T + 1, name
        if rt['prec'] == 'fp64':          # U - 1 and U + 1 run on different tile sizes of the complex128 kernels
            ts = circ_ts if rt['kind'] == 'circ' else fp64_dense_ts
            assert ts(T + 1) == T and ts(U - 1) == T and ts(U + 1) == 2 * T, name
    assert host_chunk(64 * 16) == 32768 and host_batch_sizes(64 * 16) == [32767, 32769, 131073]
    assert QUANT_SIZES[-1] > QUANT_GRID_THREADS          # the last quantiser size takes a second pass of the grid-stride loop
    assert set(TC_ROUTES) >= {'tc_fused', 'tc_hard_top1', 'tc_split_pairs', 'tc_three_pass', 'circ_tc', 'tc_n256_split',
                              'circ_tc_plain256', 'tc_two_pilot', 'tc_padded', 'tc_k1'}


def test_size_lists_reach_the_bucketed_dispatches():
    """The pair-bucketed modes of the split shapes and the label-bucketed top-1 run on guarded batches (test_mode_domain's
    predicates of the dispatch thresholds), and the sizes around T and U stay on the launches without buckets."""
    reach = {}
    for name in BOUND_ROUTES:
        rt = route_spec(name)
        sizes = route_sizes(name)
        reach[name] = dict(pairs={str(m) for B, ms in sizes for m in ms if pair_call(rt, B, m)},
                           bucket=any(bucketed_call(rt, B, m) for B, ms in sizes for m in ms))
        assert not any(pair_call(rt, B, m) for B in batch_sizes(rt['T'], rt['U']) for m in MODES), name
    assert reach['tc_split_pairs']['pairs'] == {'all', '3', '0.9'}
    assert reach['tc_n256_split']['pairs'] == {'all', '3'}
    for name in ('tc_fused', 'tc_three_pass', 'tc_split_pairs', 'tc_n256_split'):
        assert reach[name]['bucket'], name
    assert not bucketed_call(route_spec('tc_fused'), BUCKET_B - TC_UNIT, 1)
    assert max(B for B, _ in route_sizes('tc_split_pairs')) % TC_UNIT == TC_TILE + 1


def test_extra_routes_reach_their_shapes():
    from quantized_channel_estimation_b200 import engine
    assert engine.tc_shape_ok(256, 256, on_grid=True) and not engine.tc_shape_ok(256, 256)
    assert engine.tc_shape_ok(64, 32) and not engine.tc_shape_ok(40, 40)
    assert engine.tc_padded_shape(40, 40, on_grid=True) not in (None, (40, 40))
    assert engine.tc_shape_ok(128, 128)          # the three-pass model of the stream-history tests (tiles twice as wide)


# ----------------------------------------------------------------------------------------------------- GPU side

@pytest.fixture(scope='module')
def qce():
    import quantized_channel_estimation_b200 as q
    from quantized_channel_estimation_b200 import _lib
    _lib.require_device()
    return q


def _lib_():
    from quantized_channel_estimation_b200 import _lib
    return _lib


def _cur_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sync():
    import torch
    torch.cuda.synchronize()


class Case:
    """A route's model handle, its pilots / channels for the largest batch size, and the oracle's pieces on them."""


_CASES = {}


def two_pilot_A(N):
    return np.kron(np.array([[1.0], [1j]]), np.eye(N))


def case(qce, name):
    if name in _CASES:
        return _CASES[name]
    from quantized_channel_estimation_b200 import engine, precompute
    b, rt = BOUND_ROUTES[name], route_spec(name)
    Bmax = max(B for B, _ in route_sizes(name))
    if rt['kind'] == 'gmm' and rt['prec'] == 'tc':
        Bmax = max(Bmax, 1537)                # test_mode_chunk_of_512_rows
    K, snr, nb, qt = rt['K'], rt['snr'], rt['nb'], rt['qt']
    seed = 1000 + sum(map(ord, name))
    A = None
    if 'base' in b:
        d = route_data(b['base'])
        params, qz = d['params'], d['qz']
        model = engine_model(qce, b['base'], params)
    else:
        qz = orc.get_quantizer([snr], nb, qt)[snr]
        if rt['kind'] == 'circ':
            c, covs, w, _ = orc.circulant_gmm(K, *rt['blocks'], seed=seed)
            params = dict(means=np.zeros((K, c.shape[1]), dtype=complex), covs=covs, w=w, c=c)
            model = engine.CircModel(precompute.prepare_circulant(c, w, rt['blocks'], snr, nb, qt, qz))
        else:
            means, covs, w = orc.random_psd_gmm(K, rt['N'], seed=seed, mean_scale=rt['ms'])
            params = dict(means=means, covs=covs, w=w)
            A = two_pilot_A(rt['N']) if rt.get('pilots') == 2 else None
            model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(rt['N']) if A is None else A, snr, nb, qt, qz),
                                      pad=rt.get('pad', False))
            assert model.padded == bool(rt.get('pad')), name
    h, noise, _ = orc.sample_gmm_channels(params['means'], params['covs'], params['w'], Bmax, seed=seed + 1)
    if A is not None:
        noise = orc.crandn(Bmax, A.shape[0], rng=np.random.default_rng(seed + 2))
    r = orc.get_observation_nbit(h, snr, noise, A, nb, qz[0], qz[1])
    with np.errstate(divide='ignore'):
        if A is None:
            o = oracle_eval(rt['kind'], params, r, snr, nb, qt, qz)
        else:
            from scipy.special import logsumexp
            prep = orc.gmm_prepare(params['means'], params['covs'], A, snr, nb, qt, qz)
            wlp = orc.gmm_weighted_log_prob(r, prep, params['w'])
            o = dict(wlp=wlp, proba=np.exp(wlp - logsumexp(wlp, axis=1)[:, None]),
                     hk=orc._component_lmmse(r, params['means'], params['covs'], prep), labels=wlp.argmax(axis=1))
    cs = Case()
    cs.name, cs.rt, cs.model, cs.kind, cs.prec = name, rt, model, rt['kind'], rt['prec']
    cs.K = K
    cs.n_true = h.shape[1]
    cs.No = getattr(model, 'pad_obs', model.n_obs)
    cs.N = getattr(model, 'pad_ant', model.n_ant)
    cs.r = np.zeros((Bmax, cs.No), dtype=complex)
    cs.r[:, :r.shape[1]] = r
    cs.h = np.zeros((Bmax, cs.N), dtype=complex)
    cs.h[:, :cs.n_true] = h
    cs.ref = {str(m): oracle_mode(o, m) for m in MODES}
    cs.wlp = o['wlp']
    cs.qz = qz
    _CASES[name] = cs
    return cs


def run_estimate(cs, B, mode, poison='zero', offset=0, h_est=True, logp=False, acc=True, stream=None, r=None):
    """One guarded call of the route's estimate entry point on the first B rows; returns its outputs and fix count."""
    from quantized_channel_estimation_b200 import engine
    _lib = _lib_()
    lib = _lib.load()
    md, n_top, rho = engine.parse_mode(mode)
    s = stream if stream is not None else _cur_stream()
    _sync()                                   # a raw stream does not wait for work of torch's streams
    rs = _in(cs.r[:B] if r is None else r, poison, offset)
    hts = _in(cs.h[:B], poison, offset) if acc else None
    he = Slab(B, cs.N * 16, offset=offset) if h_est else None
    lp = Slab(B, cs.K * 8, offset=offset) if logp else None
    ac = acc_slab(offset=offset) if acc else None
    for sl in (rs, hts, he, lp, ac):
        assert sl is None or sl.addr % 32 == offset % 32, (sl.addr, offset)
    _sync()
    P = lambda x: x.ptr if x is not None else None          # noqa: E731
    prec = _lib.PREC_TC if cs.prec == 'tc' else _lib.PREC_FP64
    if cs.kind == 'gmm':
        st = lib.qce_estimate(cs.model.handle, s, rs.ptr, B, md, n_top, rho, prec, P(he), P(lp), P(hts), P(ac))
    elif cs.kind == 'circ':
        st = lib.qce_circ_estimate_prec(cs.model.handle, s, rs.ptr, B, md, n_top, rho, prec, P(he), P(lp), P(hts), P(ac))
    else:
        st = lib.qce_mfa_estimate(cs.model.handle, s, rs.ptr, B, md, n_top, rho, P(he), P(lp), P(hts), P(ac))
    _lib.check(st)
    _sync()
    out = dict(fix=lib.qce_last_fix_count(s) if cs.prec == 'tc' else None)
    where = f'{cs.name} B={B} mode={mode} poison={poison} offset={offset}'
    for nm, sl in (('r', rs), ('h_true', hts), ('h_est', he), ('logp', lp), ('acc', ac)):
        if sl is not None:
            sl.check(f'{where} {nm}')
    out['h_est'] = he.read(np.complex128).reshape(B, cs.N) if he else None
    out['logp'] = lp.read(np.float64).reshape(B, cs.K) if lp else None
    out['acc'] = ac.read(np.float64) if ac else None
    return out


def check_against_oracle(cs, B, mode, out):
    tg, tr = TOL[cs.prec]
    est = out['h_est']
    assert np.isfinite(est.view(np.float64)).all(), (cs.name, B, mode)
    ref = cs.ref[str(mode)][:B]
    sub = est[:, :cs.n_true]
    per = np.linalg.norm(sub - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert relerr(sub, ref) < tg and per.max() < tr, (cs.name, B, mode, relerr(sub, ref), per.max(), int(np.argmax(per)))
    assert (est[:, cs.n_true:] == 0).all(), cs.name                 # zero-padded columns stay zero
    acc = out['acc']
    assert acc[2] == B, (cs.name, B, mode, acc[2])
    h = cs.h[:B]
    np.testing.assert_allclose(acc[1], np.sum(np.abs(h) ** 2), rtol=1e-12 if cs.prec == 'fp64' else 1e-5)
    np.testing.assert_allclose(acc[0], np.sum(np.abs(est - h) ** 2), rtol=1e-9 if cs.prec == 'fp64' else 1e-5)


def check_logp(cs, B, lp):
    wlp = cs.wlp[:B]
    scale = np.abs(wlp).max()
    bound = (1e-9 * max(1.0, scale) if cs.prec == 'fp64' else 2e-3 * max(1.0, scale / 300) if cs.kind == 'circ'
             else 2e-4 * max(1.0, scale / 50))
    assert np.isfinite(lp).all() and np.abs(lp - wlp).max() < bound, (cs.name, B, np.abs(lp - wlp).max(), bound)


def same_outputs(a, b, what, acc_rtol=1e-12, fp32_rows=False):
    """Bit for bit (the accumulators to ``acc_rtol``: FP64 atomics).  ``fp32_rows``: the pair-bucketed combination adds the rows in
    FP32 atomics, in any order -- estimates to 1e-6 per row, accumulators to 1e-6."""
    if fp32_rows:
        per = np.linalg.norm(a['h_est'] - b['h_est'], axis=1) / np.linalg.norm(b['h_est'], axis=1)
        assert np.isfinite(a['h_est']).all() and per.max() < 1e-6, (what, per.max(), int(np.argmax(per)))
        a, b = dict(a, h_est=None), dict(b, h_est=None)
        acc_rtol = max(acc_rtol, 1e-6)
    for k in ('h_est', 'logp'):
        if a[k] is not None:
            assert np.array_equal(a[k].view(np.uint64), b[k].view(np.uint64)), (what, k, int(np.argmax(
                (a[k] != b[k]).reshape(a[k].shape[0], -1).any(1))))
    if a['acc'] is not None:
        assert a['acc'][2] == b['acc'][2], (what, a['acc'], b['acc'])
        np.testing.assert_allclose(a['acc'], b['acc'], rtol=acc_rtol, atol=0, err_msg=str(what))
    assert a['fix'] == b['fix'], (what, a['fix'], b['fix'])


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(BOUND_ROUTES))
def test_estimate_rows_guards_and_poison(qce, name):
    """Every batch size around the route's tile and work unit, modes 'all', 1, 3 and 0.9, and the sizes that reach the bucketed
    dispatches: every row against the oracle, every guard intact, the inputs unchanged, and the same outputs and fix count with zero,
    NaN and 1e300 neighbours (pair-bucketed calls: to 1e-6 per row)."""
    cs = case(qce, name)
    rt = cs.rt
    for B, modes in route_sizes(name):
        for mode in modes:
            base = run_estimate(cs, B, mode)
            check_against_oracle(cs, B, mode, base)
            for poison in ('nan', 'big'):
                same_outputs(run_estimate(cs, B, mode, poison), base, (name, B, mode, poison), fp32_rows=pair_call(rt, B, mode))
        # log-probability export (the dense tensor-core models take the selection launch)
        out = run_estimate(cs, B, 'all', logp=True)
        check_logp(cs, B, out['logp'])
        same_outputs(run_estimate(cs, B, 'all', 'nan', logp=True), out, (name, B, 'logp', 'nan'), fp32_rows=pair_call(rt, B, 'all'))


@pytest.mark.gpu
def test_mode_chunk_of_512_rows(qce, monkeypatch):
    """QCE_TC_MODE_CHUNK=512: the mode path walks a 1537-row batch in four chunks, the last one row long."""
    monkeypatch.setenv('QCE_TC_MODE_CHUNK', '512')
    for name in ('tc_fused', 'tc_split_pairs'):
        cs = case(qce, name)
        for mode in (1, 3, 0.9):
            base = run_estimate(cs, 1537, mode)
            check_against_oracle(cs, 1537, mode, base)
            same_outputs(run_estimate(cs, 1537, mode, 'nan'), base, (name, mode))


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(BOUND_ROUTES))
def test_partial_outputs_and_alignment(qce, name):
    """Only the accumulators, or only the log-probabilities: the same values as the full call and nothing else written.  Every
    device array 16- but not 32-byte aligned: the same results as the aligned call."""
    cs = case(qce, name)
    B = max(B for B, _ in route_sizes(name))
    for mode in ('all', 3):
        fp32 = pair_call(cs.rt, B, mode)
        full = run_estimate(cs, B, mode, logp=True)
        only_acc = run_estimate(cs, B, mode, h_est=False)
        np.testing.assert_allclose(only_acc['acc'], full['acc'], rtol=1e-12 if cs.prec == 'fp64' else 1e-6)
        assert only_acc['acc'][2] == B
        only_lp = run_estimate(cs, B, mode, h_est=False, acc=False, logp=True)
        if mode == 'all':
            assert np.array_equal(only_lp['logp'], full['logp']), (name, mode)
        else:      # (with estimates, the near-ties of a hard selection get complex128 log-probabilities)
            check_logp(cs, B, only_lp['logp'])
        shifted = run_estimate(cs, B, mode, offset=16, logp=True)
        same_outputs(shifted, full, (name, mode, 'offset 16'), fp32_rows=fp32)
        aligned = run_estimate(cs, B, mode, logp=False)
        same_outputs(run_estimate(cs, B, mode, offset=16), aligned, (name, mode, 'offset 16, no export'), fp32_rows=fp32)


# ----------------------------------------------------------------------------------------------------- quantiser

@pytest.mark.gpu
@pytest.mark.parametrize('nb', [1, 3])
def test_quantize_guards(qce, nb):
    from quantized_channel_estimation_b200 import engine
    _lib = _lib_()
    lib = _lib.load()
    snr = 5
    qz = orc.get_quantizer([snr], nb, 'lloyd')[snr] if nb > 1 else (None, None, None)
    q = engine.Quantizer.get(nb, qz[0], qz[1]) if nb > 1 else engine.Quantizer.get(1)
    rng = np.random.default_rng(nb)
    for n in QUANT_SIZES:
        y = orc.crandn(n, rng=rng)
        y[:min(n, 2)] = [0.0, np.nan + 0j][:min(n, 2)]
        want_r, want_c = orc.quant(y, nb, qz[0], qz[1]), orc.quant_codes(y, nb, qz[0])
        outs = {}
        for poison in POISON:
            ys = _in(y, poison)
            rs, cs_ = Slab(n, 16), Slab(n, 2)
            _lib.check(lib.qce_quantize(q.handle, _cur_stream(), ys.ptr, n, rs.ptr, cs_.ptr))
            _sync()
            for nm, sl in (('y', ys), ('r', rs), ('codes', cs_)):
                sl.check(f'quantize n={n} {poison} {nm}')
            outs[poison] = (rs.read(np.complex128), cs_.read(np.uint8).reshape(n, 2))
        r, codes = outs['zero']
        assert np.array_equal(r.view(np.uint64), want_r.view(np.uint64)) and np.array_equal(codes, want_c), n
        for poison in ('nan', 'big'):
            assert np.array_equal(outs[poison][0].view(np.uint64), r.view(np.uint64)) and np.array_equal(outs[poison][1], codes)


@pytest.mark.gpu
@pytest.mark.parametrize('h_c64', [False, True])
@pytest.mark.parametrize('nb', [None, 1, 2])
def test_observe_quantize_guards(qce, nb, h_c64):
    """y = h + s * noise, then the quantiser; with q = NULL only y is written (a call that also asks for r or codes is refused and
    writes nothing)."""
    from quantized_channel_estimation_b200 import engine
    _lib = _lib_()
    lib = _lib.load()
    snr = 3
    scale = 10 ** (-snr / 20)
    qz = orc.get_quantizer([snr], nb, 'uniform')[snr] if nb and nb > 1 else (None, None, None)
    q = None if nb is None else (engine.Quantizer.get(nb, qz[0], qz[1]) if nb > 1 else engine.Quantizer.get(1))
    rng = np.random.default_rng(7)
    for n in QUANT_SIZES:
        h = orc.crandn(n, rng=rng)
        if h_c64:
            h = h.astype(np.complex64)
        noise = orc.crandn(n, rng=rng)
        y_ref = h.astype(np.complex128) + scale * noise
        res = {}
        for poison in POISON:
            hs, ns = _in(h, poison), _in(noise, poison)
            ys, rs, cs_ = Slab(n, 16), Slab(n, 16), Slab(n, 2)
            if q is None:          # r or codes without a quantiser are refused
                assert lib.qce_observe_quantize(None, _cur_stream(), hs.ptr, int(h_c64), ns.ptr, scale, n, ys.ptr, rs.ptr, cs_.ptr) == -1
            _lib.check(lib.qce_observe_quantize(q.handle if q else None, _cur_stream(), hs.ptr, int(h_c64), ns.ptr, scale, n,
                                                ys.ptr, rs.ptr if q else None, cs_.ptr if q else None))
            _sync()
            for nm, sl in (('h', hs), ('noise', ns), ('y', ys), ('r', rs), ('codes', cs_)):
                sl.check(f'observe n={n} {poison} {nm}')
            res[poison] = [ys.read(np.complex128)]
            if q is None:
                assert (rs.raw() == SENTINEL).all() and (cs_.raw() == SENTINEL).all(), 'q = NULL wrote r or codes'
            else:
                res[poison] += [rs.read(np.complex128), cs_.read(np.uint8).reshape(n, 2)]
        assert np.array_equal(res['zero'][0].view(np.uint64), y_ref.view(np.uint64)), n
        if q is not None:
            assert np.array_equal(res['zero'][1].view(np.uint64), orc.quant(y_ref, nb, qz[0], qz[1]).view(np.uint64))
            assert np.array_equal(res['zero'][2], orc.quant_codes(y_ref, nb, qz[0]))
        for poison in ('nan', 'big'):
            assert all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip(res[poison], res['zero'])), (n, poison)


# ----------------------------------------------------------------------------------------------------- fused pipeline

@pytest.mark.gpu
@pytest.mark.parametrize('h_c64', [False, True])
@pytest.mark.parametrize('name', ['dense_fp64_ts8', 'tc_fused', 'tc_split_pairs'])
def test_pipeline_guards(qce, name, h_c64):
    """observe -> quantise -> estimate -> NMSE on guarded, poisoned channels and noise: the estimates of the route's oracle on the
    pilots the oracle quantises from the same draw."""
    from quantized_channel_estimation_b200 import engine
    _lib = _lib_()
    lib = _lib.load()
    cs = case(qce, name)
    rt = cs.rt
    nb, snr, qz = rt['nb'], rt['snr'], cs.qz
    q = engine.Quantizer.get(nb, qz[0], qz[1]) if nb > 1 else engine.Quantizer.get(1)
    scale = 10 ** (-snr / 20)
    sizes = [1, rt['T'] + 1, rt['U'] + 1, max(batch_sizes(rt['T'], rt['U']))]
    Bmax = sizes[-1]
    rng = np.random.default_rng(11)
    d = route_data(BOUND_ROUTES[name]['base'])
    h = cs.h[:Bmax].astype(np.complex64) if h_c64 else cs.h[:Bmax]
    noise = orc.crandn(Bmax, cs.N, rng=rng)
    r = orc.get_observation_nbit(h.astype(np.complex128), snr, noise, None, nb, qz[0], qz[1])
    o = oracle_eval(rt['kind'], d['params'], r, snr, nb, rt['qt'], qz)
    prec = _lib.PREC_TC if cs.prec == 'tc' else _lib.PREC_FP64
    tg, tr = TOL[cs.prec]
    for B in sizes:
        for mode in ('all', 1):
            md, n_top, rho = engine.parse_mode(mode)
            res = {}
            for poison in POISON:
                hs, ns = _in(h[:B], poison), _in(noise[:B], poison)
                he, ac = Slab(B, cs.N * 16), acc_slab()
                _lib.check(lib.qce_pipeline(cs.model.handle, q.handle, _cur_stream(), hs.ptr, int(h_c64), ns.ptr, scale, B, md, n_top,
                                            rho, prec, he.ptr, ac.ptr))
                _sync()
                fix = lib.qce_last_fix_count(_cur_stream()) if cs.prec == 'tc' else None
                for nm, sl in (('h', hs), ('noise', ns), ('h_est', he), ('acc', ac)):
                    sl.check(f'pipeline {name} B={B} {mode} {poison} {nm}')
                res[poison] = dict(h_est=he.read(np.complex128).reshape(B, cs.N), logp=None, acc=ac.read(np.float64), fix=fix)
            est, acc = res['zero']['h_est'], res['zero']['acc']
            ref = oracle_mode(o, mode)[:B]
            per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
            assert relerr(est, ref) < tg and per.max() < tr, (name, B, mode, relerr(est, ref), per.max())
            assert acc[2] == B
            hh = h[:B].astype(np.complex128)
            np.testing.assert_allclose(acc[0], np.sum(np.abs(est - hh) ** 2), rtol=1e-9 if cs.prec == 'fp64' else 1e-5)
            for poison in ('nan', 'big'):
                same_outputs(res[poison], res['zero'], (name, B, mode, poison))


# ----------------------------------------------------------------------------------------------------- formatted pilots

def _formatted_case(qce):
    cs = case(qce, 'tc_fused')
    B_fmt = 1000
    r = cs.r[:B_fmt].copy()
    r[900, 0] = 0.123                     # off the quantiser grid: on the fix list
    r[950, 3] = np.nan                    # NaN: on the fix list
    return cs, r, B_fmt


@pytest.mark.gpu
def test_estimate_formatted_on_fewer_rows_than_formatted(qce):
    """qce_format_pilots of 1000 pilots (an off-grid row at 900, a NaN row at 950), then qce_estimate_formatted on the first 700:
    the fix-list rows past 700 are neither written, nor read from h_true, nor counted."""
    from test_stream_scratch import raw_stream
    _lib = _lib_()
    lib = _lib.load()
    cs, r, B_fmt = _formatted_case(qce)
    B = 700
    results = {}
    for poison in POISON:
        rs = _in(r, poison)
        hts = _in(cs.h[:B], poison)
        he, ac = Slab(B, cs.N * 16), acc_slab()
        _sync()
        with raw_stream() as s:
            _lib.check(lib.qce_format_pilots(cs.model.handle, s, rs.ptr, B_fmt))
            _lib.check(lib.qce_estimate_formatted(cs.model.handle, s, B, he.ptr, hts.ptr, ac.ptr))
        _sync()
        for nm, sl in (('r', rs), ('h_true', hts), ('h_est', he), ('acc', ac)):
            sl.check(f'estimate_formatted B={B} of {B_fmt} poison={poison} {nm}')
        acc = ac.read(np.float64)
        assert acc[2] == B and np.isfinite(acc).all(), (poison, acc)
        results[poison] = (he.read(np.complex128).reshape(B, cs.N), acc)
    # the same as qce_estimate on the first 700 pilots (which has no listed row)
    ref = run_estimate(cs, B, 'all', stream=None, r=r[:B])
    assert ref['fix'] == 0
    for poison, (est, acc) in results.items():
        assert np.array_equal(est.view(np.uint64), ref['h_est'].view(np.uint64)), poison
        np.testing.assert_allclose(acc, ref['acc'], rtol=1e-12)
    check_against_oracle(cs, B, 'all', ref)


@pytest.mark.gpu
@pytest.mark.parametrize('B', [1, 127, 129, 511, 513, 1000])
def test_estimate_formatted_guards(qce, B):
    """The pair on batch sizes around the tile and the work unit, with the listed rows inside the batch where it has them."""
    from test_stream_scratch import raw_stream
    _lib = _lib_()
    lib = _lib.load()
    cs, r, B_fmt = _formatted_case(qce)
    r = r[:B]
    res = {}
    for poison in POISON:
        rs, hts = _in(r, poison), _in(cs.h[:B], poison)
        he, ac = Slab(B, cs.N * 16), acc_slab()
        _sync()
        with raw_stream() as s:
            _lib.check(lib.qce_format_pilots(cs.model.handle, s, rs.ptr, B))
            _lib.check(lib.qce_estimate_formatted(cs.model.handle, s, B, he.ptr, hts.ptr, ac.ptr))
            fix = lib.qce_last_fix_count(s)
        for nm, sl in (('r', rs), ('h_true', hts), ('h_est', he), ('acc', ac)):
            sl.check(f'estimate_formatted B={B} poison={poison} {nm}')
        res[poison] = dict(h_est=he.read(np.complex128).reshape(B, cs.N), logp=None, acc=ac.read(np.float64), fix=fix)
    assert res['zero']['fix'] == (B > 900) + (B > 950)
    same_outputs(res['zero'], run_estimate(cs, B, 'all', r=r), ('formatted vs estimate', B))
    for poison in ('nan', 'big'):
        same_outputs(res[poison], res['zero'], ('formatted', B, poison))


# ----------------------------------------------------------------------------------------------------- rate accumulators

@pytest.mark.gpu
@pytest.mark.parametrize('h_c64', [False, True])
def test_rate_accumulate_guards(qce, h_c64):
    from quantized_channel_estimation_b200 import engine
    _lib = _lib_()
    lib = _lib.load()
    N = 64
    rng = np.random.default_rng(5)
    bdiag = 0.5 + rng.random(N)
    X = orc.crandn(N, 2 * N, rng=rng)
    Cq = X @ X.conj().T / (2 * N)
    model = engine.RateModel(np.diag(bdiag), Cq)
    Bmax = 2 * TC_UNIT + TC_TILE + 1
    he_all = orc.crandn(Bmax, N, rng=rng) * 0.3
    h_all = orc.crandn(Bmax, N, rng=rng)
    if h_c64:
        h_all = h_all.astype(np.complex64)
    for B in batch_sizes(TC_TILE, TC_UNIT):
        he, h = he_all[:B], h_all[:B]
        g = he / np.maximum(np.sum(np.abs(he) ** 2, axis=1), 0.1)[:, None]
        inner = np.sum(g.conj() * bdiag * h.astype(np.complex128), axis=1)
        qf = np.real(np.einsum('bi,ij,bj->b', g.conj(), Cq, g))
        want = np.array([inner.real.sum(), inner.imag.sum(), np.sum(np.abs(inner) ** 2), qf.sum(), B])
        res = {}
        for poison in POISON:
            hes, hs, ac = _in(he, poison), _in(h, poison), acc_slab(5)
            _lib.check(lib.qce_rate_accumulate(model.handle, _cur_stream(), hes.ptr, hs.ptr, int(h_c64), B, ac.ptr))
            _sync()
            for nm, sl in (('h_est', hes), ('h_true', hs), ('acc', ac)):
                sl.check(f'rate B={B} {poison} {nm}')
            res[poison] = ac.read(np.float64)
        acc = res['zero']
        assert acc[4] == B
        np.testing.assert_allclose(acc[:3], want[:3], rtol=1e-9, atol=1e-9 * np.abs(want[:3]).max())
        np.testing.assert_allclose(acc[3], want[3], rtol=1e-5)
        for poison in ('nan', 'big'):
            np.testing.assert_allclose(res[poison], acc, rtol=1e-12, atol=0)


# ----------------------------------------------------------------------------------------------------- parameter uploads

def _poisoned_arrays(tensors, poison):
    """Device copies of the parameter arrays, each between two guards of its own size filled with the poison."""
    import torch
    out = []
    for t in tensors:
        a = t.detach().cpu().contiguous().numpy()
        out.append(Slab(1, a.nbytes, front=1, back=1).write(a.reshape(1, -1), POISON[poison]))
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['dense', 'dense_split', 'circ', 'mfa', 'rate'])
def test_set_params_reads_only_its_blocks(qce, kind):
    """*_set_params with every parameter array between poisoned neighbours: the models estimate the same, bit for bit."""
    import torch
    from quantized_channel_estimation_b200 import engine, precompute
    _lib = _lib_()
    lib = _lib.load()
    s = _cur_stream()
    snr, B = 10, 700
    outs = {}
    for poison in POISON:
        rng = np.random.default_rng(3)          # the same pilots for every poison
        h = C.c_void_p()
        if kind in ('dense', 'dense_split'):
            K, N = (12, 64) if kind == 'dense' else (16, 128)
            means, covs, w = orc.random_psd_gmm(K, N, seed=4, mean_scale=0.1)
            prep = precompute.prepare(means, covs, w, np.eye(N), snr, 1)
            sl = _poisoned_arrays([prep[k] for k in ('Linv', 'W', 'zoff', 'hoff', 'logc')], poison)
            _lib.check(lib.qce_model_create(N, N, K, 0, C.byref(h)))
            _lib.check(lib.qce_model_set_params(h, s, *[x.ptr for x in sl], float(prep['data_scale'])))
            create, destroy, est = None, lib.qce_model_destroy, 'dense'
        elif kind == 'circ':
            K, n1, n2 = 64, 16, 16
            N = n1 * n2
            c, covs, w, _ = orc.circulant_gmm(K, n1, n2, seed=4)
            prep = precompute.prepare_circulant(c, w, (n1, n2), snr, 1)
            sl = _poisoned_arrays([prep[k] for k in ('inv_lambda_t', 'gain', 'logc')], poison)
            _lib.check(lib.qce_circ_model_create(n1, n2, K, 0, C.byref(h)))
            _lib.check(lib.qce_circ_model_set_params(h, s, *[x.ptr for x in sl]))
            destroy, est = lib.qce_circ_model_destroy, 'circ'
        elif kind == 'mfa':
            K, N, M = 8, 64, 8
            means, lam, psi, amps = orc.random_mfa(K, N, M, seed=4, mean_scale=0.1)
            qz = orc.get_quantizer([snr], 3, 'lloyd')[snr]
            prep = precompute.prepare_mfa_woodbury(means, lam, psi, amps, snr, 3, 'lloyd', qz)
            sl = _poisoned_arrays([prep[k] for k in ('inv_delta', 'evec', 'D', 'Y', 'm_r', 'mu', 'logc')], poison)
            _lib.check(lib.qce_mfa_model_create(N, M, K, 0, C.byref(h)))
            _lib.check(lib.qce_mfa_model_set_params(h, s, *[x.ptr for x in sl]))
            destroy, est = lib.qce_mfa_model_destroy, 'mfa'
        else:
            N = 64
            bd = torch.from_numpy(0.5 + np.random.default_rng(1).random(N) + 0j)
            X = orc.crandn(N, 2 * N, rng=np.random.default_rng(2))
            cq = torch.from_numpy(X @ X.conj().T / (2 * N))
            sl = _poisoned_arrays([bd, cq], poison)
            _lib.check(lib.qce_rate_model_create(N, C.byref(h)))
            _lib.check(lib.qce_rate_model_set_params(h, s, *[x.ptr for x in sl]))
            destroy, est = lib.qce_rate_model_destroy, 'rate'
        _sync()
        for x in sl:
            x.check(f'set_params {kind} {poison}')
        r = (np.sign(rng.standard_normal((B, N))) + 1j * np.sign(rng.standard_normal((B, N)))) / np.sqrt(2)
        if kind == 'mfa':
            r = rng.choice(orc.get_quantizer([snr], 3, 'lloyd')[snr][1], (B, N)) + 1j * rng.choice(
                orc.get_quantizer([snr], 3, 'lloyd')[snr][1], (B, N))
        rt = torch.from_numpy(r).cuda()
        got = []
        if est == 'rate':
            acc = torch.zeros(5, dtype=torch.float64, device='cuda')
            _lib.check(lib.qce_rate_accumulate(h, s, C.c_void_p(rt.data_ptr()), C.c_void_p(rt.data_ptr()), 0, B,
                                               C.c_void_p(acc.data_ptr())))
            got.append(acc.cpu().numpy())
        else:
            precs = [_lib.PREC_FP64] if est == 'mfa' else [_lib.PREC_FP64, _lib.PREC_TC]
            for p in precs:
                for mode in ('all', 1):
                    md, n_top, rho = engine.parse_mode(mode)
                    out = torch.empty((B, N), dtype=torch.complex128, device='cuda')
                    lp = torch.empty((B, K), dtype=torch.float64, device='cuda')
                    args = (h, s, C.c_void_p(rt.data_ptr()), B, md, n_top, rho)
                    tail = (C.c_void_p(out.data_ptr()), C.c_void_p(lp.data_ptr()), None, None)
                    if est == 'dense':
                        _lib.check(lib.qce_estimate(*args, p, *tail))
                    elif est == 'circ':
                        _lib.check(lib.qce_circ_estimate_prec(*args, p, *tail))
                    else:
                        _lib.check(lib.qce_mfa_estimate(*args, *tail))
                    got += [out.cpu().numpy(), lp.cpu().numpy()]
        _sync()
        destroy(h)
        outs[poison] = got
    for poison in ('nan', 'big'):
        for a, b in zip(outs[poison], outs['zero']):
            assert np.isfinite(b).all(), (kind, poison)
            if kind == 'rate':      # FP64 atomics across CTAs: any order
                np.testing.assert_allclose(a, b, rtol=1e-12, atol=0, err_msg=f'{kind} {poison}')
            else:
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (kind, poison)


# ----------------------------------------------------------------------------------------------------- host-buffer entry points

def _labels(qz, nb):
    return np.array([-1.0, 1.0]) / np.sqrt(2) if nb == 1 else np.asarray(qz[1])


@pytest.mark.gpu
@pytest.mark.parametrize('where', ['host', 'pinned'])
@pytest.mark.parametrize('entry', ['dense_tc', 'dense_fp64', 'codes_c64', 'codes_c128', 'circ_tc', 'mfa'])
def test_host_entry_points_guards(qce, entry, where):
    """The host-buffer entry points on pageable and page-locked slabs, at one chunk - 1, one chunk + 1 and four chunks + 1 (every
    staging slot used, then the first again): guards intact, inputs unchanged, and the estimates of the device entry point."""
    import torch
    from quantized_channel_estimation_b200 import engine
    _lib = _lib_()
    lib = _lib.load()
    name = {'circ_tc': 'circ_tc', 'mfa': 'mfa_ts8'}.get(entry, 'tc_fused')
    d = route_data(name)
    rt = ROUTES[name]
    model = engine_model(qce, name, d['params'])
    No, N, K = model.n_obs, model.n_ant, model.n_comp
    prec = _lib.PREC_FP64 if entry in ('dense_fp64', 'mfa') else _lib.PREC_TC
    codes = entry.startswith('codes')
    out_c64 = entry == 'codes_c64'
    in_row, out_row = (No * 2, N * (8 if out_c64 else 16)) if codes else (No * 16, N * 16)
    widest = max(in_row, out_row, No * 16 if codes else 0, N * 16 if out_c64 else 0)
    sizes = host_batch_sizes(widest)
    rng = np.random.default_rng(9)
    lab = _labels(d['qz'], rt['nb'])
    Bmax = sizes[-1]
    if codes:
        cds = rng.choice(np.array([0, 2], np.uint8), (Bmax, No, 2))
        r_all = ((cds[..., 0].astype(float) - 1) + 1j * (cds[..., 1].astype(float) - 1)) / np.sqrt(2)
        q = engine.Quantizer.get(1)
    else:
        r_all = rng.choice(lab, (Bmax, No)) + 1j * rng.choice(lab, (Bmax, No))
    rdev = torch.from_numpy(r_all).cuda()
    ref_all = torch.empty((Bmax, N), dtype=torch.complex128, device='cuda')
    md, n_top, rho = engine.parse_mode('all')
    args = (C.c_void_p(rdev.data_ptr()), Bmax, md, n_top, rho)
    if rt['kind'] == 'gmm':
        _lib.check(lib.qce_estimate(model.handle, _cur_stream(), *args, prec, C.c_void_p(ref_all.data_ptr()), None, None, None))
    elif rt['kind'] == 'circ':
        _lib.check(lib.qce_circ_estimate_prec(model.handle, _cur_stream(), *args, prec, C.c_void_p(ref_all.data_ptr()), None, None, None))
    else:
        _lib.check(lib.qce_mfa_estimate(model.handle, _cur_stream(), *args, C.c_void_p(ref_all.data_ptr()), None, None, None))
    ref_all = ref_all.cpu().numpy()
    tol = 1e-12 if prec == _lib.PREC_FP64 else (1e-6 if not out_c64 else 1e-5)
    for B in sizes:
        src = cds[:B] if codes else r_all[:B]
        ins = Slab(B, in_row, where).write(src, POISON['nan'])
        outs = Slab(B, out_row, where)
        if entry in ('dense_tc', 'dense_fp64'):
            st = lib.qce_estimate_host(model.handle, ins.ptr, B, md, n_top, rho, prec, outs.ptr)
        elif codes:
            st = lib.qce_estimate_host_codes(model.handle, q.handle, ins.ptr, B, md, n_top, rho, prec, outs.ptr, int(out_c64))
        elif entry == 'circ_tc':
            st = lib.qce_circ_estimate_host(model.handle, ins.ptr, B, md, n_top, rho, prec, outs.ptr)
        else:
            st = lib.qce_mfa_estimate_host(model.handle, ins.ptr, B, md, n_top, rho, outs.ptr)
        _lib.check(st)
        ins.check(f'{entry} {where} B={B} input')
        outs.check(f'{entry} {where} B={B} output')
        est = outs.read(np.complex64 if out_c64 else np.complex128).reshape(B, N).astype(np.complex128)
        ref = ref_all[:B]
        per = np.linalg.norm(est - ref, axis=1) / np.linalg.norm(ref, axis=1)
        assert np.isfinite(est).all() and per.max() < tol, (entry, where, B, per.max(), int(np.argmax(per)))
        del ins, outs


# ----------------------------------------------------------------------------------------------------- stream history

HISTORY_TARGETS = [n for n in BOUND_ROUTES if route_spec(n)['prec'] == 'tc']


@contextmanager
def fresh_stream():
    """A stream whose handle carries no tensor-core scratch of the library (qce_last_fix_count = -1).  The runtime may hand out the
    handle of a destroyed stream again, and the library keys its scratch by handle: streams are created -- and kept until the end, so
    that no handle repeats -- until one is new to the library."""
    lib = _lib_().load()
    rt = C.CDLL('libcudart.so.12')          # the runtime libqce_b200.so is linked against, already loaded
    made = []
    try:
        for _ in range(256):
            s = C.c_void_p()
            assert rt.cudaStreamCreateWithFlags(C.byref(s), 1) == 0          # cudaStreamNonBlocking
            made.append(s)
            if lib.qce_last_fix_count(s) == -1:
                break
        else:
            pytest.fail('no stream handle new to the library among 256')
        yield made[-1]
    finally:
        for s in made:
            rt.cudaStreamSynchronize(s)
            rt.cudaStreamDestroy(s)
PREDECESSORS = ['large_offgrid_nan', 'wide_tiles', 'pair_top4', 'format_other', 'staging_release']


def _predecessor(qce, what, target, s):
    """Enqueue the predecessor call on stream ``s``."""
    import torch
    from quantized_channel_estimation_b200 import engine, precompute
    _lib = _lib_()
    lib = _lib.load()
    keep = []
    B = 20000
    if what == 'large_offgrid_nan':
        cs = target
        reps = -(-B // cs.r.shape[0])
        r = np.tile(cs.r, (reps, 1))[:B].copy()
        r[::997, 0] = 0.123                      # off the quantiser grid
        r[5::1499, 1] = np.nan
        rt = torch.from_numpy(r).cuda()
        ht = torch.from_numpy(np.tile(cs.h, (reps, 1))[:B].copy()).cuda()
        out = torch.empty((B, cs.N), dtype=torch.complex128, device='cuda')
        lp = torch.empty((B, cs.K), dtype=torch.float64, device='cuda')
        acc = torch.zeros(3, dtype=torch.float64, device='cuda')
        keep += [rt, ht, out, lp, acc]
        torch.cuda.synchronize()
        md, n_top, rho = engine.parse_mode(3)
        fn = lib.qce_estimate if cs.kind == 'gmm' else lib.qce_circ_estimate_prec
        _lib.check(fn(cs.model.handle, s, C.c_void_p(rt.data_ptr()), B, md, n_top, rho, _lib.PREC_TC, C.c_void_p(out.data_ptr()),
                      C.c_void_p(lp.data_ptr()), C.c_void_p(ht.data_ptr()), C.c_void_p(acc.data_ptr())))
    elif what == 'wide_tiles':
        K, N, snr = 12, 128, 10
        means, covs, w = orc.random_psd_gmm(K, N, seed=31, mean_scale=0.1)
        qz = orc.get_quantizer([snr], 3, 'lloyd')[snr]
        model = engine.DenseModel(precompute.prepare(means, covs, w, np.eye(N), snr, 3, 'lloyd', qz))
        rng = np.random.default_rng(32)
        r = rng.choice(qz[1], (B, N)) + 1j * rng.choice(qz[1], (B, N))
        rt = torch.from_numpy(r).cuda()
        out = torch.empty((B, N), dtype=torch.complex128, device='cuda')
        lp = torch.empty((B, K), dtype=torch.float64, device='cuda')
        keep += [model, rt, out, lp]
        torch.cuda.synchronize()
        for mode in ('all', 1):
            md, n_top, rho = engine.parse_mode(mode)
            _lib.check(lib.qce_estimate(model.handle, s, C.c_void_p(rt.data_ptr()), B, md, n_top, rho, _lib.PREC_TC,
                                        C.c_void_p(out.data_ptr()), C.c_void_p(lp.data_ptr()), None, None))
    elif what == 'pair_top4':
        d = route_data('tc_split_pairs')
        model = engine_model(qce, 'tc_split_pairs', d['params'])
        rt = torch.from_numpy(d['r']).cuda()
        out = torch.empty((rt.shape[0], model.n_ant), dtype=torch.complex128, device='cuda')
        keep += [model, rt, out]
        torch.cuda.synchronize()
        md, n_top, rho = engine.parse_mode(4)
        _lib.check(lib.qce_estimate(model.handle, s, C.c_void_p(rt.data_ptr()), rt.shape[0], md, n_top, rho, _lib.PREC_TC,
                                    C.c_void_p(out.data_ptr()), None, None, None))
    elif what == 'format_other':
        other = case(qce, 'tc_three_pass' if target.name != 'tc_three_pass' else 'tc_fused')
        reps = -(-B // other.r.shape[0])
        rt = torch.from_numpy(np.tile(other.r, (reps, 1))[:B].copy()).cuda()
        keep += [rt]
        torch.cuda.synchronize()
        _lib.check(lib.qce_format_pilots(other.model.handle, s, C.c_void_p(rt.data_ptr()), B))
    else:
        lib.qce_host_staging_release()
    return keep


@pytest.mark.gpu
@pytest.mark.parametrize('name', HISTORY_TARGETS)
def test_result_does_not_depend_on_stream_history(qce, name):
    """A small ragged batch on a stream after each predecessor equals the same call on a stream new to the library: estimates and
    log-probabilities bit for bit, the accumulators to 1e-12 (FP64 atomics add in any order), the same fix count.  Routes with a
    pair-bucketed combination also run a ragged batch that takes it, compared to 1e-6 per row (FP32 atomics)."""
    from test_stream_scratch import raw_stream
    cs = case(qce, name)
    B = cs.rt['U'] + cs.rt['T'] + 3
    calls = [('all', False, B), (1, False, B), (3, True, B)]
    calls += [(m, False, Bx) for Bx, ms in BOUND_ROUTES[name].get('extra', []) for m in ms if pair_call(cs.rt, Bx, m)]

    def target(s):
        return [run_estimate(cs, Bc, mode, stream=s, logp=lp) for mode, lp, Bc in calls]

    _sync()
    with fresh_stream() as fresh:
        ref = target(fresh)
    for what in PREDECESSORS:
        _sync()
        with raw_stream() as s:
            keep = _predecessor(qce, what, cs, s)
            got = target(s)
            del keep
        for (mode, _, Bc), a, b in zip(calls, got, ref):
            same_outputs(a, b, (name, what, mode, Bc), fp32_rows=pair_call(cs.rt, Bc, mode))
    for (mode, _, Bc), out in zip(calls, ref):
        check_against_oracle(cs, Bc, mode, out)
    assert any(pair_call(cs.rt, Bc, m) for m, _, Bc in calls) == (name in ('tc_split_pairs', 'tc_n256_split'))
