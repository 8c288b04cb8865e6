"""Thin host-side wrappers over the C ABI (include/qce_b200.h): quantiser and model handles,
argument marshalling from torch CUDA tensors / numpy arrays.  All compute happens in
libqce_b200.so; nothing here falls back to the CPU."""
import ctypes as C

import numpy as np
import torch

from . import _lib

PRECISIONS = {'fp64': _lib.PREC_FP64, 'tc': _lib.PREC_TC}


def parse_mode(n_summands_or_proba):
    """Dispatch of ``n_summands_or_proba`` exactly as the reference tests it (gmm:197, :220, :229):
    ``isinstance(x, int)`` first (so ``np.int64(3)`` takes the probability branch), then ``== 'all'``,
    anything else is a cumulative probability."""
    x = n_summands_or_proba
    if isinstance(x, int):
        if x == 1:
            return _lib.MODE_TOP1, 1, 0.0
        return _lib.MODE_TOPN, int(x), 0.0
    if isinstance(x, str):
        if x == 'all':
            return _lib.MODE_ALL, 0, 0.0
        raise ValueError(f"n_summands_or_proba = {x!r} is neither an int, 'all' nor a probability")
    return _lib.MODE_CUMPROB, 0, float(x)


def tc_shape_ok(n_obs, n_ant, on_grid=False):
    """Shapes the tensor-core kernels are instantiated for (mirrors tc_instantiated / tc_split_shape / tc_supported in
    qce_dense_tc.cu).  ``on_grid``: the pilots lie on an integer grid (``data_scale > 0``: 1 bit, or uniform b bit).  n_obs = 256
    (one pilot per antenna on 256 antennas, or two pilots on 128) takes only such pilots; off the grid it runs on the complex128
    kernel."""
    if n_obs % 16 or n_ant % 16:
        return False
    if n_obs <= 64 and n_ant <= 64:
        return n_obs == n_ant or (n_obs, n_ant) in ((64, 32), (32, 16))
    if on_grid and (n_obs, n_ant) in ((256, 128), (256, 256)):
        return True
    return (n_obs, n_ant) in ((128, 64), (128, 128), (96, 48), (96, 96))


def tc_padded_shape(n_obs, n_ant, on_grid=False):
    """Smallest tensor-core shape that holds an (n_obs, n_ant) model after zero padding (None: there is none).  Padded rows / columns
    of the parameter blocks are zero, padded pilot entries are zero: they add exact zeros to the quadratic forms and produce estimate
    entries that are cut off again.  ``on_grid`` as for ``tc_shape_ok``: only on-grid models are padded up to n_obs = 256."""
    if tc_shape_ok(n_obs, n_ant, on_grid):
        return n_obs, n_ant
    sizes = (16, 32, 48, 64, 96, 128, 256)
    cands = [(o, a) for o in sizes for a in sizes
             if o >= n_obs and a >= n_ant and tc_shape_ok(o, a, on_grid)]
    return min(cands, key=lambda c: c[0] * (c[0] + c[1])) if cands else None


def _pad_prep(prep, No_p, N_p):
    """Zero-pad the parameter blocks of ``precompute.prepare`` to (No_p, N_p)."""
    K, No, N = int(prep['n_comp']), int(prep['n_obs']), int(prep['n_ant'])
    out = dict(prep)
    dev = prep['Linv'].device

    def z(*shape):
        return torch.zeros(shape, dtype=torch.complex128, device=dev)
    Linv, W, zoff, hoff = z(K, No_p, No_p), z(K, N_p, No_p), z(K, No_p), z(K, N_p)
    Linv[:, :No, :No] = prep['Linv']
    W[:, :N, :No] = prep['W']
    zoff[:, :No] = prep['zoff']
    hoff[:, :N] = prep['hoff']
    out.update(Linv=Linv, W=W, zoff=zoff, hoff=hoff, n_obs=No_p, n_ant=N_p)
    return out


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _as_c128_cuda(x, name):
    if not (isinstance(x, torch.Tensor) and x.is_cuda):
        raise TypeError(f'{name} must be a torch CUDA tensor')
    if x.dtype != torch.complex128:
        x = x.to(torch.complex128)
    return x.contiguous()


class Quantizer:
    """Device-resident quantiser tables (qce_quantizer)."""
    _cache = {}

    def __init__(self, n_bits, thresholds=None, labels=None):
        lib = _lib.require_device()
        self.n_bits = int(n_bits)
        self.handle = C.c_void_p()
        if self.n_bits == 1:
            _lib.check(lib.qce_quantizer_create(1, None, None, C.byref(self.handle)))
        else:
            thr = np.ascontiguousarray(np.asarray(thresholds, dtype=np.float64))
            lab = np.ascontiguousarray(np.asarray(labels, dtype=np.float64))
            if thr.size != 2 ** self.n_bits - 1 or lab.size != 2 ** self.n_bits:
                raise ValueError('quantiser tables must have 2^b - 1 thresholds and 2^b labels')
            _lib.check(lib.qce_quantizer_create(self.n_bits, thr.ctypes.data_as(C.c_void_p),
                                                lab.ctypes.data_as(C.c_void_p), C.byref(self.handle)))

    def __del__(self):
        try:
            if getattr(self, 'handle', None) and self.handle.value:
                _lib.load().qce_quantizer_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    @classmethod
    def get(cls, n_bits, thresholds=None, labels=None):
        key = (int(n_bits),) if int(n_bits) == 1 else (
            int(n_bits), np.asarray(thresholds, dtype=np.float64).tobytes(), np.asarray(labels, dtype=np.float64).tobytes())
        q = cls._cache.get(key)
        if q is None:
            if len(cls._cache) > 64:
                cls._cache.clear()
            q = cls._cache[key] = cls(n_bits, thresholds, labels)
        return q

    def quantize(self, y, want_codes=False):
        """``y`` c128 CUDA tensor -> quantised tensor (and uint8 level codes ``[..., 2]``)."""
        y = _as_c128_cuda(y, 'y')
        r = torch.empty_like(y)
        codes = torch.empty(y.shape + (2,), dtype=torch.uint8, device=y.device) if want_codes else None
        with torch.cuda.device(y.device):
            _lib.check(_lib.load().qce_quantize(self.handle, _stream(), _ptr(y), y.numel(), _ptr(r), _ptr(codes)))
        return (r, codes) if want_codes else r


def observe_quantize(h, noise, noise_scale, quantizer=None, want_y=False, want_codes=False):
    """``y = h + noise_scale * noise`` then quantise (A = I), one kernel.  ``h`` c64/c128 CUDA, ``noise`` c128."""
    lib = _lib.require_device()
    if not (isinstance(h, torch.Tensor) and h.is_cuda):
        raise TypeError('h must be a torch CUDA tensor')
    h_c64 = h.dtype == torch.complex64
    if not h_c64:
        h = h.to(torch.complex128)
    h = h.contiguous()
    noise = _as_c128_cuda(noise, 'noise')
    if noise.shape != h.shape:
        raise ValueError('noise and h must have the same shape')
    y = torch.empty(h.shape, dtype=torch.complex128, device=h.device) if (want_y or quantizer is None) else None
    r = torch.empty(h.shape, dtype=torch.complex128, device=h.device) if quantizer is not None else None
    codes = torch.empty(h.shape + (2,), dtype=torch.uint8, device=h.device) if (want_codes and quantizer is not None) else None
    with torch.cuda.device(h.device):
        _lib.check(lib.qce_observe_quantize(quantizer.handle if quantizer is not None else None, _stream(), _ptr(h),
                                            int(h_c64), _ptr(noise), float(noise_scale), h.numel(), _ptr(y), _ptr(r),
                                            _ptr(codes)))
    return y, r, codes


class DenseModel:
    """One (SNR, bit width, quantiser) parameter set resident on the GPU (qce_model)."""

    def __init__(self, prep, flags=0, pad=False):
        """``pad=True``: a shape the tensor-core kernels are not instantiated for (n_obs / n_ant not multiples of 16, or an unlisted
        pair) is zero-padded to the next one that is, instead of running on the complex128 kernel (~100x slower)."""
        lib = _lib.require_device()
        self.n_obs, self.n_ant, self.n_comp = int(prep['n_obs']), int(prep['n_ant']), int(prep['n_comp'])
        self.pad_obs, self.pad_ant = self.n_obs, self.n_ant          # shape of the library handle
        on_grid = float(prep['data_scale']) > 0
        if pad and not tc_shape_ok(self.n_obs, self.n_ant, on_grid):
            ps = tc_padded_shape(self.n_obs, self.n_ant, on_grid)
            if ps is not None:
                self.pad_obs, self.pad_ant = ps
        self.handle = C.c_void_p()
        _lib.check(lib.qce_model_create(self.pad_obs, self.pad_ant, self.n_comp, int(flags), C.byref(self.handle)))
        self.device = torch.device('cuda', torch.cuda.current_device())
        self.update(prep)

    @property
    def padded(self):
        return (self.pad_obs, self.pad_ant) != (self.n_obs, self.n_ant)

    def update(self, prep):
        """(Re)load the parameter blocks of ``precompute.prepare`` (same shape): ``fit()`` calls this once per EM iteration."""
        if self.padded:
            prep = _pad_prep(prep, self.pad_obs, self.pad_ant)
        t = {k: prep[k].to(self.device).contiguous() for k in ('Linv', 'W', 'zoff', 'hoff', 'logc')}
        assert t['Linv'].dtype == torch.complex128 and t['logc'].dtype == torch.float64
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().qce_model_set_params(self.handle, _stream(), _ptr(t['Linv']), _ptr(t['W']), _ptr(t['zoff']),
                                                        _ptr(t['hoff']), _ptr(t['logc']), float(prep['data_scale'])))
            torch.cuda.current_stream().synchronize()      # the library copied the blocks; t may now be freed

    def _pad_in(self, r):
        if self.pad_obs == self.n_obs:
            return r
        out = torch.zeros((r.shape[0], self.pad_obs), dtype=r.dtype, device=r.device)
        out[:, :self.n_obs] = r
        return out

    def __del__(self):
        try:
            if getattr(self, 'handle', None) and self.handle.value:
                _lib.load().qce_model_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    def _precision(self, precision, mode):
        if precision in ('fp64', 'tc'):
            return [PRECISIONS[precision]]
        if precision == 'auto':
            return [_lib.PREC_TC, _lib.PREC_FP64]      # TC when the shape/mode is supported, else complex128 CUDA
        raise ValueError(f'unknown precision {precision!r}')

    def _call(self, precision, mode, fn):
        precs = self._precision(precision, mode)
        for i, p in enumerate(precs):
            st = fn(p)
            if st == _lib.ERR_UNSUPPORTED and i + 1 < len(precs):
                continue
            _lib.check(st)
            return

    def estimate(self, r, n_summands_or_proba='all', precision='auto', want_logp=False, h_true=None):
        """r: CUDA c128 [B, n_obs] -> h_est CUDA c128 [B, n_ant] (and l [B,K], and NMSE accumulators)."""
        mode, n_top, rho = parse_mode(n_summands_or_proba)
        r = _as_c128_cuda(r, 'y')
        if r.dim() != 2 or r.shape[1] != self.n_obs:
            raise ValueError(f'y must be [B, {self.n_obs}]')
        B = r.shape[0]
        r = self._pad_in(r)
        h_est = torch.empty((B, self.pad_ant), dtype=torch.complex128, device=r.device)
        logp = torch.empty((B, self.n_comp), dtype=torch.float64, device=r.device) if want_logp else None
        acc = None
        if h_true is not None:
            h_true = _as_c128_cuda(h_true, 'h_true')
            if self.pad_ant != self.n_ant:
                ht = torch.zeros((B, self.pad_ant), dtype=h_true.dtype, device=h_true.device)
                ht[:, :self.n_ant] = h_true
                h_true = ht
            acc = torch.zeros(3, dtype=torch.float64, device=r.device)
        lib = _lib.load()
        with torch.cuda.device(r.device):
            self._call(precision, mode, lambda p: lib.qce_estimate(self.handle, _stream(), _ptr(r), B, mode, n_top, rho, p,
                                                                   _ptr(h_est), _ptr(logp), _ptr(h_true), _ptr(acc)))
        if self.pad_ant != self.n_ant:
            h_est = h_est[:, :self.n_ant].contiguous()
        out = (h_est,)
        if want_logp:
            out += (logp,)
        if h_true is not None:
            out += (acc,)
        return out if len(out) > 1 else h_est

    def log_prob(self, r, precision='auto'):
        """Weighted log-probabilities ``l [B, K]`` float64 only (no estimate: the library skips the combination launches)."""
        r = _as_c128_cuda(r, 'y')
        if r.dim() != 2 or r.shape[1] != self.n_obs:
            raise ValueError(f'y must be [B, {self.n_obs}]')
        B = r.shape[0]
        r = self._pad_in(r)
        logp = torch.empty((B, self.n_comp), dtype=torch.float64, device=r.device)
        lib = _lib.load()
        with torch.cuda.device(r.device):
            self._call(precision, _lib.MODE_ALL, lambda p: lib.qce_estimate(self.handle, _stream(), _ptr(r), B, _lib.MODE_ALL, 0, 0.0, p,
                                                                            None, _ptr(logp), None, None))
        return logp

    def estimate_host(self, r, n_summands_or_proba='all', precision='auto'):
        """r: numpy c128 [B, n_obs] (host) -> numpy c128 [B, n_ant]; copies run inside the library."""
        mode, n_top, rho = parse_mode(n_summands_or_proba)
        r = np.ascontiguousarray(np.asarray(r, dtype=np.complex128))
        if r.ndim != 2 or r.shape[1] != self.n_obs:
            raise ValueError(f'y must be [B, {self.n_obs}]')
        if self.padded:       # padded models: pad on the device (the host path of the library moves whole rows)
            est = self.estimate(torch.from_numpy(r).to(self.device), n_summands_or_proba, precision)
            return est.cpu().numpy()
        out = np.empty((r.shape[0], self.n_ant), dtype=np.complex128)
        lib = _lib.load()
        with torch.cuda.device(self.device):
            self._call(precision, mode, lambda p: lib.qce_estimate_host(self.handle, r.ctypes.data_as(C.c_void_p), r.shape[0],
                                                                        mode, n_top, rho, p, out.ctypes.data_as(C.c_void_p)))
        return out

    def estimate_host_codes(self, codes, quantizer, n_summands_or_proba='all', precision='auto', out_dtype=np.complex64):
        """Compact host transfer formats: ``codes`` uint8 ``[B, n_obs, 2]`` (level indices per real dimension, as ``Quantizer.quantize(...,
        want_codes=True)`` returns them) -> estimates ``[B, n_ant]`` complex64 (default) or complex128 on the host."""
        mode, n_top, rho = parse_mode(n_summands_or_proba)
        codes = np.ascontiguousarray(np.asarray(codes, dtype=np.uint8))
        if codes.ndim != 3 or codes.shape[1:] != (self.n_obs, 2):
            raise ValueError(f'codes must be [B, {self.n_obs}, 2] uint8')
        if self.padded:
            raise ValueError('estimate_host_codes(): zero-padded models are not supported')
        out_dtype = np.dtype(out_dtype)
        if out_dtype not in (np.dtype(np.complex64), np.dtype(np.complex128)):
            raise ValueError('out_dtype must be complex64 or complex128')
        out = np.empty((codes.shape[0], self.n_ant), dtype=out_dtype)
        lib = _lib.load()
        with torch.cuda.device(self.device):
            self._call(precision, mode, lambda p: lib.qce_estimate_host_codes(self.handle, quantizer.handle, codes.ctypes.data_as(C.c_void_p),
                                                                              codes.shape[0], mode, n_top, rho, p, out.ctypes.data_as(C.c_void_p),
                                                                              int(out_dtype == np.dtype(np.complex64))))
        return out

    def pipeline(self, quantizer, h, noise, noise_scale, n_summands_or_proba='all', precision='auto', want_est=False,
                 acc=None):
        """observe -> quantise -> estimate -> NMSE accumulators for device-resident channels (A = I)."""
        mode, n_top, rho = parse_mode(n_summands_or_proba)
        if self.padded:
            raise ValueError('pipeline(): zero-padded models are not supported (create the DenseModel with pad=False)')
        h_c64 = h.dtype == torch.complex64
        if not h_c64:
            h = h.to(torch.complex128)
        h = h.contiguous()
        noise = _as_c128_cuda(noise, 'noise')
        B = h.shape[0]
        if acc is None:
            acc = torch.zeros(3, dtype=torch.float64, device=h.device)
        h_est = torch.empty((B, self.n_ant), dtype=torch.complex128, device=h.device) if want_est else None
        lib = _lib.load()
        with torch.cuda.device(h.device):
            self._call(precision, mode, lambda p: lib.qce_pipeline(self.handle, quantizer.handle, _stream(), _ptr(h), int(h_c64),
                                                                   _ptr(noise), float(noise_scale), B, mode, n_top, rho, p,
                                                                   _ptr(h_est), _ptr(acc)))
        return (h_est, acc) if want_est else acc


class CircModel:
    """Circulant / block-circulant parameter set on the GPU (qce_circ_model); zero means, A = I."""

    def __init__(self, prep, flags=0):
        lib = _lib.require_device()
        self.n_obs = self.n_ant = int(prep['n_ant'])
        self.n_comp = int(prep['n_comp'])
        self.handle = C.c_void_p()
        _lib.check(lib.qce_circ_model_create(int(prep['n1']), int(prep['n2']), self.n_comp, int(flags), C.byref(self.handle)))
        dev = torch.device('cuda', torch.cuda.current_device())
        t = {k: prep[k].to(dev).contiguous() for k in ('inv_lambda_t', 'gain', 'logc')}
        _lib.check(lib.qce_circ_model_set_params(self.handle, _stream(), _ptr(t['inv_lambda_t']), _ptr(t['gain']), _ptr(t['logc'])))
        torch.cuda.current_stream().synchronize()
        self.device = dev

    def __del__(self):
        try:
            if getattr(self, 'handle', None) and self.handle.value:
                _lib.load().qce_circ_model_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    def estimate(self, r, n_summands_or_proba='all', precision='auto', want_logp=False, h_true=None):
        mode, n_top, rho = parse_mode(n_summands_or_proba)
        r = _as_c128_cuda(r, 'y')
        if r.dim() != 2 or r.shape[1] != self.n_obs:
            raise ValueError(f'y must be [B, {self.n_obs}]')
        B = r.shape[0]
        h_est = torch.empty((B, self.n_ant), dtype=torch.complex128, device=r.device)
        logp = torch.empty((B, self.n_comp), dtype=torch.float64, device=r.device) if want_logp else None
        acc = None
        if h_true is not None:
            h_true = _as_c128_cuda(h_true, 'h_true')
            acc = torch.zeros(3, dtype=torch.float64, device=r.device)
        with torch.cuda.device(r.device):
            self._run(precision, (_stream(), _ptr(r), B, mode, n_top, rho), (_ptr(h_est), _ptr(logp), _ptr(h_true), _ptr(acc)))
        out = (h_est,)
        if want_logp:
            out += (logp,)
        if h_true is not None:
            out += (acc,)
        return out if len(out) > 1 else h_est

    def log_prob(self, r, precision='auto'):
        return self.estimate(r, 'all', precision, want_logp=True)[1]

    def _run(self, precision, head, tail):
        """'fp64': complex128 kernel; 'tc': FP32-FFT / tensor-core kernel (16 x 16 blocks, K = 64 or 128); 'auto': the latter
        when the shape is supported."""
        lib = _lib.load()
        if precision not in ('fp64', 'tc', 'auto'):
            raise ValueError(f'unknown precision {precision!r}')
        if precision != 'fp64':
            st = lib.qce_circ_estimate_prec(self.handle, *head, _lib.PREC_TC, *tail)
            if not (st == _lib.ERR_UNSUPPORTED and precision == 'auto'):
                _lib.check(st)
                return
        _lib.check(lib.qce_circ_estimate_prec(self.handle, *head, _lib.PREC_FP64, *tail))

    def estimate_host(self, r, n_summands_or_proba='all', precision='auto'):
        """r: numpy c128 [B, n_ant] (host) -> numpy c128 [B, n_ant]; chunked, overlapped copies inside the library."""
        mode, n_top, rho = parse_mode(n_summands_or_proba)
        r = np.ascontiguousarray(np.asarray(r, dtype=np.complex128))
        if r.ndim != 2 or r.shape[1] != self.n_obs:
            raise ValueError(f'y must be [B, {self.n_obs}]')
        out = np.empty((r.shape[0], self.n_ant), dtype=np.complex128)
        with torch.cuda.device(self.device):
            self._run_host(precision, r.ctypes.data_as(C.c_void_p), r.shape[0], mode, n_top, rho, out.ctypes.data_as(C.c_void_p))
        return out

    def _run_host(self, precision, r_ptr, B, mode, n_top, rho, out_ptr):
        lib = _lib.load()
        if precision not in ('fp64', 'tc', 'auto'):
            raise ValueError(f'unknown precision {precision!r}')
        if precision != 'fp64':
            st = lib.qce_circ_estimate_host(self.handle, r_ptr, B, mode, n_top, rho, _lib.PREC_TC, out_ptr)
            if not (st == _lib.ERR_UNSUPPORTED and precision == 'auto'):
                _lib.check(st)
                return
        _lib.check(lib.qce_circ_estimate_host(self.handle, r_ptr, B, mode, n_top, rho, _lib.PREC_FP64, out_ptr))


class RateModel:
    """Accumulators of the scripts' achievable-rate lower bound (qce_rate_model): ``utils.rate_lower_bound`` as five sums that add
    across batches and ranks, so that the bound needs no stored estimates.  ``buss`` is the ``[N, N]`` Bussgang matrix of the global
    model (must be diagonal), ``Cq`` the ``[N, N]`` quantisation-noise covariance ``C_r - B C B^H`` (``utils.rate_params`` builds
    both); 1 <= N <= 256."""

    def __init__(self, buss, Cq):
        lib = _lib.require_device()
        buss = torch.as_tensor(buss).to(torch.complex128)
        Cq = torch.as_tensor(Cq).to(torch.complex128)
        if buss.dim() != 2 or buss.shape[0] != buss.shape[1] or Cq.shape != buss.shape:
            raise ValueError('buss and Cq must both be [N, N]')
        diag = torch.diagonal(buss)
        if bool((buss - torch.diag_embed(diag)).abs().max() != 0):
            raise ValueError('buss must be diagonal (utils.rate_lower_bound handles a full Bussgang matrix)')
        self.n_ant = int(buss.shape[0])
        self.handle = C.c_void_p()
        _lib.check(lib.qce_rate_model_create(self.n_ant, C.byref(self.handle)))
        self.device = torch.device('cuda', torch.cuda.current_device())
        d, cq = diag.to(self.device).contiguous(), Cq.to(self.device).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(lib.qce_rate_model_set_params(self.handle, _stream(), _ptr(d), _ptr(cq)))
            torch.cuda.current_stream().synchronize()      # the library copied / packed them; d and cq may now be freed

    def __del__(self):
        try:
            if getattr(self, 'handle', None) and self.handle.value:
                _lib.load().qce_rate_model_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    def accumulate(self, h_est, h_true, acc=None):
        """Add ``{sum Re inner, sum Im inner, sum |inner|^2, sum Re g^H C_q g, B}`` of the estimates ``h_est [B, N]`` (CUDA, complex128)
        and channels ``h_true [B, N]`` (CUDA, complex64 or complex128) into ``acc`` (float64 ``[5]`` on the device, zeros if None) and
        return it.  ``utils.rate_from_accumulators(acc)`` is the bound."""
        h_est = _as_c128_cuda(h_est, 'h_est')
        if not (isinstance(h_true, torch.Tensor) and h_true.is_cuda):
            raise TypeError('h_true must be a torch CUDA tensor')
        h_c64 = h_true.dtype == torch.complex64
        h_true = (h_true if h_c64 else h_true.to(torch.complex128)).contiguous()
        if h_est.dim() != 2 or h_est.shape[1] != self.n_ant or h_true.shape != h_est.shape:
            raise ValueError(f'h_est and h_true must both be [B, {self.n_ant}]')
        if acc is None:
            acc = torch.zeros(5, dtype=torch.float64, device=h_est.device)
        elif not (isinstance(acc, torch.Tensor) and acc.is_cuda and acc.dtype == torch.float64 and acc.numel() == 5 and acc.is_contiguous()):
            raise TypeError('acc must be a contiguous float64 CUDA tensor of 5 elements')
        with torch.cuda.device(h_est.device):
            _lib.check(_lib.load().qce_rate_accumulate(self.handle, _stream(), _ptr(h_est), _ptr(h_true), int(h_c64), h_est.shape[0],
                                                       _ptr(acc)))
        return acc


class MfaModel(CircModel):
    """Woodbury-form MFA parameter set on the GPU (qce_mfa_model); A = I, n_bits > 1 or infinite resolution."""

    def __init__(self, prep, flags=0):          # noqa: D107  (does not call CircModel.__init__: different handle type)
        lib = _lib.require_device()
        self.n_obs = self.n_ant = int(prep['n_ant'])
        self.n_comp = int(prep['n_comp'])
        self.handle = C.c_void_p()
        _lib.check(lib.qce_mfa_model_create(self.n_ant, int(prep['latent']), self.n_comp, int(flags), C.byref(self.handle)))
        dev = torch.device('cuda', torch.cuda.current_device())
        names = ('inv_delta', 'evec', 'D', 'Y', 'm_r', 'mu', 'logc')
        t = [prep[k].to(dev).contiguous() for k in names]
        _lib.check(lib.qce_mfa_model_set_params(self.handle, _stream(), *[_ptr(x) for x in t]))
        torch.cuda.current_stream().synchronize()
        self.device = dev

    def __del__(self):
        try:
            if getattr(self, 'handle', None) and self.handle.value:
                _lib.load().qce_mfa_model_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    def _run(self, precision, head, tail):          # complex128 only
        if precision not in ('fp64', 'tc', 'auto'):
            raise ValueError(f'unknown precision {precision!r}')
        _lib.check(_lib.load().qce_mfa_estimate(self.handle, *head, *tail))

    def _run_host(self, precision, r_ptr, B, mode, n_top, rho, out_ptr):
        if precision not in ('fp64', 'tc', 'auto'):
            raise ValueError(f'unknown precision {precision!r}')
        _lib.check(_lib.load().qce_mfa_estimate_host(self.handle, r_ptr, B, mode, n_top, rho, out_ptr))
