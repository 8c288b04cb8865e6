"""Drop-in for the quantiser pieces of the reference's ``modules/utils.py``: ``quant`` (:189-203),
``get_observation_nbit`` (:241-251), ``crandn`` (:13-14), ``get_quantizer`` / ``get_quantizer_gauss``
(:531-590), ``cplx_1bit`` (:527-528), ``mse`` (:617-618), ``get_pilot_matrix`` semantics (:337-367).

Array arguments may be torch CUDA tensors (results stay on the GPU) or numpy arrays (staged to
the GPU and returned as numpy, like the reference).  The element-wise work runs in the CUDA kernels of
libqce_b200.so; there is no CPU implementation here."""
import numpy as np
import torch

from . import engine
from .lloyd_max_quantizer import load_quantizer
from .uniform_quantizer import get_uniform_quant_step

_rng = np.random.default_rng()


def crandn(*arg, rng=None):
    """Circularly-symmetric complex standard normal draw (reference :13-14)."""
    rng = _rng if rng is None else rng
    return np.sqrt(0.5) * (rng.standard_normal(arg) + 1j * rng.standard_normal(arg))


def _is_inf(n_bits):
    return n_bits == 'inf' or n_bits == np.inf


def _to_cuda(x, dtype=None):
    if isinstance(x, torch.Tensor):
        t = x if x.is_cuda else x.cuda()
    else:
        t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return t if dtype is None or t.dtype == dtype else t.to(dtype)


def _like_input(t, proto):
    if isinstance(proto, torch.Tensor):
        return t if proto.is_cuda else t.cpu()
    return t.cpu().numpy()


def quant(inp, n_bits=1, thresholds=None, quant_labels=None):
    """Quantise real and imaginary parts independently (reference :189-203), bit-exact."""
    q = engine.Quantizer.get(n_bits, thresholds, quant_labels)
    y = _to_cuda(inp, torch.complex128)
    return _like_input(q.quantize(y), inp)


def cplx_1bit(inp):
    return quant(inp, 1)


def get_observation_nbit(h, snr, A=None, n_bits=1, thresholds=None, cluster=None, agc=False, noise=None):
    """``Q(A h + 10^(-snr/20) n)`` (reference :241-251).  ``noise`` lets the caller supply the draw
    ``n = crandn(*y.shape)`` (the reference takes it from a module-global unseeded generator); ``h`` is
    ``[B, N]``.  With ``A=None`` (all scripts) the synthesis and the quantiser are one fused kernel."""
    ht = _to_cuda(h)
    if not ht.is_complex():
        ht = ht.to(torch.complex128)
    if A is not None:
        At = _to_cuda(A, torch.complex128)
        ht = (ht.to(torch.complex128) @ At.T).contiguous()          # y = A h (plumbing GEMM, cuBLAS)
    if noise is None:
        noise = crandn(*ht.shape)
    nt = _to_cuda(noise, torch.complex128)
    scale = 10 ** (-snr / 20)
    if _is_inf(n_bits):
        y, _, _ = engine.observe_quantize(ht, nt, scale, None)
        return _like_input(y, h)
    q = engine.Quantizer.get(n_bits, thresholds, cluster)
    _, r, _ = engine.observe_quantize(ht, nt, scale, q)
    return _like_input(r, h)


def get_quantizer(snrs, n_bits, quantizer_type='uniform'):
    """Threshold / label tables per SNR: ``{snr: (thresholds, labels, rho_or_None)}`` (reference :531-562).
    1 bit and infinite resolution need no table."""
    quantizer = {}
    if _is_inf(n_bits) or n_bits == 1:
        return {snr: (None, None, None) for snr in snrs}
    levels = int(2 ** n_bits)
    half = (levels - 2) // 2
    for snr in snrs:
        if quantizer_type == 'uniform':
            step = get_uniform_quant_step(snr, n_bits)
            thresholds = np.zeros(levels - 1)
            for nb in range(half):
                thresholds[nb] = -((levels - 2) / 2 - nb) * step
                thresholds[-nb - 1] = ((levels - 2) / 2 - nb) * step
            labels = np.empty(levels)
            labels[:-1] = thresholds - step / 2
            labels[-1] = thresholds[-1] + step / 2
            quantizer[snr] = (thresholds, labels, None)
        elif quantizer_type == 'lloyd':
            quantizer[snr] = load_quantizer(snr, n_bits)[snr]
        else:
            raise NotImplementedError(f'Quantizer type {quantizer_type} not implemented!')
    return quantizer


def get_quantizer_gauss(snrs, n_bits, quantizer_type='lloyd', params=None):
    """Serial twin of :func:`get_quantizer` (reference :565-590)."""
    return get_quantizer(snrs, n_bits, quantizer_type)


def get_pilot_matrix(n_antennas, n_pilots=1, n_bits=1, pilot_type='angle_amp', return_vector=False, *, pilots=None):
    """``A = kron(x, I_N)`` for a length-``n_pilots`` pilot sequence ``x`` -- the reference's signature and pilot types
    (modules/utils.py:337-367): unquantised (``n_bits = inf``) and ``'ones'``: all ones; ``'angle'``: unit-modulus phases spread over
    [0, pi/2); ``'angle_amp'`` (default): the same phases with amplitudes rising linearly from 0.5 to 1, scaled to total power
    ``n_pilots``; ``'rand'``: one complex Gaussian draw (numpy's global generator, like the reference) scaled to that power.
    ``return_vector``: the column ``x [n_pilots, 1]`` instead of the matrix.  ``pilots=`` (keyword only, not in the reference)
    supplies a custom sequence."""
    if pilots is not None:
        x = np.asarray(pilots, dtype=complex).reshape(n_pilots, 1)
    elif n_bits == np.inf or n_bits == 'inf' or pilot_type == 'ones':
        x = np.ones((n_pilots, 1))
    elif pilot_type in ('angle', 'angle_amp'):
        phase = np.linspace(0.0, np.pi / 2, num=n_pilots, endpoint=False)
        x = np.exp(1j * phase)
        if pilot_type == 'angle_amp':
            x = np.linspace(0.5, 1.0, num=n_pilots, endpoint=True) * x
            x = x * (np.sqrt(n_pilots) / np.linalg.norm(x))
        x = x[:, None]
    elif pilot_type == 'rand':
        x = np.random.randn(n_pilots, 1) + 1j * np.random.randn(n_pilots, 1)
        x = x * (np.sqrt(n_pilots) / np.linalg.norm(x))
    else:
        raise NotImplementedError(f'Pilot type {pilot_type} is not implemented!')
    return x if return_vector else np.kron(x, np.eye(n_antennas))


def toeplitz(c, r=None):
    """Toeplitz matrix with first column ``c`` and first row ``r`` (``conj(c)`` if omitted) -- the helper of the reference
    (modules/utils.py:115-165, a copy of ``scipy.linalg.toeplitz``) the scripts use as ``toeplitz(t).T`` for channel covariances."""
    c = np.asarray(c).ravel()
    r = np.conjugate(c) if r is None else np.asarray(r).ravel()
    vals = np.concatenate((c[::-1], r[1:]))
    idx = (len(c) - 1) + np.arange(len(r))[None, :] - np.arange(len(c))[:, None]
    return vals[idx]


def mse(h_est, h):
    """The scripts' NMSE: ``sum |h_est - h|^2 / h.size`` (reference :617-618, Bussgang_GMM.py:289)."""
    if isinstance(h_est, torch.Tensor) or isinstance(h, torch.Tensor):
        a, b = torch.as_tensor(h_est), torch.as_tensor(h)
        return float(((a - b.to(a.device)).abs() ** 2).sum() / b.numel())
    return float(np.sum(np.abs(h_est - h) ** 2) / h.size)


def rate_lower_bound(h_est, h, buss, Cq):
    """Statistical lower bound on the achievable rate, the post-processing of the scripts after every estimator
    (Bussgang_GMM.py:291-309, Bussgang_MFA.py:154-172): with the normalised estimate ``g_b = h_est_b / clip(|h_est_b|^2, 0.1)``
    (the scripts divide by the SQUARED norm),
    ``inner_b = g_b^H B h_b``,  ``rate = log2(1 + |mean inner|^2 / (var inner + mean Re g_b^H C_q g_b))``.
    ``buss`` is the Bussgang matrix ``B`` and ``Cq = C_r - B C B^H`` the quantisation-noise covariance of the global model
    (``uniform_quantizer.get_Bussgang_matrix`` / ``get_Cr``).  Batched quadratic forms on the GPU (torch, complex128)."""
    he, ht = _to_cuda(h_est, torch.complex128), _to_cuda(h, torch.complex128)
    B, Cq = _to_cuda(buss, torch.complex128), _to_cuda(Cq, torch.complex128)
    norm_fac = (he.abs() ** 2).sum(dim=1).clamp(min=1e-1)
    g = he / norm_fac[:, None]
    inner = (g.conj() * (ht @ B.T)).sum(dim=1)
    num = inner.mean().abs() ** 2
    den1 = (inner - inner.mean()).abs().pow(2).mean()                       # np.var of a complex vector
    den2 = (g.conj() * (g @ Cq.T)).sum(dim=1).real.mean()
    return float(torch.log2(1 + num / (den1 + den2)))


def rate_from_accumulators(acc):
    """The bound of :func:`rate_lower_bound` from the sums ``acc [..., 5] = (sum Re inner, sum Im inner, sum |inner|^2,
    sum Re g^H C_q g, count)`` that ``engine.RateModel.accumulate`` adds up: ``m = S1 / n``, ``v = S2 / n - |m|^2`` (np.var,
    ddof 0), ``rate = log2(1 + |m|^2 / (v + Q / n))``.  Returns the rates over the leading dimensions (a float for ``[5]``)."""
    a = acc.detach().cpu().numpy() if isinstance(acc, torch.Tensor) else np.asarray(acc, dtype=np.float64)
    if a.shape[-1] != 5:
        raise ValueError('rate accumulators must have 5 entries in the last dimension')
    n = a[..., 4]
    m2 = (a[..., 0] / n) ** 2 + (a[..., 1] / n) ** 2
    rate = np.log2(1 + m2 / (a[..., 2] / n - m2 + a[..., 3] / n))
    return float(rate) if rate.ndim == 0 else rate


def rate_params(C, snr_dB, n_bits, quantizer_type='uniform', quantizer=None):
    """``(buss, Cq)`` of :func:`rate_lower_bound` for the global channel covariance ``C [N, N]`` (the scripts' construction,
    Bussgang_GMM.py:291-309): ``C_y = C + 10^(-snr/10) I``, ``buss`` the diagonal Bussgang matrix of C_y (uniform, or Lloyd-Max for
    ``quantizer_type='lloyd'`` with ``n_bits > 1``), ``Cq = get_Cr(C_y, ...) - buss C buss^H``.  ``quantizer`` is the
    ``(thresholds, labels, rho)`` table of ``get_quantizer``; it is looked up when omitted."""
    from . import lloyd_max_quantizer, uniform_quantizer
    C = np.asarray(C, dtype=complex)
    Cy = C + 10 ** (-snr_dB / 10) * np.eye(C.shape[-1])
    finite_multi = not _is_inf(n_bits) and n_bits > 1
    if _is_inf(n_bits):
        n_bits = np.inf
    if quantizer is None and finite_multi:
        quantizer = get_quantizer([snr_dB], n_bits, quantizer_type)[snr_dB]
    if quantizer_type == 'lloyd' and finite_multi:
        buss = lloyd_max_quantizer.get_Bussgang_matrix(n_bits, Cy, quantizer)
    else:
        buss = uniform_quantizer.get_Bussgang_matrix(snr_dB, n_bits, Cy).astype(complex)
    Cq = uniform_quantizer.get_Cr(Cy, n_bits, snr_dB, quantizer) - buss @ C @ buss.conj().T
    return buss, Cq


class _RefObject:
    """Attribute bag standing in for a class of the reference's ``modules`` package while unpickling."""

    def __setstate__(self, state):
        self.__dict__.update(state if isinstance(state, dict) else {})


def load_reference_model(path):
    """Load a model saved by the reference scripts (``joblib.dump(gmm, '...sav')``, Bussgang_GMM.py:262-264 /
    Bussgang_MFA.py:125-127) WITHOUT the reference on the path and return the matching estimator of this package
    (``Gmm_nbit`` or ``Mofa``) with the fitted parameters transplanted (``from_reference``)."""
    import joblib.numpy_pickle as npk

    from .gmm_cplx_bussgang import Gmm_nbit
    from .mofa_cplx_bussgang import Mofa

    kinds = {}

    class _Unpickler(npk.NumpyUnpickler):
        def find_class(self, module, name):
            if module.startswith('modules.'):
                cls = kinds.get((module, name))
                if cls is None:
                    cls = kinds[(module, name)] = type(name, (_RefObject,), {'_ref_module': module})
                return cls
            return super().find_class(module, name)

    with open(path, 'rb') as f:
        try:
            obj = _Unpickler(path, f, ensure_native_byte_order=False).load()
        except TypeError:                                     # older joblib: no ensure_native_byte_order argument
            f.seek(0)
            obj = _Unpickler(path, f).load()
    kind = type(obj).__name__
    if kind == 'Gmm_quant':
        from .gmm_cplx_quant import Gmm_quant
        return Gmm_quant.from_reference(obj)
    if kind == 'Gmm_nbit':
        return Gmm_nbit.from_reference(obj)
    if kind == 'Mofa':
        return Mofa.from_reference(obj)
    raise TypeError(f'{path}: unsupported reference object {getattr(obj, "_ref_module", "?")}.{kind}')
