"""``Mofa``: Bussgang mixture-of-factor-analysers estimator -- the API of the reference's
``modules/mofa_cplx_bussgang.py`` (``fit`` :94-113, ``estimate_from_y`` :117-159, ``predict_proba`` :342-356,
``predict_proba_max`` :359-366) over the CUDA kernels.  ``C_h,k = Lambda_k Lambda_k^H + diag(psi_k)``.
"""
import numpy as np
import torch

from . import _lib, engine, precompute
from .gmm_cplx_bussgang import _PreparedCache, _fingerprint, _frozen, _table_key


class Mofa:
    def __init__(self, n_components, latent_dim, PPCA=False, lock_psis=False, rs_clip=0.0,
                 max_condition_number=1.e6, maxiter=100, tol=1e-6, verbose=True):
        assert rs_clip >= 0.0
        self.n_components = n_components
        self.M = latent_dim
        self.PPCA = PPCA
        self.lock_psis = lock_psis
        self.rs_clip = rs_clip
        self.maxiter = maxiter
        self.tol = tol
        self.verbose = verbose
        self.max_condition_number = float(max_condition_number)
        self.N = None
        self.D = None
        self.means = None
        self.lambdas = None
        self.covs = None
        self.inv_covs = None
        self.psis = None
        self.amps = None
        self.zero_mean = False
        self.precision = 'auto'
        self.use_structure = True          # Woodbury (low-rank + diagonal) kernel when A = I and n_bits != 1
        self._cache = _PreparedCache()
        self._covs_are_low_rank = False
        self._last = None                  # handle prepared by the last estimate_from_y (for predict_proba)

    @classmethod
    def from_reference(cls, obj):
        new = cls(int(obj.n_components), int(obj.M), verbose=False)
        new.set_parameters(obj.means, obj.lambdas, obj.psis, obj.amps, covs=getattr(obj, 'covs', None))
        return new

    def set_parameters(self, means, lambdas, psis, amps, covs=None):
        self.means = _frozen(means, complex)
        self.lambdas = _frozen(lambdas, complex)
        self.psis = _frozen(psis, float)
        self.amps = _frozen(amps, float)
        self.n_components, self.D = self.means.shape
        self.M = self.lambdas.shape[-1]
        if covs is None:          # C_k = Lambda Lambda^H + diag(psi)   (reference :313-319)
            covs = self.lambdas @ np.transpose(self.lambdas.conj(), [0, 2, 1]) + np.stack([np.diag(p) for p in self.psis])
        lr = self.lambdas @ np.transpose(self.lambdas.conj(), [0, 2, 1]) + np.stack([np.diag(p) for p in self.psis])
        self.covs = _frozen(covs, complex)
        # the Woodbury kernel is only valid if the covariances really are Lambda Lambda^H + diag(psi)
        self._covs_are_low_rank = bool(np.allclose(self.covs, lr, rtol=1e-10, atol=1e-12))
        self._cache.clear()
        return self

    def fit(self, data, zero_mean=False):
        """EM for the mixture of factor analysers (reference :94-113, :219-339); see ``em.py``."""
        from . import em
        em.fit_mofa(self, data, zero_mean=zero_mean)
        self._cache.clear()
        return self

    def _prepared(self, A, snr_dB, n_bits, quantizer_type, quantizer):
        if self.means is None or self.covs is None or self.amps is None:
            raise RuntimeError('Mofa: model is not fitted (means / covs / amps missing)')
        A = np.asarray(A)
        nb = 'inf' if (n_bits == 'inf' or n_bits == np.inf) else int(n_bits)
        tables = _table_key(quantizer) if (nb != 1 and nb != 'inf' and quantizer_type == 'lloyd') else None
        woodbury = (self.use_structure and nb != 1 and self.lambdas is not None and self.psis is not None and
                    A.shape == (self.D, self.D) and np.array_equal(A, np.eye(self.D)) and self._covs_are_low_rank)
        # pilots on an integer grid and a tensor-core shape: the dense tcgen05 kernels beat the complex128 Woodbury kernel
        # (config 4: 55 M vs 0.9 M estimates/s) although they do 4x the flops
        # (off-grid pilots -- Lloyd-Max labels, unquantised data -- take three tensor passes up to D = 128; at D = 256 they have no
        # tensor-core path and stay on the Woodbury kernel)
        on_grid = precompute.data_scale_for(snr_dB, np.inf if nb == 'inf' else nb, quantizer_type) > 0
        if woodbury and self.precision != 'fp64' and engine.tc_padded_shape(A.shape[0], self.D, on_grid) is not None:
            woodbury = False
        if woodbury:
            key = ('woodbury', float(snr_dB), nb, quantizer_type if nb != 'inf' else None, tables, _fingerprint(self.means),
                   _fingerprint(self.lambdas), _fingerprint(self.psis), _fingerprint(self.amps))

            def make_w():
                prep = precompute.prepare_mfa_woodbury(self.means, self.lambdas, self.psis, self.amps, snr_dB,
                                                       np.inf if nb == 'inf' else nb, quantizer_type, quantizer)
                return engine.MfaModel(prep, flags=_lib.FLAG_TOP1_EXP_ARGMAX)
            self._last = self._cache.get(key, make_w)
            return self._last
        pad = self.precision != 'fp64'
        key = (float(snr_dB), nb, quantizer_type if nb not in (1, 'inf') else None, tables, A.shape, A.tobytes(),
               _fingerprint(self.means), _fingerprint(self.covs), _fingerprint(self.amps), pad)

        def make():
            prep = precompute.prepare(self.means, self.covs, self.amps, A, snr_dB, np.inf if nb == 'inf' else nb,
                                      quantizer_type, quantizer)
            return engine.DenseModel(prep, flags=_lib.FLAG_TOP1_EXP_ARGMAX, pad=pad)
        self._last = self._cache.get(key, make)
        return self._last

    def estimate_from_y(self, y, snr_dB, A=None, n_summands_or_proba=1, n_bits=1, quantizer_type='uniform',
                        quantizer=None):
        """Channel estimates ``[B, A.shape[-1]]`` from quantised pilots (reference :117-159)."""
        if A is None:
            A = np.eye(self.D, dtype=complex)
        model = self._prepared(A, snr_dB, n_bits, quantizer_type, quantizer)
        if isinstance(y, torch.Tensor):
            if y.is_cuda:
                return model.estimate(y, n_summands_or_proba, self.precision)
            return torch.from_numpy(model.estimate_host(y.numpy(), n_summands_or_proba, self.precision))
        return model.estimate_host(y, n_summands_or_proba, self.precision).astype(np.asarray(y).dtype, copy=False) \
            if np.iscomplexobj(y) else model.estimate_host(y, n_summands_or_proba, self.precision)

    def _log_resp(self, data):
        if self._last is None:
            # no observation setting prepared yet: the trained mixture itself, which is what the reference's predict_proba sees
            # right after fit() (mofa:109-111: _means / _covs / _inv_covs hold the fitted channel-domain parameters)
            if self.means is None or self.covs is None:
                raise RuntimeError('Mofa.predict_proba: the model is not fitted')
            self._prepared(np.eye(self.D, dtype=complex), np.inf, np.inf, 'uniform', None)
        dt = data if isinstance(data, torch.Tensor) and data.is_cuda else torch.as_tensor(np.asarray(data)).cuda()
        return self._last.log_prob(dt, self.precision)

    def predict_proba(self, data):
        """Responsibilities ``[B, K]`` for the most recently prepared setting (reference :342-356)."""
        p = torch.softmax(self._log_resp(data), dim=1)
        return p if isinstance(data, torch.Tensor) and data.is_cuda else p.cpu().numpy()

    def predict_proba_max(self, data):
        """Hard labels: argmax of ``exp`` of the un-normalised log responsibilities (reference :359-366)."""
        lab = torch.exp(self._log_resp(data)).argmax(dim=1)
        return lab if isinstance(data, torch.Tensor) and data.is_cuda else lab.cpu().numpy()
