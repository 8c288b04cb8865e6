"""Training (EM) for the complex GMM and the mixture of factor analysers -- SURVEY.md section 8f-1, the first row
after the inference hot path.  On a GPU the E-step of the 'full' / Toeplitz GMM is the whitening launch of the inference path
(``engine.DenseModel.log_prob``: the same ``l_k = logc_k - |L_k^-1 x - L_k^-1 mu_k|^2`` on the tensor cores, three-pass split for
unquantised data, shapes zero-padded to the next instantiated one; near-ties do not matter for soft responsibilities) and the
M-step is one batched GEMM over all components; the per-iteration Cholesky factors are cuSOLVER "plumbing".  Everything else is
torch float64 / complex128.

GMM (reference modules/gmm_cplx_bussgang.py:96-163, 437-848): sklearn-style EM on complex data -- k-means initialisation
on the (Re, Im) features, E-step with Cholesky-whitened complex Gaussian log-densities, M-step with weighted sample
covariances + ``reg_covar``, stop when the mean log-likelihood changes by less than ``tol``; ``n_init`` restarts.
'circulant' / 'block-circulant' run the diagonal EM in the (2-D) DFT domain and densify afterwards, as the reference does.
The Toeplitz types run the Barton-Fuhrmann inverse EM on the twofold-oversampled DFT grid (gmm:787-826).

MFA (reference modules/mofa_cplx_bussgang.py:94-113, 219-339, 403-421): k-means means, random small loadings, per-component
EM with Woodbury inverses, optional PPCA / locked psis.

The EM trajectories depend on the k-means and random initialisations, so results agree with the reference statistically
(same likelihood level, same estimator NMSE), not bit-wise.
"""
import math
import warnings

import numpy as np
import torch

from . import precompute


def _device():
    return torch.device('cuda') if torch.cuda.is_available() else torch.device('cpu')


def _generator(seed, device):
    g = torch.Generator(device=device)
    if seed is None:
        g.seed()
    else:
        g.manual_seed(int(seed))
    return g


def kmeans_labels(Xr, K, gen, n_iter=100):
    """k-means++ initialisation + Lloyd iterations on real features ``Xr [B, F]``; returns labels ``[B]``."""
    B = Xr.shape[0]
    idx = torch.randint(0, B, (1,), generator=gen, device=Xr.device)
    centers = Xr[idx].clone()
    d2 = ((Xr - centers[0]) ** 2).sum(1)
    for _ in range(1, K):
        prob = d2 / d2.sum().clamp_min(1e-300)
        nxt = torch.multinomial(prob, 1, generator=gen)
        centers = torch.cat([centers, Xr[nxt]], 0)
        d2 = torch.minimum(d2, ((Xr - Xr[nxt]) ** 2).sum(1))
    labels = None
    for _ in range(n_iter):
        dist = (Xr ** 2).sum(1, keepdim=True) - 2 * Xr @ centers.T + (centers ** 2).sum(1)[None]
        new = dist.argmin(1)
        if labels is not None and bool((new == labels).all()):
            break
        labels = new
        onehot = torch.zeros(B, K, dtype=Xr.dtype, device=Xr.device).scatter_(1, labels[:, None], 1.0)
        cnt = onehot.sum(0)
        upd = (onehot.T @ Xr) / cnt.clamp_min(1.0)[:, None]
        centers = torch.where(cnt[:, None] > 0, upd, centers)
    return labels


# ------------------------------------------------------------------------------------------------------------ GMM

def _m_step(X, resp, reg_covar, diag, zero_mean):
    """``estimate_gaussian_parameters`` (gmm:692-728): weights (un-normalised counts), means, covariances."""
    nk = resp.sum(0) + 10 * torch.finfo(resp.dtype).eps
    means = (resp.T.to(X.dtype) @ X) / nk[:, None]
    if zero_mean:
        means = torch.zeros_like(means)
    K, N = means.shape
    if diag:                                                            # gmm:768-786
        avg_x2 = (resp.T @ (X.real ** 2 + X.imag ** 2)) / nk[:, None]
        avg_xm = (means.conj() * ((resp.T.to(X.dtype) @ X) / nk[:, None])).real
        covs = avg_x2 - 2 * avg_xm + (means.real ** 2 + means.imag ** 2) + reg_covar
    else:                                                               # gmm:730-766
        covs = _weighted_scatter(X, resp, nk, means) + reg_covar * torch.eye(N, dtype=X.dtype, device=X.device)
    return nk, means, covs


def _weighted_scatter(X, resp, nk, means, chunk=4096):
    """``S_k = sum_b r_bk (x_b - mu_k)(x_b - mu_k)^T*`` / n_k for all components at once: one GEMM ``resp^T [K, B] x (x x^H) [B, N^2]``
    per chunk of samples instead of a Python loop of K weighted Gram products, then the rank-one mean terms (with ``mu_k`` the
    resp-weighted mean -- or zero -- the centred form equals the raw second moment minus mean terms)."""
    B, N = X.shape
    K = resp.shape[1]
    S = torch.zeros((K, N * N), dtype=X.dtype, device=X.device)
    rT = resp.T.to(X.dtype)
    for b0 in range(0, B, chunk):
        xb = X[b0:b0 + chunk]
        outer = (xb[:, :, None] * xb.conj()[:, None, :]).reshape(xb.shape[0], N * N)
        S += rT[:, b0:b0 + chunk] @ outer
    S = S.reshape(K, N, N) / nk[:, None, None]
    xbar = (rT @ X) / nk[:, None]                                       # resp-weighted sample means
    # sum r (x - m)(x - m)^H / n = S - xbar m^H - m xbar^H + m m^H
    m = means
    return S - xbar[:, :, None] * m.conj()[:, None, :] - m[:, :, None] * xbar.conj()[:, None, :] + m[:, :, None] * m.conj()[:, None, :]


def _m_step_inv(X, resp, reg_covar, zero_mean, covs_prev, Sigma, F2):
    """Toeplitz / block-Toeplitz M-step (``estimate_gaussian_covariances_inv``, gmm:792-826; Barton & Fuhrmann's inverse EM):
    the covariance lives on the diagonal ``Sigma_k`` of the twofold-oversampled DFT domain, ``C_k = F2^H diag(Sigma_k) F2``, and
    is updated with ``Theta = diag(F2 (C^-1 S C^-1 - C^-1) F2^H)`` of the previous covariance: ``Sigma += Sigma^2 Theta``."""
    nk = resp.sum(0) + 10 * torch.finfo(resp.dtype).eps
    means = (resp.T.to(X.dtype) @ X) / nk[:, None]
    if zero_mean:
        means = torch.zeros_like(means)
    K, N = means.shape
    covs = torch.empty((K, N, N), dtype=X.dtype, device=X.device)
    eye = torch.eye(N, dtype=X.dtype, device=X.device)
    Cinv = torch.linalg.pinv(covs_prev, hermitian=True)
    S_all = _weighted_scatter(X, resp, nk, means)                       # one batched GEMM for all components
    for k in range(K):
        S = S_all[k]
        theta = ((F2 @ (Cinv[k] @ S @ Cinv[k] - Cinv[k])) * F2.conj()).sum(1).real
        Sigma[k] = (Sigma[k] + Sigma[k] ** 2 * theta).clamp(min=reg_covar)
        covs[k] = (F2.conj().T * Sigma[k]) @ F2 + reg_covar * eye
    return nk, means, covs


class _KernelEStep:
    """E-step of the full-covariance GMM on the inference path's whitening launch (GPU only): the mixture is loaded into a
    ``qce_model`` with a zero LMMSE block and ``log_prob`` returns ``l [B, K]`` -- the quantity ``_log_prob`` computes with K
    triangular solves in torch."""

    def __init__(self, X):
        from . import engine
        self.engine, self.X, self.model = engine, X.contiguous(), None
        # unquantised data (data_scale = 0): off the integer grid
        self.ok = X.is_cuda and engine.tc_padded_shape(X.shape[1], X.shape[1], on_grid=False) is not None

    def log_prob(self, weights, means, covs):
        K, N = means.shape
        L, info = torch.linalg.cholesky_ex(covs)
        if int(info.max()) != 0:
            raise ValueError(precompute.NOT_PD_MSG)
        eye = torch.eye(N, dtype=covs.dtype, device=covs.device)
        Linv = torch.linalg.solve_triangular(L, eye.expand(K, N, N), upper=False)
        logdet = 2 * torch.log(torch.diagonal(L, dim1=1, dim2=2).real).sum(1)
        prep = dict(Linv=Linv.contiguous(), W=torch.zeros_like(Linv), zoff=(Linv @ means[:, :, None])[:, :, 0].contiguous(),
                    hoff=torch.zeros_like(means), logc=(torch.log(weights) - N * math.log(math.pi) - logdet).contiguous(),
                    data_scale=0.0, n_obs=N, n_ant=N, n_comp=K)             # data_scale 0: unquantised data (three-pass split)
        if self.model is None:
            self.model = self.engine.DenseModel(prep, pad=True)
        else:
            self.model.update(prep)
        return self.model.log_prob(self.X, 'auto')


def _log_prob(X, weights, means, covs, diag):
    """Weighted log-densities ``[B, K]`` of the circularly-symmetric complex Gaussians (gmm:369-435)."""
    B, N = X.shape
    K = means.shape[0]
    out = torch.empty((B, K), dtype=torch.float64, device=X.device)
    if diag:
        for k in range(K):
            d = X - means[k]
            out[:, k] = -N * math.log(math.pi) - torch.log(covs[k]).sum() - ((d.real ** 2 + d.imag ** 2) / covs[k]).sum(1)
    else:
        L, info = torch.linalg.cholesky_ex(covs)
        if int(info.max()) != 0:
            raise ValueError(precompute.NOT_PD_MSG)
        logdet = 2 * torch.log(torch.diagonal(L, dim1=1, dim2=2).real).sum(1)
        for k in range(K):
            z = torch.linalg.solve_triangular(L[k], (X - means[k]).T, upper=False)
            out[:, k] = -N * math.log(math.pi) - logdet[k] - (z.real ** 2 + z.imag ** 2).sum(0)
    return out + torch.log(weights)[None]


def _em_gmm(X, K, diag, zero_mean, reg_covar, tol, max_iter, n_init, init_params, seed, verbose=0, F2=None):
    dev = X.device
    gen = _generator(seed, dev)
    B = X.shape[0]
    best = None
    converged_any = False
    kernel_e = _KernelEStep(X) if not diag else None
    for init in range(n_init):
        if init_params == 'kmeans':                                     # gmm:560-567
            labels = kmeans_labels(torch.cat([X.real, X.imag], 1), K, gen)
            resp = torch.zeros(B, K, dtype=torch.float64, device=dev).scatter_(1, labels[:, None], 1.0)
        elif init_params == 'random':
            resp = torch.rand(B, K, generator=gen, dtype=torch.float64, device=dev)
            resp = resp / resp.sum(1, keepdim=True)
        else:
            raise ValueError("Unimplemented initialization method '%s'" % init_params)
        nk, means, covs = _m_step(X, resp, reg_covar, diag, zero_mean)
        weights = nk / B
        Sigma = None
        if F2 is not None:                                              # gmm:600-604: start from the unstructured covariances
            Sigma = torch.stack([((F2 @ covs[k]) * F2.conj()).sum(1).real for k in range(K)]).clamp(min=reg_covar)
        lower, converged, n_iter = -np.inf, False, 0
        for n_iter in range(1, max_iter + 1):
            prev = lower
            if kernel_e is not None and kernel_e.ok:                    # E-step (gmm:612-650) on the whitening launch
                wlp = kernel_e.log_prob(weights, means, covs)
            else:
                wlp = _log_prob(X, weights, means, covs, diag)
            lpn = torch.logsumexp(wlp, 1)
            resp = torch.exp(wlp - lpn[:, None])
            if F2 is None:
                nk, means, covs = _m_step(X, resp, reg_covar, diag, zero_mean)   # M-step (gmm:659-690)
            else:
                nk, means, covs = _m_step_inv(X, resp, reg_covar, zero_mean, covs, Sigma, F2)
            weights = nk / B
            lower = float(lpn.mean())
            if verbose:
                print(f'  init {init} iter {n_iter}: lower bound {lower:.6f}')
            if abs(lower - prev) < tol:
                converged = True
                break
        converged_any |= converged
        if best is None or lower > best[0]:
            best = (lower, weights, means, covs, n_iter, converged)
    best = best[:5] + (converged_any,)                                  # sklearn keeps converged_ sticky over the n_init restarts
    if not converged_any:
        warnings.warn('EM did not converge. Try different init parameters, or increase max_iter, tol or check for degenerate data.')
    return best


def fit_gmm(model, h, blocks=None, zero_mean=False):
    """``Gmm_nbit.fit`` (gmm:96-163): 'full', 'circulant', 'block-circulant' (EM in the DFT domain) and 'toeplitz' / 'block-toeplitz'
    (inverse EM)."""
    gm = model.gm
    ctype = gm.covariance_type
    dev = _device()
    X = torch.as_tensor(np.asarray(h), dtype=torch.complex128, device=dev)
    if X.dim() != 2:
        raise ValueError('h must be [n_samples, n_antennas]')
    N = X.shape[1]
    model.params['zero_mean'] = bool(zero_mean)
    F2 = None
    if ctype in ('toeplitz', 'block-toeplitz'):                         # inverse EM on the oversampled DFT grid (gmm:142-160)
        if ctype == 'block-toeplitz' and blocks is None:
            raise ValueError("covariance_type='block-toeplitz' needs blocks=(n1, n2)")
        dims = (N,) if ctype == 'toeplitz' else tuple(blocks)
        Fn = np.ones((1, 1), dtype=complex)
        for n in dims:
            Fn = np.kron(Fn, np.fft.fft(np.eye(2 * n))[:, :n] / np.sqrt(2 * n))
        model.F2 = Fn
        model.params['inv-em'] = True
        F2 = torch.as_tensor(Fn, dtype=torch.complex128, device=dev)
        n1, n2 = 1, N
    elif ctype == 'circulant':
        n1, n2 = 1, N
    elif ctype == 'block-circulant':
        if blocks is None:
            raise ValueError("covariance_type='block-circulant' needs blocks=(n1, n2)")
        n1, n2 = blocks
    elif ctype != 'full':
        raise NotImplementedError(f'Fitting for covariance_type = {ctype} is not implemented.')
    diag = ctype in ('circulant', 'block-circulant')
    if diag:
        F = torch.as_tensor(precompute.dft_matrix(n1, n2), dtype=torch.complex128, device=dev)
        X = X @ F.T                                                     # DFT-domain data (gmm:105-106, :123-126)
    lower, weights, means, covs, n_iter, converged = _em_gmm(
        X, int(gm.n_components), diag, bool(zero_mean), float(gm.reg_covar), float(gm.tol), int(gm.max_iter), int(gm.n_init),
        gm.init_params, gm.random_state, getattr(gm, 'verbose', 0), F2)
    gm.converged_, gm.n_iter_, gm.lower_bound_ = bool(converged), int(n_iter), float(lower)
    w = weights.cpu().numpy()
    if diag:
        c = covs.cpu().numpy()
        mu_f = means.cpu().numpy()
        Fn = precompute.dft_matrix(n1, n2)
        model.fft_covs, model.fft_means = c, mu_f
        if ctype == 'block-circulant':
            model.F2 = Fn
        dense_means = mu_f @ Fn.conj()                                  # gmm:109 / :127
        dense_covs = np.einsum('ji,kj,jl->kil', Fn.conj(), c.astype(complex), Fn)
        model.means_cplx, model.covs_cplx = dense_means, dense_covs
        model.gm.weights_ = w
        model.blocks = (n1, n2)
    else:
        model.means_cplx, model.covs_cplx = means.cpu().numpy(), covs.cpu().numpy()
        model.gm.weights_ = w
        model.blocks, model.fft_covs = None, None
    model.gm.covariance_type = 'full'                                   # every type is dense after fit (gmm:116, :134)
    model.gm.means_, model.gm.covariances_ = model.means_cplx, model.covs_cplx
    model.chol = None
    return model


# ------------------------------------------------------------------------------------------------------------ MFA

def _mfa_inv_covs(lambdas, psis):
    """Woodbury inverse of ``Lambda Lambda^H + diag(psi)`` for all components (mofa:412-421)."""
    M = lambdas.shape[-1]
    psiI = 1 / psis
    inner = torch.eye(M, dtype=lambdas.dtype, device=lambdas.device) + (lambdas.conj().transpose(1, 2) * psiI[:, None, :]) @ lambdas
    step = psiI[:, :, None] * (lambdas @ torch.linalg.inv(inner) @ lambdas.conj().transpose(1, 2)) * psiI[:, None, :]
    return torch.diag_embed(psiI.to(lambdas.dtype)) - step, inner


def fit_mofa(model, data, zero_mean=False, seed=None):
    """``Mofa.fit`` (mofa:94-113, :219-339)."""
    dev = _device()
    X = torch.as_tensor(np.asarray(data), dtype=torch.complex128, device=dev)
    B, D = X.shape
    K, M = int(model.n_components), int(model.M)
    gen = _generator(seed, dev)
    model.zero_mean, model.N, model.D = bool(zero_mean), B, D
    # ---- initialisation (mofa:219-243)
    labels = kmeans_labels(torch.cat([X.real, X.imag], 1), K, gen)
    onehot = torch.zeros(B, K, dtype=torch.float64, device=dev).scatter_(1, labels[:, None], 1.0)
    means = (onehot.T.to(X.dtype) @ X) / onehot.sum(0).clamp_min(1.0)[:, None]
    if zero_mean:
        means = torch.zeros_like(means)
    lam = torch.view_as_complex(torch.randn((K, D, M, 2), generator=gen, dtype=torch.float64, device=dev)) \
        / math.sqrt(model.max_condition_number) / math.sqrt(2)
    psis = torch.var(X, dim=0, unbiased=False).real[None, :].repeat(K, 1)
    amps = torch.rand(K, generator=gen, dtype=torch.float64, device=dev)
    amps = amps / amps.sum()
    L_prev, L_all = -np.inf, []
    it = 0
    for it in range(int(model.maxiter)):                                 # run_em (mofa:246-267)
        inv_covs, inner = _mfa_inv_covs(lam, psis)
        # log-likelihoods / responsibilities (mofa:322-339): logdet via the matrix determinant lemma
        logdet = torch.log(psis).sum(1) + torch.linalg.slogdet(inner)[1]
        logrs = torch.empty((K, B), dtype=torch.float64, device=dev)
        for k in range(K):
            d = X - means[k]
            logrs[k] = torch.log(amps[k]) - D * math.log(math.pi) - logdet[k] - (d.conj() * (d @ inv_covs[k].T)).sum(1).real
        L = torch.logsumexp(logrs, 0)
        rs = torch.exp(logrs - L[None])
        if model.rs_clip > 0.0:
            rs = torch.where((rs.sum(1) < model.rs_clip)[:, None], torch.full_like(rs, model.rs_clip), rs)
        sumrs = rs.sum(1)
        betas = lam.conj().transpose(1, 2) @ inv_covs                    # [K,M,D]
        eyeM = torch.eye(M, dtype=X.dtype, device=dev)
        for k in range(K):                                               # _EM_per_component (mofa:270-310)
            zero0 = X.T if zero_mean else X.T - means[k][:, None]
            latents = betas[k] @ zero0                                   # [M,B]
            lat_cov_sum = (eyeM - betas[k] @ lam[k]) * sumrs[k] + (latents * rs[k]) @ latents.conj().T
            lamlat = lam[k] @ latents
            if zero_mean:
                means[k] = 0.0
            else:
                means[k] = ((X.T - lamlat) * rs[k]).sum(1) / sumrs[k]
            zeroed = X.T - means[k][:, None]
            lam[k] = ((zeroed * rs[k]) @ latents.conj().T) @ torch.linalg.inv(lat_cov_sum)
            p = (((zeroed - lamlat) * zeroed.conj()) @ rs[k].to(X.dtype)).real / sumrs[k]
            psis[k] = p.clamp_min(1e-6)
            if model.PPCA:
                psis[k] = psis[k].mean()
            amps[k] = sumrs[k] / B
        if model.lock_psis:
            psis = ((sumrs @ psis) / sumrs.sum())[None, :].repeat(K, 1)
        newL = float(L.sum())
        L_all.append(newL)
        if model.verbose:
            print(f'Iteration {it} | lower bound: {newL:.5f}', end='\r')
        dL = abs((newL - L_prev) / newL)
        if it > 5 and dL < model.tol:
            break
        L_prev = newL
    if it >= int(model.maxiter) - 1:
        warnings.warn(f"EM didn't converge after {it} iterations")
    model.L_all = L_all
    model.set_parameters(means.cpu().numpy(), lam.cpu().numpy(), psis.cpu().numpy(), amps.cpu().numpy())
    model.inv_covs = _mfa_inv_covs(lam, psis)[0].cpu().numpy()
    return model
