"""CPU reference for the batched surrogate Hessians (used by tests/test_hess_batch_cpu.py and tests/test_gpu_hess_batch.py).

eval_model_hess_batch runs oracle/gegp_oracle.py's one-point eval_model_hess arithmetic at every row of Xs, but factors K
once: calling eval_model_hess per point would repeat the cho_factor for every point (at N = 5500, one factorisation per
point).  Built only from the oracle's public functions; the oracle itself is unchanged."""
import numpy as np
from scipy import linalg

from oracle import gegp_oracle as O


def eval_model_hess_batch(X, fval, grad, theta, varK, beta, Xs, mode="precon", eta=None, kernel=None, noise_vec=None,
                          mask=None):
    """(mu [nx], sig [nx], dmudx [nx, d], dsigdx [nx, d], d2mudx2 [nx, d, d], d2sigdx2 [nx, d, d]), each row what
    O.eval_model_hess(..., Xs[i], ...) returns (eval/GpEvalModel.py:175-180, 356-382)."""
    n, d = X.shape
    Xs = np.atleast_2d(Xs)
    nx = Xs.shape[0]
    if eta is None:
        eta = O.nugget(n, d, mode, kernel=kernel)[1]
    ka = O.all_K_w_chofac(X, theta, mode, eta, noise_vec, 1.0, mask, kernel=kernel)
    sel = np.arange(n) if mask is None else np.flatnonzero(np.asarray(mask, dtype=bool))
    y = O.make_data_vec(fval, grad)
    H = O.aug_vand(n, sel.size, d)
    a = linalg.cho_solve(ka.chofac, y - H @ np.atleast_1d(beta))
    rows = np.concatenate([np.arange(n)] + [n + j * n + sel for j in range(d)])
    sigK = np.sqrt(varK)
    mu, sig = np.empty(nx), np.empty(nx)
    dmu, dsig = np.empty((nx, d)), np.empty((nx, d))
    d2mu, d2sig = np.empty((nx, d, d)), np.empty((nx, d, d))
    for i in range(nx):
        Kg = O.kern_grad(X, Xs[i:i + 1], theta, mask, None, kernel=kernel)   # [N, 1 + d]
        Kyx, dKxy = Kg[:, 0], Kg[:, 1:].T
        KinvK = linalg.cho_solve(ka.chofac, Kyx)
        s2 = 1.0 - Kyx @ KinvK
        sig[i] = np.sqrt(max(s2, 0.0)) * sigK
        mu[i] = float(np.atleast_1d(beta)[0]) + Kyx @ a
        dmu[i] = dKxy @ a
        inv_sig = 1.0 / sig[i] if sig[i] != 0 else 0.0
        dsig[i] = -inv_sig * (dKxy @ KinvK) * sigK ** 2
        d2mu[i], term1 = _d2k_dot(X, Xs[i], theta, kernel, rows, (a, KinvK))
        term2 = dKxy @ linalg.cho_solve(ka.chofac, dKxy.T)
        d2sig2 = -2.0 * varK * (term1 + term2)
        s = sig[i] if sig[i] != 0 else np.nan
        d2sig[i] = (d2sig2 - 2.0 * np.outer(dsig[i], dsig[i])) / (2.0 * s)
    return mu, sig, dmu, dsig, d2mu, d2sig


def _d2k_dot(X, xs, theta, kernel, rows, vecs):
    """[O.kern_hess_x(X, xs, theta, kernel=kernel)[:, :, rows] @ v for v in vecs], each [d, d]: the same entries in
    profile form, built with array operations one row block k at a time instead of the oracle's d^3 Python loop, so
    that the reference stays usable at d in the hundreds.  rho = x_test - x_train and u = theta rho, as in the oracle."""
    n, d = X.shape
    rho = xs[None, :] - X
    u = theta[None, :] * rho                                            # [n, d]
    _, f1, f2, f3 = O._radial(kernel, np.sum(u * rho, axis=1))
    uT, diag = u.T, np.arange(d)
    out = [np.empty((d, d)) for _ in vecs]
    for k in range(d):
        Hk = np.empty((d, n * (d + 1)))                                 # [i, value p | gradient (j, p)]
        Hk[:, :n] = 4.0 * uT * (u[:, k] * f2)
        Hk[k, :n] += 2.0 * theta[k] * f1
        G = -8.0 * (uT[:, None, :] * uT[None, :, :]) * (u[:, k] * f3)   # [i, j, p]
        G[k] -= 4.0 * theta[k] * uT * f2                                 # i = k
        G[:, k] -= 4.0 * theta[k] * uT * f2                              # j = k
        G[diag, diag] -= 4.0 * theta[:, None] * (u[:, k] * f2)           # i = j
        Hk[:, n:] = G.reshape(d, d * n)
        for o, v in zip(out, vecs):
            o[k] = Hk[:, rows] @ v
    return out
