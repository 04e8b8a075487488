"""Dense CPU reference for the likelihood path's two on-the-fly generators (used by tests/test_lml_dense_ref_cpu.py and
tests/test_gpu_lml_kernels.py): the covariance build and the dKcov/dhp contraction.

cov() is the matrix gegp_build_cov writes in each mode, assembled by oracle/gegp_oracle.py's all_K_w_chofac.  contract()
is sum(W .* dKcov/dhp) for every hyper-parameter, laid out as GEGP_OUT_*, with dKcov/dhp_m built one at a time from the
oracle's profile blocks (_blocks_from_profile), so that N ~ 1500 at d = 24 stays within a few hundred MB.  Built only
from the oracle's functions; the oracle itself is unchanged."""
import numpy as np

from gpgradpy_b200._lib import (MODE_BASE, MODE_PRECON, MODE_PRECON_COV, OUT_DKERN, OUT_DVARF, OUT_DVARG, OUT_DVARK,
                                OUT_GRAD, out_len)
from oracle import gegp_oracle as O


def _is_ratqu(kernel):
    return O._kernel_spec(kernel)[0] == "RatQu"


def cov(X, theta, mode, eta=0.0, mask=None, kernel=None, noise=None, varK=1.0):
    """What gegp_build_cov(noise, mode, eta, varK) writes, noise already divided by varK as that call expects:
      MODE_BASE        varK (K + diag(noise) + eta I)
      MODE_PRECON      varK (P^-1 (K + diag(noise)) P^-1 + eta I), returned with p = sqrt(diag(K + noise))
      MODE_PRECON_COV  varK (K + diag(noise) + eta diag(K + noise))
    -> (matrix [N, N], p [N] or None)."""
    theta = np.asarray(theta, dtype=float)
    nv = None if noise is None else np.asarray(noise, dtype=float) * varK     # the oracle divides by varK again
    ka = O.all_K_w_chofac(X, theta, "base" if mode == MODE_BASE else "precon", eta, nv, varK, mask, calc_chofac=False,
                          kernel=kernel)
    if mode == MODE_PRECON:
        return varK * (ka.Kcor + eta * np.eye(ka.Kcor.shape[0])), ka.pvec
    return ka.Kcov, None


def dcov_hp(X, theta, mode=MODE_BASE, eta=0.0, mask=None, kernel=None, noisy=False, varK=1.0):
    """Yield (GEGP_OUT_* index, dKcov/dhp [N, N]) one hyper-parameter at a time: theta_m (OUT_GRAD + m), the
    rational-quadratic alpha (OUT_DKERN) and, when noisy, varK / var_fval / var_fgrad.  The same matrices as the
    oracle's kerngrad_hp (noise-free, optz/GpHparaGrad.py:13-56) and kcov_grad_hp_noisy (:58-155); dK/dtheta_m in the
    profile form of _kern_grad_dtheta_profile for every family (the Gaussian kernel is f1 = f3 = -k, f2 = k)."""
    theta = np.asarray(theta, dtype=float)
    n, d = X.shape
    s = O._sel(n, mask)
    g = s.size
    N = n + g * d
    precon = mode == MODE_PRECON
    vk = varK if noisy else 1.0
    R = O.calc_rtensor(X, X)
    sq = O._sqdist(R, theta)
    _, f1, f2, f3 = O._radial(kernel, sq)
    up = O._blocks_from_profile(X, X, theta, f1, f2, f3, mask, mask)
    gg = np.ix_(s, s)

    def blk(i):
        return slice(n + i * g, n + (i + 1) * g)

    def finish(D):
        if noisy:
            D *= varK
        if precon:     # d(eta p^2)/dhp: eta times the diagonal of dK/dhp (optz/GpHparaGrad.py:40-50, :105-109)
            D[np.diag_indices(N)] *= 1.0 + eta
        return D

    for m in range(d):
        r2 = R[m] ** 2
        row = np.hstack([r2] + [r2[:, s]] * d)
        D = np.vstack([row] + [row[s, :]] * d)
        D *= up
        D[blk(m), :n] += 2.0 * R[m][s, :] * f1[s, :]
        D[:n, blk(m)] += -2.0 * R[m][:, s] * f1[:, s]
        D[blk(m), blk(m)] += -2.0 * f1[gg]
        for j in range(d):
            t = -4.0 * theta[j] * R[m][gg] * R[j][gg] * f2[gg]
            D[blk(m), blk(j)] += t
            D[blk(j), blk(m)] += t
        yield OUT_GRAD + m, finish(D)
    del up
    if _is_ratqu(kernel):
        d0, d1, d2 = O._radial_dalpha(kernel, sq)
        yield OUT_DKERN, finish(O._blocks_from_profile(X, X, theta, d0, d1, d2, mask, mask))
    if noisy:
        K = O.kern_grad(X, X, theta, mask, mask, kernel=kernel)
        if precon:
            K[np.diag_indices(N)] *= 1.0 + eta
        else:
            K[np.diag_indices(N)] += eta
        yield OUT_DVARK, K
        sc = (1.0 + eta) if precon else 1.0
        yield OUT_DVARF, np.diag(np.hstack((sc * np.ones(n), np.zeros(g * d))))
        yield OUT_DVARG, np.diag(np.hstack((np.zeros(n), sc * np.ones(g * d))))


def weigh(D, W):
    """(sum(W .* D), sum(|W .* D|)); a 1-D W = v stands for W = v v^T, which is never formed."""
    if W.ndim == 1:
        return float(W @ (D @ W)), float(np.abs(W) @ (np.abs(D) @ np.abs(W)))
    P = W * D
    return float(np.sum(P)), float(np.sum(np.abs(P)))


def contract(X, theta, W, mode=MODE_BASE, eta=0.0, mask=None, kernel=None, noisy=False, varK=1.0):
    """sum(W .* dKcov/dhp) for every hyper-parameter -> (g, scale), both [GEGP_OUT_LEN(d)] with the entries of
    dcov_hp filled and the others 0; scale = sum(|W .* dKcov/dhp|), the yardstick of the tolerance rule
    |g - g_ref| <= 1e-12 scale (which, unlike a tolerance relative to |g|, holds where g cancels)."""
    W = np.asarray(W, dtype=float)
    g, sc = np.zeros(out_len(X.shape[1])), np.zeros(out_len(X.shape[1]))
    for k, D in dcov_hp(X, theta, mode, eta, mask, kernel, noisy, varK):
        g[k], sc[k] = weigh(D, W)
    return g, sc


def hp_slots(d, kernel=None, noisy=False):
    """The GEGP_OUT_* entries contract fills (the ones a contraction test compares)."""
    k = [OUT_GRAD + m for m in range(d)]
    if _is_ratqu(kernel):
        k.append(OUT_DKERN)
    if noisy:
        k += [OUT_DVARK, OUT_DVARF, OUT_DVARG]
    return k


def contract_err(g, g_ref, scale, slots):
    """max over the compared entries of |g - g_ref| / scale (the tolerance rule asks for <= 1e-12)."""
    slots = list(slots)
    return float(np.max(np.abs(np.asarray(g)[slots] - np.asarray(g_ref)[slots]) / np.asarray(scale)[slots]))
