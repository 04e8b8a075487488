"""CPU oracle for the gradient-enhanced GP hot path  --  TEST INFRASTRUCTURE ONLY.

This module is a NumPy/SciPy restatement of the reference algorithm (marchildon/gpgradpy
v1.3.2).  It exists to CHECK the CUDA path (tests/, __graft_entry__.smoke(), bench.py's
cpu_baseline / --impl reference leg).  Nothing under gpgradpy_b200/ may import it.

Parity pin: the reference ships NO golden vectors (its unit tests are finite-difference
self-consistency checks, SURVEY.md section 4).  This oracle is pinned by running the reference
itself in the build container: oracle/make_golden.py imports /root/reference, evaluates the
same inputs and writes tests/golden/*.npz; tests/test_oracle_golden.py compares this file
against those fixtures on CPU.

Conventions (SURVEY.md appendix B):
  * data / matrix order is dimension-major: [f(x_0..x_{n-1}) | d/dx_0 at grad points | d/dx_1 ...]
    (gradients flattened Fortran-order; base/CommonFun.py:170, kernel/Kernel.py:353)
  * r = x_row - x_col (base/CommonFun.py:82)
  * noise-free LML uses varK = 1 inside K and the closed form sigma^2 (optz/CalcLkd.py:157-159)
"""
from __future__ import annotations

import dataclasses
import numpy as np
from scipy import linalg


# ----------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md section 8d; plt/plt_cond.py:54-85 for the test function)
# ----------------------------------------------------------------------------------------------

def rosenbrock(x, a=10.0):
    """d-dimensional Rosenbrock value, restated from plt/plt_cond.py:54-64."""
    x = np.asarray(x, dtype=float)
    return np.sum(a * (x[:, 1:] - x[:, :-1] ** 2) ** 2 + (1.0 - x[:, :-1]) ** 2, axis=1)


def rosenbrock_grad(x, a=10.0):
    """Gradient of the above, restated from plt/plt_cond.py:66-85."""
    x = np.asarray(x, dtype=float)
    g = np.zeros_like(x)
    g[:, :-1] += -2.0 * (1.0 - x[:, :-1]) - 4.0 * a * x[:, :-1] * (x[:, 1:] - x[:, :-1] ** 2)
    g[:, 1:] += 2.0 * a * (x[:, 1:] - x[:, :-1] ** 2)
    return g


def synthetic_problem(n, d, seed=0, lo=-2.0, hi=2.0):
    """X ~ U[lo,hi]^d, Rosenbrock a=10 value and gradient (SURVEY.md 8d)."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(lo, hi, (n, d))
    if d == 1:  # Rosenbrock is empty in 1-D: use f = sin(3x) + x^2 instead
        return x, np.sin(3.0 * x[:, 0]) + x[:, 0] ** 2, 3.0 * np.cos(3.0 * x) + 2.0 * x
    return x, rosenbrock(x), rosenbrock_grad(x)


def bench_theta(d):
    """theta_i = 0.05*linspace(0.5,1.5,d)*(10/d)  (SURVEY.md 8d)."""
    return 0.05 * np.linspace(0.5, 1.5, d) * (10.0 / d)


# ----------------------------------------------------------------------------------------------
# kernel matrices
# ----------------------------------------------------------------------------------------------

def calc_rtensor(X, Y):
    """R[i,a,b] = X[a,i] - Y[b,i]   (base/CommonFun.py:58-84)."""
    return (X[:, None, :] - Y[None, :, :]).transpose(2, 0, 1).copy()


def kern_base(X, Y, theta, kernel=None):
    """k = exp(-sum_i theta_i r_i^2), accumulated i = 0..d-1 (kernel/KernelSqExp.py:18-46); the Matern-5/2 and
    rational-quadratic values through _radial (kernel/KernelMatern5f2.py:17-52, kernel/KernelRatQuad.py:18-51)."""
    R = calc_rtensor(X, Y)
    if kernel is not None and _kernel_spec(kernel)[0] != "SqExp":
        return _radial(kernel, _sqdist(R, theta))[0]
    e = np.zeros(R.shape[1:])
    for i in range(R.shape[0]):
        e -= theta[i] * R[i] ** 2
    return np.exp(e)


def _sel(n, mask):
    return np.arange(n) if mask is None else np.flatnonzero(np.asarray(mask, dtype=bool))


def _kernel_spec(kernel):
    """kernel = None | 'SqExp' | 'Ma5f2' | ('RatQu', alpha)  ->  (name, alpha-or-None).  Names are the reference's
    (kernel/Kernel.py:27-107); RatQu defaults to alpha = 2 (kernel/KernelRatQuad.py:849)."""
    if kernel is None:
        return "SqExp", None
    if isinstance(kernel, str):
        return kernel, (2.0 if kernel == "RatQu" else None)
    name, hp = kernel
    return name, (None if hp is None else float(np.ravel(hp)[0]))


def kernel_diag_coef(kernel=None):
    """diag(K) of a gradient row is c * theta_i: gamma_i^2 of theta2gamma (kernel/KernelSqExp.py:581-583 and
    kernel/KernelRatQuad.py:853-855: 2; kernel/KernelMatern5f2.py:655-657: 5/3)."""
    return 5.0 / 3.0 if _kernel_spec(kernel)[0] == "Ma5f2" else 2.0


def _radial(kernel, s):
    """(phi, phi', phi'', phi''') of the kernel as a function of s = sum_i theta_i r_i^2, written with the reference's
    own intermediate quantities:
      SqExp  kernel/KernelSqExp.py:18-46:        phi = exp(-s)
      Ma5f2  kernel/KernelMatern5f2.py:38-52, 149-186:  nu = sqrt(s), Abase = exp(-sqrt5 nu), mat1 = 5/3 (1 + sqrt5 nu) Abase;
             phi = (1 + sqrt5 nu + 5/3 nu^2) Abase, phi' = -mat1 / 2, phi'' = 25/12 Abase,
             phi''' = -(25 sqrt5 / 24) Abase / max(nu, 1e-16)    (:574 inv_nu_mat clamp)
      RatQu  kernel/KernelRatQuad.py:18-51, 451-458:    B = 1 + s / alpha; phi = B^-alpha, phi' = -B^(-alpha-1),
             phi'' = (1 + 1/alpha) B^(-alpha-2), phi''' = -(1 + 1/alpha)(alpha + 2)/alpha B^(-alpha-3)"""
    name, alpha = _kernel_spec(kernel)
    if name == "SqExp":
        k = np.exp(-s)
        return k, -k, k, -k
    if name == "Ma5f2":
        sqrt5 = np.sqrt(5.0)
        nu = np.sqrt(s)
        Abase = np.exp(-sqrt5 * nu)
        mat1 = (5.0 / 3.0) * (1.0 + sqrt5 * nu) * Abase
        return ((1.0 + sqrt5 * nu + (5.0 / 3.0) * nu ** 2) * Abase, -0.5 * mat1, (25.0 / 12.0) * Abase,
                -(25.0 * sqrt5 / 24.0) * Abase / np.maximum(nu, 1e-16))
    if name == "RatQu":
        B = 1.0 + s / alpha
        return (B ** (-alpha), -B ** (-alpha - 1.0), (1.0 + 1.0 / alpha) * B ** (-alpha - 2.0),
                -(1.0 + 1.0 / alpha) * (alpha + 2.0) / alpha * B ** (-alpha - 3.0))
    raise ValueError(f"unknown kernel {name}")


def _radial_dalpha(kernel, s):
    """d/dalpha of (phi, phi', phi'') for the rational-quadratic kernel, in the reference's T0 / T1 / T2 form
    (kernel/KernelRatQuad.py:133-163 and :770-782): dphi = B^(-alpha-1) (s/alpha - B ln B), dphi' = T0 / 2,
    dphi'' = -T2 / 4."""
    name, alpha = _kernel_spec(kernel)
    assert name == "RatQu"
    B = 1.0 + s / alpha
    B_lnB = B * np.log(B)
    d0 = B ** (-alpha - 1.0) * (s / alpha - B_lnB)
    T0 = 2.0 * B ** (-alpha - 2.0) * (((-alpha - 1.0) / alpha ** 2) * s + B_lnB)
    T2 = 4.0 * B ** (-alpha - 3.0) * (B / alpha ** 2 - ((1.0 + 1.0 / alpha) * (alpha + 2.0) / alpha ** 2) * s
                                      + (1.0 + 1.0 / alpha) * B_lnB)
    return d0, 0.5 * T0, -0.25 * T2


def _sqdist(R, theta):
    s = np.zeros(R.shape[1:])
    for i in range(R.shape[0]):
        s += theta[i] * R[i] ** 2
    return s


def _blocks_from_profile(X, Y, theta, f0, f1, f2, mask1, mask2):
    """Assemble [K00 | K0j ; Ki0 | Kij] from profile values: K00 = f0, K_i0 = 2 th_i r_i f1, K_0j = -2 th_j r_j f1,
    K_ij = -2 th_i delta_ij f1 - 4 th_i th_j r_i r_j f2  (the common structure of kernel/KernelSqExp.py:380-408,
    kernel/KernelMatern5f2.py:424-449 and kernel/KernelRatQuad.py:520-551)."""
    n1, d = X.shape
    n2 = Y.shape[0]
    s1, s2 = _sel(n1, mask1), _sel(n2, mask2)
    g1, g2 = s1.size, s2.size
    R = calc_rtensor(X, Y)
    K = np.zeros((n1 + g1 * d, n2 + g2 * d))
    K[:n1, :n2] = f0
    for i in range(d):
        ri = slice(n1 + i * g1, n1 + (i + 1) * g1)
        ci = slice(n2 + i * g2, n2 + (i + 1) * g2)
        K[ri, :n2] = 2.0 * theta[i] * R[i][s1, :] * f1[s1, :]
        K[:n1, ci] = -2.0 * theta[i] * R[i][:, s2] * f1[:, s2]
        Rgg_i = R[i][np.ix_(s1, s2)]
        f1gg, f2gg = f1[np.ix_(s1, s2)], f2[np.ix_(s1, s2)]
        K[ri, ci] = -2.0 * theta[i] * f1gg - 4.0 * theta[i] ** 2 * Rgg_i ** 2 * f2gg
        for j in range(i + 1, d):
            rj = slice(n1 + j * g1, n1 + (j + 1) * g1)
            cj = slice(n2 + j * g2, n2 + (j + 1) * g2)
            term = -4.0 * theta[i] * theta[j] * (Rgg_i * R[j][np.ix_(s1, s2)] * f2gg)
            K[ri, cj] += term
            K[rj, ci] += term
    return K


def kern_grad_dalpha(X, theta, kernel, mask=None):
    """d K / d alpha of the rational-quadratic kernel, [N, N] (kernel/KernelRatQuad.py:752-843): the blocks of K with
    (phi, phi', phi'') replaced by their alpha-derivatives."""
    theta = np.asarray(theta, dtype=float)
    s = _sqdist(calc_rtensor(X, X), theta)
    d0, d1, d2 = _radial_dalpha(kernel, s)
    return _blocks_from_profile(X, X, theta, d0, d1, d2, mask, mask)


def kern_grad(X, Y, theta, mask1=None, mask2=None, kernel=None):
    """Gradient-enhanced kernel matrix (kernel/KernelSqExp.py:322-410).

    Blocks: K00 = k; K_i0 = -2 th_i r_i k (:392); K_0j = +2 th_j r_j k (:393);
    K_ii = (2 th_i - 4 th_i^2 r_i^2) k (:396); K_ij = -4 th_i th_j r_i r_j k (:406-408).
    Gradient rows/cols are restricted to the masked points (:349-377).
    """
    theta = np.asarray(theta, dtype=float)
    if kernel is not None and _kernel_spec(kernel)[0] != "SqExp":
        # kernel/KernelMatern5f2.py:354-451 (KernelMatern5f2GradMod), kernel/KernelRatQuad.py:439-553
        f0, f1, f2, _ = _radial(kernel, _sqdist(calc_rtensor(X, Y), theta))
        return _blocks_from_profile(X, Y, theta, f0, f1, f2, mask1, mask2)
    n1, d = X.shape
    n2 = Y.shape[0]
    s1, s2 = _sel(n1, mask1), _sel(n2, mask2)
    g1, g2 = s1.size, s2.size
    R = calc_rtensor(X, Y)
    k = kern_base(X, Y, theta)
    K = np.zeros((n1 + g1 * d, n2 + g2 * d))
    K[:n1, :n2] = k
    for i in range(d):
        ri = slice(n1 + i * g1, n1 + (i + 1) * g1)
        ci = slice(n2 + i * g2, n2 + (i + 1) * g2)
        K[ri, :n2] = -2.0 * theta[i] * R[i][s1, :] * k[s1, :]
        K[:n1, ci] = 2.0 * theta[i] * R[i][:, s2] * k[:, s2]
        Rgg_i = R[i][np.ix_(s1, s2)]
        kgg = k[np.ix_(s1, s2)]
        K[ri, ci] = (2.0 * theta[i] - 4.0 * theta[i] ** 2 * Rgg_i ** 2) * kgg
        for j in range(i + 1, d):
            rj = slice(n1 + j * g1, n1 + (j + 1) * g1)
            cj = slice(n2 + j * g2, n2 + (j + 1) * g2)
            term = -4.0 * theta[i] * theta[j] * (Rgg_i * R[j][np.ix_(s1, s2)] * kgg)
            K[ri, cj] += term
            K[rj, ci] += term
    return K


def _kern_grad_dtheta_profile(X, theta, kernel, mask=None):
    """d K / d theta_m for the Matern-5/2 and rational-quadratic kernels (kernel/KernelMatern5f2.py:534-643,
    kernel/KernelRatQuad.py:636-749) in profile form: r_m^2 times the blocks one s-derivative up, plus the explicit
    theta_m dependence:  dK_i0 += 2 d_im r_i f1 ; dK_ij += -2 d_ij d_im f1 - 4 (d_im th_j + d_jm th_i) r_i r_j f2."""
    theta = np.asarray(theta, dtype=float)
    n, d = X.shape
    s = _sel(n, mask)
    g = s.size
    N = n + g * d
    R = calc_rtensor(X, X)
    _, f1, f2, f3 = _radial(kernel, _sqdist(R, theta))
    up = _blocks_from_profile(X, X, theta, f1, f2, f3, mask, mask)
    out = np.zeros((d, N, N))

    def blk(i):
        return slice(n + i * g, n + (i + 1) * g)

    def rep(r2):    # r_m^2 on the block structure [values | d gradient blocks]
        row = np.hstack([r2] + [r2[:, s]] * d)
        return np.vstack([row] + [row[s, :]] * d)

    gg = np.ix_(s, s)
    for m in range(d):
        D = out[m]
        D[:] = rep(R[m] ** 2) * up
        D[blk(m), :n] += 2.0 * R[m][s, :] * f1[s, :]
        D[:n, blk(m)] += -2.0 * R[m][:, s] * f1[:, s]
        D[blk(m), blk(m)] += -2.0 * f1[gg]
        for j in range(d):
            t = -4.0 * theta[j] * R[m][gg] * R[j][gg] * f2[gg]
            D[blk(m), blk(j)] += t
            D[blk(j), blk(m)] += t
    return out


def kern_grad_dtheta(X, theta, mask=None, kernel=None):
    """d K / d theta_m for all m -> [d, N, N]  (kernel/KernelSqExp.py:471-568).

    Restated from the closed form (SURVEY.md 8a):
      dK00 = -r_m^2 k ; dK_i0 = -r_m^2 K_i0 - 2 d_im r_m k ; dK_0j = transpose sign ;
      dK_ij = -r_m^2 K_ij + (2 d_ij d_im - 4 (d_im th_j + d_jm th_i) r_i r_j) k.
    With a mask this is the derivative of K_full[sel, sel] (the semantics the builder has);
    the reference's jit is only right for None/prefix masks (SURVEY.md section 4).
    """
    if kernel is not None and _kernel_spec(kernel)[0] != "SqExp":
        return _kern_grad_dtheta_profile(X, theta, kernel, mask)
    theta = np.asarray(theta, dtype=float)
    n, d = X.shape
    s = _sel(n, mask)
    g = s.size
    N = n + g * d
    R = calc_rtensor(X, X)
    k = kern_base(X, X, theta)
    K = kern_grad(X, X, theta, mask, mask)
    out = np.zeros((d, N, N))

    def blk(i):
        return slice(n + i * g, n + (i + 1) * g)

    for m in range(d):
        r2 = R[m] ** 2
        D = out[m]
        D[:n, :n] = -r2 * k
        for i in range(d):
            D[blk(i), :n] = -r2[s, :] * K[blk(i), :n]
            D[:n, blk(i)] = -r2[:, s] * K[:n, blk(i)]
            for j in range(d):
                D[blk(i), blk(j)] = -r2[np.ix_(s, s)] * K[blk(i), blk(j)]
        D[blk(m), :n] += -2.0 * R[m][s, :] * k[s, :]
        D[:n, blk(m)] += 2.0 * R[m][:, s] * k[:, s]
        kgg = k[np.ix_(s, s)]
        D[blk(m), blk(m)] += 2.0 * kgg
        for j in range(d):
            t = -4.0 * theta[j] * R[m][np.ix_(s, s)] * R[j][np.ix_(s, s)] * kgg
            D[blk(m), blk(j)] += t
            D[blk(j), blk(m)] += t
    return out


# ----------------------------------------------------------------------------------------------
# nugget (base/GpWellCond.py)
# ----------------------------------------------------------------------------------------------

def vreq_rescale_origin(n, d):
    """base/GpWellCond.py:26-40."""
    if n == 1:
        return 1.0
    ds = 2.0 * np.sqrt(d)
    v = (2.0 + np.sqrt(4.0 + 2.0 * np.exp(2.0) * np.log((n - 1) * (1.0 + ds) / 2.0))) / np.exp(1.0)
    return min(v, ds)


def nugget(n, d, mode, cond_max_target=1e10, use_grad=True, eta_set_mtd="Kbase_eta", eta_dflt=1e-8, kernel=None):
    """(eta_Kbase, eta_Kgrad) per conditioning mode  (base/GpWellCond.py:116-154, :78-99, :109-114)."""
    if eta_set_mtd == "dflt_eta":
        return eta_dflt, eta_dflt
    eta_base = n / (cond_max_target - 1.0)
    if not use_grad:
        return eta_base, np.nan
    if n == 1:
        return eta_base, eta_base
    if mode == "precon":
        if _kernel_spec(kernel)[0] == "Ma5f2":      # base/GpWellCond.py:130-132
            al = (np.sqrt(3.0 * d) - 1.0 + np.sqrt(15.0 * d + 2.0 * np.sqrt(3.0 * d) + 1.0)) / (2.0 * (3.0 * d + np.sqrt(3.0 * d)))
            u = (n - 1) * (1.0 + (d + np.sqrt(3.0 * d)) * al + d * (1.0 + np.sqrt(3.0 * d)) * al ** 2) * np.exp(-np.sqrt(3.0 * d) * al)
        else:                                        # 'SqExp' and 'RatQu' share the bound (:127-129)
            u = 0.5 * (n - 1) * (1.0 + np.sqrt(1.0 + 4.0 * d)) * np.exp(-(1.0 + 2.0 * d - np.sqrt(1.0 + 4.0 * d)) / (4.0 * d))
        return eta_base, (1.0 + u) / (cond_max_target - 1.0)
    if "rescale" in mode:
        vmin = vreq_rescale_origin(n, d)
        vf = 2.0 * np.sqrt(d) / vmin
        return eta_base, (1.0 + (n - 1) * vf * np.exp(1.0 / vf - 1.0)) / (cond_max_target - 1.0)
    if eta_set_mtd == "Kbase_eta_w_dim":
        return eta_base, eta_base * (d + 1)
    return eta_base, eta_base


# ----------------------------------------------------------------------------------------------
# data packing, mean function
# ----------------------------------------------------------------------------------------------

def make_data_vec(fval, grad=None):
    """[fval, grad.reshape(order='F')]  (base/CommonFun.py:152-173)."""
    if grad is None:
        return np.atleast_1d(fval).astype(float)
    return np.hstack((fval, grad.reshape(grad.size, order="F")))


def aug_vand(n, n_g, d):
    """Constant-mean augmented Vandermonde column H = [1_n ; 0]  (eval/GpMeanFun.py:172-191)."""
    H = np.zeros((n + n_g * d, 1))
    H[:n, 0] = 1.0
    return H


# ----------------------------------------------------------------------------------------------
# covariance assembly + factorisation  (kernel/Kernel.py:140-307)
# ----------------------------------------------------------------------------------------------

@dataclasses.dataclass
class KAll:
    Kern: np.ndarray
    Kcor: np.ndarray | None
    Kcov: np.ndarray
    chofac: tuple | None       # (factor, lower) exactly as the reference returns it
    eta: float
    pvec: np.ndarray | None
    Ltilde: np.ndarray | None  # precon: chol(varK (Kcor + eta I)), lower
    idx_eta_argmax: int | None = None


def all_K_w_chofac(X, theta, mode="precon", eta=None, noise_vec=None, varK=1.0, mask=None,
                   cond_max_target=1e10, eta_is_const=True, calc_chofac=True, kernel=None):
    """Faithful restatement of calc_all_K_w_chofac (kernel/Kernel.py:213-302) with use_grad=True.

    precon (:220-266): p = sqrt(diag(K + noise/varK)); Kcor = P^-1 (K+noise/varK) P^-1;
    Kt = varK (Kcor + eta I); Kcov = P Kt P; factor returned as (P Lt, lower=True).
    otherwise (:268-302): Kcov = varK (K + noise/varK + eta I); cho_factor default (upper).
    """
    K = kern_grad(X, X, theta, mask, mask, kernel=kernel)
    N = K.shape[0]
    if noise_vec is None:
        noise_vec = np.zeros(N)
    Kw = K + np.diag(noise_vec / varK)
    idx = None
    if mode == "precon":
        p = np.sqrt(np.diag(Kw))
        pinv = 1.0 / p
        Kcor = (pinv[:, None] * Kw) * pinv[None, :]      # (P_inv @ Kw) @ P_inv, same rounding
        if not eta_is_const:
            rs = np.sum(np.abs(Kcor), axis=1)
            idx = int(np.argmax(rs))
            eta = rs[idx] / (cond_max_target - 1.0)
        Kt = varK * (Kcor + eta * np.eye(N))
        Kcov = (p[:, None] * Kt) * p[None, :]
        fac = Lt = None
        if calc_chofac:
            try:
                Lt = linalg.cholesky(Kt, lower=True)
                fac = (p[:, None] * Lt, True)
            except linalg.LinAlgError:
                fac = Lt = None
        return KAll(K, Kcor, Kcov, fac, eta, p, Lt, idx)
    if not eta_is_const:
        rs = np.sum(np.abs(K), axis=1)
        idx = int(np.argmax(rs))
        eta = rs[idx] / (cond_max_target - 1.0)
    Kcov = varK * (Kw + eta * np.eye(N))
    fac = None
    if calc_chofac:
        try:
            fac = linalg.cho_factor(Kcov)
        except linalg.LinAlgError:
            fac = None
    return KAll(K, None, Kcov, fac, eta, None, None, idx)


def kerngrad_hp(X, theta, mode, eta, mask=None, kernel=None):
    """d(K + eta-term)/d[theta.., alpha?] stack, noise-free  (optz/GpHparaGrad.py:13-56).

    precon adds 2 eta gamma_m dgamma_m/dtheta_m = c eta on the diagonal of gradient block m (:40-50): d(eta p^2)/d theta_m
    (c = 2; Matern-5/2: 5/3).  A kernel with a hyper-parameter of its own (RatQu) appends dK/dalpha (:52-55).
    """
    n, d = X.shape
    g = _sel(n, mask).size
    D = kern_grad_dtheta(X, theta, mask, kernel=kernel)
    if mode == "precon":
        for m in range(d):
            idx = np.arange(n + m * g, n + (m + 1) * g)
            D[m, idx, idx] += kernel_diag_coef(kernel) * eta
    if _kernel_spec(kernel)[0] == "RatQu":
        D = np.concatenate((D, kern_grad_dalpha(X, theta, kernel, mask)[None]), axis=0)
    return D


# ----------------------------------------------------------------------------------------------
# LML and gradient
# ----------------------------------------------------------------------------------------------

@dataclasses.dataclass
class Lkd:
    ln_lkd: float | None = None
    ln_lkd_grad: np.ndarray | None = None
    hp_varK: float | None = None
    hp_beta: np.ndarray | None = None
    ln_det: float | None = None
    alpha: np.ndarray | None = None
    chofac_good: bool = True
    eta: float | None = None
    post: tuple | None = None   # (mu, sig, sig2) at the test points handed to lkd_wo_noise_lean


def gls_beta(chofac, H, y):
    """beta = (H^T K^-1 H)^-1 H^T K^-1 y  (eval/GpMeanFun.py:98-108)."""
    invK_H = linalg.cho_solve(chofac, H)
    term1 = np.linalg.solve(H.T @ invK_H, invK_H.T)
    return term1 @ y


def lkd_wo_noise(X, fval, grad, theta, mode="precon", eta=None, mask=None, calc_grad=True,
                 pnlt_grad=0.0, pnlt_val=0.0, kernel=None):
    """Noise-free LML + d/dtheta, adjoint form.  Follows calc_lkd_all (optz/CalcLkd.py:322-339),
    calc_lkd_all_wo_noise (:30-95) and calc_lkd_w_Kern_mtd_adjoint (:149-181) with varK := 1 inside
    K (kernel/Kernel.py:128-138).  Materialises everything exactly as the reference does."""
    n, d = X.shape
    if eta is None:
        eta = nugget(n, d, mode, kernel=kernel)[1]
    ka = all_K_w_chofac(X, theta, mode, eta, None, 1.0, mask, kernel=kernel)
    if ka.chofac is None:
        return Lkd(chofac_good=False, eta=eta)
    g = _sel(n, mask).size
    y = make_data_vec(fval, grad)
    N = y.size
    H = aug_vand(n, g, d)
    beta = gls_beta(ka.chofac, H, y)
    res = y - H @ beta
    alpha = linalg.cho_solve(ka.chofac, res)
    varK = max(1e-32, float(res @ alpha) / N)
    ln_det = 2.0 * np.sum(np.log(np.diag(ka.chofac[0])))
    lml = -(N * np.log(varK) + ln_det) / 2.0 - pnlt_val
    out = Lkd(lml, None, varK, beta, ln_det, alpha, True, eta)
    if calc_grad:
        D = kerngrad_hp(X, theta, mode, eta, mask, kernel=kernel)     # rows: theta_1..d, then alpha (RatQu)
        adj_varK = np.outer(alpha, -alpha / N)
        Kinv = linalg.cho_solve(ka.chofac, np.eye(N))
        adj = -adj_varK * (pnlt_grad + N / (2.0 * varK)) - 0.5 * Kinv
        out.ln_lkd_grad = np.einsum("ijk,jk", D, adj)
    return out


def cross_cov_values(X, Xs, theta):
    """Value columns of calc_KernGrad(Rtensor(X, X*)): Kyx[N, nx] with rows [k ; -2 theta_i r_i k], r = x_train - x_test
    (eval/GpEvalModel.py:133-139, kernel/KernelSqExp.py:392) -- without the nx*d test-gradient columns the reference
    builds and drops."""
    n, d = X.shape
    R = X[:, None, :] - Xs[None, :, :]
    k = np.exp(-np.einsum("abi,i->ab", R ** 2, theta))
    out = np.empty((n * (d + 1), Xs.shape[0]))
    out[:n] = k
    for i in range(d):
        out[n + i * n: n + (i + 1) * n] = -2.0 * theta[i] * R[:, :, i] * k
    return out


def lkd_wo_noise_lean(X, fval, grad, theta, mode="precon", eta=None, calc_grad=True, tile=256, Xs=None):
    """Same quantities as lkd_wo_noise for sizes where the reference cannot run (its dK/dtheta
    tensor is d*N*N*8 bytes).  In-place LAPACK potrf/potri; dK/dtheta contracted tile by tile.
    All gradients used (mask=None).  Must agree with lkd_wo_noise (checked in tests).
    With Xs [nx, d] the posterior of eval_model (eval/GpEvalModel.py:154-168) at the closed-form (beta, varK)
    is taken from the same factor and returned as out.post = (mu, sig, sig2)."""
    n, d = X.shape
    theta = np.asarray(theta, dtype=float)
    if eta is None:
        eta = nugget(n, d, mode)[1]
    K = kern_grad(X, X, theta)
    N = K.shape[0]
    if mode == "precon":
        p = np.sqrt(np.diag(K)).copy()
        K /= p[:, None]
        K /= p[None, :]
    else:
        p = np.ones(N)
    K[np.diag_indices(N)] += eta
    y = make_data_vec(fval, grad)
    H = aug_vand(n, n, d)[:, 0]
    c, info = linalg.lapack.dpotrf(K, lower=1, overwrite_a=1, clean=0)
    if info != 0:
        return Lkd(chofac_good=False, eta=eta)
    rhs = np.stack((y / p, H / p), axis=1)
    sol, _ = linalg.lapack.dpotrs(c, rhs, lower=1)
    beta = float(rhs[:, 1] @ sol[:, 0]) / float(rhs[:, 1] @ sol[:, 1])
    alpha_t = sol[:, 0] - beta * sol[:, 1]
    res_t = rhs[:, 0] - beta * rhs[:, 1]
    varK = max(1e-32, float(res_t @ alpha_t) / N)
    ln_det = 2.0 * np.sum(np.log(np.diag(c) * p))
    lml = -(N * np.log(varK) + ln_det) / 2.0
    out = Lkd(lml, None, varK, np.array([beta]), ln_det, alpha_t / p, True, eta)
    if Xs is not None:
        # mu = beta + K*^T K^-1 (y - H beta); sig2 = 1 - diag(K*^T K^-1 K*) with the varK := 1 factor, in chunks
        mu, sig2 = np.empty(Xs.shape[0]), np.empty(Xs.shape[0])
        for s0 in range(0, Xs.shape[0], 512):
            Kyx = cross_cov_values(X, Xs[s0:s0 + 512], theta)
            mu[s0:s0 + 512] = beta + Kyx.T @ (alpha_t / p)
            Z = linalg.solve_triangular(c, Kyx / p[:, None], lower=True, check_finite=False)
            sig2[s0:s0 + 512] = 1.0 - np.einsum("ij,ij->j", Z, Z)
        out.post = (mu, np.sqrt(np.maximum(sig2, 0.0)) * np.sqrt(varK), sig2)
    if not calc_grad:
        return out
    Kinv, info = linalg.lapack.dpotri(c, lower=1, overwrite_c=1)
    il = np.tril_indices(N, -1)
    Kinv.T[il] = Kinv[il]
    # W = alpha alpha^T/(2 varK) - K^-1/2 in un-preconditioned coordinates
    W = np.outer(alpha_t, alpha_t) / (2.0 * varK) - 0.5 * Kinv
    W /= p[:, None]
    W /= p[None, :]
    gradv = np.zeros(d)
    for a0 in range(0, n, tile):
        a1 = min(n, a0 + tile)
        rows = np.concatenate([np.arange(a0, a1)] + [n + i * n + np.arange(a0, a1) for i in range(d)])
        Xa = X[a0:a1]
        R = Xa[:, None, :] - X[None, :, :]                    # [ta, n, d]
        k = np.exp(-np.einsum("abi,i->ab", R ** 2, theta))
        Wt = W[rows].reshape(d + 1, a1 - a0, d + 1, n)        # [i, a, j, b]
        u = R * theta[None, None, :]
        W00 = Wt[0, :, 0, :]
        Wi0 = Wt[1:, :, 0, :]                                  # [i, a, b]
        W0j = Wt[0, :, 1:, :].transpose(1, 0, 2)               # [j, a, b]
        Wij = Wt[1:, :, 1:, :]                                 # [i, a, j, b]
        Wii = np.einsum("iaib->iab", Wij)
        uT = u.transpose(2, 0, 1)                              # [i, a, b]
        rT = R.transpose(2, 0, 1)
        Wu = np.einsum("iajb,jab->iab", Wij, uT)               # sum_j W_ij u_j
        WTu = np.einsum("iajb,iab->jab", Wij, uT)              # sum_i W_ij u_i
        S = W00 + 2.0 * np.sum(uT * (W0j - Wi0), axis=0) + 2.0 * np.einsum("i,iab->ab", theta, Wii) \
            - 4.0 * np.sum(uT * Wu, axis=0)
        T = 2.0 * rT * (W0j - Wi0) + 2.0 * Wii - 4.0 * rT * (Wu + WTu)
        gradv += np.einsum("ab,mab->m", k, T - rT ** 2 * S[None])
    if mode == "precon":
        dW = np.diag(W)
        for m in range(d):
            gradv[m] += 2.0 * eta * np.sum(dW[n + m * n: n + (m + 1) * n])
    out.ln_lkd_grad = gradv
    return out


def kcov_grad_hp_noisy(X, theta, Kern, mode, eta, varK, has_var_fval, has_var_fgrad, mask=None, kernel=None):
    """dKcov/d[theta.., alpha?, varK, var_fval?, var_fgrad?]  (optz/GpHparaGrad.py:58-155; hp order of
    optz/GpHparaOptz.py:76-126)."""
    n, d = X.shape
    g = _sel(n, mask).size
    N = n + g * d
    stack = []
    Dth = varK * kern_grad_dtheta(X, theta, mask, kernel=kernel)
    if mode == "precon":
        for i in range(d):
            Dth[i] += np.diag(np.diag(Dth[i])) * eta            # :105-109
    stack.extend(list(Dth))
    if _kernel_spec(kernel)[0] == "RatQu":                      # :111-123 (diag(dK/dalpha) = 0: no nugget term)
        Da = varK * kern_grad_dalpha(X, theta, kernel, mask)
        if mode == "precon":
            Da = Da + np.diag(np.diag(Da)) * eta
        stack.append(Da)
    if mode == "precon":
        stack.append(Kern + eta * np.diag(np.diag(Kern)))        # :132-133
    else:
        stack.append(Kern + eta * np.eye(N))
    sc = (1.0 + eta) if mode == "precon" else 1.0
    if has_var_fval:
        stack.append(sc * np.diag(np.hstack((np.ones(n), np.zeros(g * d)))))
    if has_var_fgrad:
        stack.append(sc * np.diag(np.hstack((np.zeros(n), np.ones(g * d)))))
    return np.array(stack)


def lkd_w_noise(X, fval, grad, theta, varK, noise_vec, mode="precon", eta=None, mask=None,
                calc_grad=True, has_var_fval=False, has_var_fgrad=False, kernel=None):
    """Noisy-data LML + gradient wrt [theta, varK, (var_fval), (var_fgrad)], adjoint form
    (optz/CalcLkd.py:185-251, :299-320).  LML = -(ln det Kcov + res^T alpha)/2."""
    n, d = X.shape
    if eta is None:
        eta = nugget(n, d, mode, kernel=kernel)[1]
    ka = all_K_w_chofac(X, theta, mode, eta, noise_vec, varK, mask, kernel=kernel)
    if ka.chofac is None:
        return Lkd(chofac_good=False, eta=eta)
    g = _sel(n, mask).size
    y = make_data_vec(fval, grad)
    N = y.size
    H = aug_vand(n, g, d)
    beta = gls_beta(ka.chofac, H, y)
    res = y - H @ beta
    alpha = linalg.cho_solve(ka.chofac, res)
    ln_det = 2.0 * np.sum(np.log(np.diag(ka.chofac[0])))
    lml = -(ln_det + float(res @ alpha)) / 2.0
    out = Lkd(lml, None, varK, beta, ln_det, alpha, True, eta)
    if calc_grad:
        D = kcov_grad_hp_noisy(X, theta, ka.Kern, mode, eta, varK, has_var_fval, has_var_fgrad, mask, kernel=kernel)
        adj = 0.5 * (np.outer(alpha, alpha) - linalg.cho_solve(ka.chofac, np.eye(N)))
        out.ln_lkd_grad = np.einsum("ijk,jk", D, adj)
    return out


# ----------------------------------------------------------------------------------------------
# condition number and its gradient  (optz/GpHparaCon.py:161-235; kernel/Kernel.py:240,280)
# ----------------------------------------------------------------------------------------------

def cond_l2_w_grad(Kmat, Kgrad_hp=None):
    """kappa_2 = np.linalg.cond(K, 2); d kappa/d hp = sum((v_max v_max^T - kappa v_min v_min^T) * dK/dhp)
    / max(lambda_min, 1e-16) from a full eigen-decomposition (optz/GpHparaCon.py:161-193).  The reference calls the
    general np.linalg.eig on the symmetric matrix; eigh gives the same extreme pairs with orthonormal vectors."""
    cond = float(np.linalg.cond(Kmat, p=2))
    if Kgrad_hp is None:
        return cond, None
    w, V = np.linalg.eigh(Kmat)
    vmax, vmin = V[:, -1], V[:, 0]
    emin = max(float(w[0]), 1e-16)
    diff = np.outer(vmax, vmax) - cond * np.outer(vmin, vmin)
    return cond, np.array([np.sum(diff * Kgrad_hp[i]) / emin for i in range(Kgrad_hp.shape[0])])


def cond_fro_w_grad(Kmat, Kgrad_hp=None):
    """Frobenius condition number |K|_F |K^-1|_F and its gradient sum((frac K - K^-3 / frac) * dK/dhp),
    frac = |K^-1|_F / |K|_F  (optz/GpHparaCon.py:237-261)."""
    Kinv = np.linalg.inv(Kmat)
    nk, ni = np.linalg.norm(Kmat, "fro"), np.linalg.norm(Kinv, "fro")
    if Kgrad_hp is None:
        return nk * ni, None
    frac = ni / nk
    W = frac * Kmat - (Kinv @ Kinv @ Kinv) / frac
    return nk * ni, np.sum(W[None, :, :] * Kgrad_hp, axis=(1, 2))


def cond_wo_noise(X, theta, mode, eta, mask=None, calc_grad=True):
    """Condition number of the matrix calc_lkd_all factors for noise-free data (K + eta-term, varK := 1) and its
    theta-gradient (optz/CalcLkd.py:322-343).  The reference has no gradient in precon mode (:171-173)."""
    ka = all_K_w_chofac(X, theta, mode, eta, None, 1.0, mask, calc_chofac=False)
    if mode == "precon":
        # reference quirk: without calc_grad the number is kappa(Kcor + eta I) (kernel/Kernel.py:240); with calc_grad
        # calc_lkd_all overwrites it with kappa of the UN-preconditioned Kcov = P (Kcor + eta I) P (optz/CalcLkd.py:341)
        N = ka.Kern.shape[0]
        return cond_l2_w_grad(ka.Kcov if calc_grad else ka.Kcor + eta * np.eye(N))[0], None
    return cond_l2_w_grad(ka.Kcov, kerngrad_hp(X, theta, mode, eta, mask) if calc_grad else None)


def cond_w_noise(X, theta, varK, noise_vec, mode, eta, has_var_fval=False, has_var_fgrad=False, mask=None,
                 calc_grad=True):
    """Noisy-data counterpart: kappa_2(Kcov) and d/d[theta.., varK, var_fval?, var_fgrad?] (optz/CalcLkd.py:299-320)."""
    ka = all_K_w_chofac(X, theta, mode, eta, noise_vec, varK, mask, calc_chofac=False)
    if mode == "precon":   # same quirk as cond_wo_noise
        N = ka.Kern.shape[0]
        return cond_l2_w_grad(ka.Kcov if calc_grad else varK * (ka.Kcor + eta * np.eye(N)))[0], None
    D = kcov_grad_hp_noisy(X, theta, ka.Kern, mode, eta, varK, has_var_fval, has_var_fgrad, mask)
    return cond_l2_w_grad(ka.Kcov, D)


# ----------------------------------------------------------------------------------------------
# posterior  (eval/GpEvalModel.py:17-57, 59-198)
# ----------------------------------------------------------------------------------------------

def eval_model(X, fval, grad, theta, varK, beta, Xs, mode="precon", eta=None, noise_vec=None, mask=None, kernel=None):
    """mu = beta + K*^T K^-1 (y - H beta); sig = sqrt(varK) sqrt(max(0, 1 - diag(K*^T K^-1 K*)))
    with the factor built for varK := 1 (kernel/Kernel.py:196-197)."""
    n, d = X.shape
    if eta is None:
        eta = nugget(n, d, mode, kernel=kernel)[1]
    ka = all_K_w_chofac(X, theta, mode, eta, noise_vec, 1.0, mask, kernel=kernel)
    g = _sel(n, mask).size
    y = make_data_vec(fval, grad)
    H = aug_vand(n, g, d)
    fdiff = y - H @ np.atleast_1d(beta)
    a = linalg.cho_solve(ka.chofac, fdiff)
    Kyx = kern_grad(X, Xs, theta, mask, None, kernel=kernel)[:, : Xs.shape[0]]
    KinvK = linalg.cho_solve(ka.chofac, Kyx)
    sig2 = 1.0 - np.einsum("ij,ij->j", Kyx, KinvK)
    n_neg = int(np.sum(sig2 < 0))
    sig = np.sqrt(np.maximum(sig2, 0.0)) * np.sqrt(varK)
    mu = float(np.atleast_1d(beta)[0]) + Kyx.T @ a
    return mu, sig, sig2, n_neg


def eval_model_grad(X, fval, grad, theta, varK, beta, Xs, mode="precon", eta=None, noise_vec=None, mask=None,
                    kernel=None):
    """eval_model(calc_grad=True): additionally d mu / d x and d sig / d x, [nx, d]
    (eval/GpEvalModel.py:134-139 test-gradient columns of K(X, X*); :319-354 calc_dmudx / calc_dsigdx)."""
    n, d = X.shape
    nx = Xs.shape[0]
    if eta is None:
        eta = nugget(n, d, mode, kernel=kernel)[1]
    ka = all_K_w_chofac(X, theta, mode, eta, noise_vec, 1.0, mask, kernel=kernel)
    g = _sel(n, mask).size
    y = make_data_vec(fval, grad)
    H = aug_vand(n, g, d)
    a = linalg.cho_solve(ka.chofac, y - H @ np.atleast_1d(beta))
    Kg = kern_grad(X, Xs, theta, mask, None, kernel=kernel)           # [N, nx (1 + d)]
    Kyx, dKxy = Kg[:, :nx], Kg[:, nx:].T               # dKxy[(j, x), row]
    KinvK = linalg.cho_solve(ka.chofac, Kyx)           # [N, nx]
    sig2 = 1.0 - np.einsum("ij,ij->j", Kyx, KinvK)
    sigK = np.sqrt(varK)
    sig = np.sqrt(np.maximum(sig2, 0.0)) * sigK
    mu = float(np.atleast_1d(beta)[0]) + Kyx.T @ a
    dmudx = (dKxy @ a).reshape((nx, d), order="F")
    inv_sig = np.divide(1.0, sig, out=np.zeros_like(sig), where=sig != 0)
    t2 = np.sum(dKxy * np.tile(KinvK.T, (d, 1)), axis=1).reshape((nx, d), order="F") * sigK ** 2
    return mu, sig, dmudx, -inv_sig[:, None] * t2


def kern_hess_x(X, xs, theta, kernel=None):
    """Second derivatives of the cross covariance k*(x) with respect to the test point x, [d, d, N], every training
    point carrying a gradient (kernel/KernelSqExp.py:66-88 value entries, :432-468 gradient entries; the reference
    builds them with R = x_test - x_train)."""
    n, d = X.shape
    rho = xs[None, :] - X                                # [n, d] = x_test - x_train
    if kernel is not None and _kernel_spec(kernel)[0] != "SqExp":
        # kernel/KernelMatern5f2.py:54-96, 272-331; kernel/KernelRatQuad.py:54-97, 556-633, in profile form
        # (rho = -r: the odd powers of r change sign against the training-minus-test convention of the CUDA kernels)
        _, f1, f2, f3 = _radial(kernel, np.sum(theta[None, :] * rho ** 2, axis=1))
        H = np.zeros((d, d, n * (d + 1)))
        for kk in range(d):
            for i in range(d):
                H[kk, i, :n] = 2.0 * theta[i] * (i == kk) * f1 + 4.0 * theta[i] * theta[kk] * rho[:, i] * rho[:, kk] * f2
                for j in range(d):
                    H[kk, i, n + j * n: n + (j + 1) * n] = (
                        -4.0 * theta[i] * theta[j] * ((i == kk) * rho[:, j] + (j == kk) * rho[:, i]) * f2
                        - 4.0 * (i == j) * theta[i] * theta[kk] * rho[:, kk] * f2
                        - 8.0 * theta[i] * theta[j] * theta[kk] * rho[:, i] * rho[:, j] * rho[:, kk] * f3)
        return H
    k = np.exp(-np.sum(theta[None, :] * rho ** 2, axis=1))
    H = np.zeros((d, d, n * (d + 1)))
    for kk in range(d):
        for i in range(d):
            H[kk, i, :n] = (-2.0 * theta[i] * (i == kk) + 4.0 * theta[i] * theta[kk] * rho[:, i] * rho[:, kk]) * k
            for j in range(d):
                H[kk, i, n + j * n: n + (j + 1) * n] = (
                    -4.0 * theta[i] * theta[j] * ((i == kk) * rho[:, j] + (j == kk) * rho[:, i])
                    - 4.0 * (i == j) * theta[i] * theta[kk] * rho[:, kk]
                    + 8.0 * theta[i] * theta[j] * theta[kk] * rho[:, i] * rho[:, j] * rho[:, kk]) * k
    return H


def eval_model_hess(X, fval, grad, theta, varK, beta, xs, mode="precon", eta=None, kernel=None, noise_vec=None,
                    mask=None):
    """eval_model(calc_grad=True, calc_hess=True) at ONE point: (mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2)
    (eval/GpEvalModel.py:175-180, 356-382).  noise_vec and mask as in eval_model_grad (grad then holds the rows of
    the masked points only).  With a mask the rows of k* are a subset of the all-gradient rows, in the order
    value p, then gradient (j, slot) = all-gradient row n + j n + p; the masked Hessian selects those rows."""
    n, d = X.shape
    if eta is None:
        eta = nugget(n, d, mode, kernel=kernel)[1]
    xs = np.atleast_2d(xs)
    mu, sig, dmu, dsig = eval_model_grad(X, fval, grad, theta, varK, beta, xs, mode, eta, noise_vec, mask, kernel=kernel)
    ka = all_K_w_chofac(X, theta, mode, eta, noise_vec, 1.0, mask, kernel=kernel)
    sel = _sel(n, mask)
    y = make_data_vec(fval, grad)
    H = aug_vand(n, sel.size, d)
    a = linalg.cho_solve(ka.chofac, y - H @ np.atleast_1d(beta))
    Kg = kern_grad(X, xs, theta, mask, None, kernel=kernel)
    Kyx, dKxy = Kg[:, :1], Kg[:, 1:].T
    KinvK = linalg.cho_solve(ka.chofac, Kyx)[:, 0]
    rows = np.concatenate([np.arange(n)] + [n + j * n + sel for j in range(d)])
    d2K = kern_hess_x(X, xs[0], theta, kernel=kernel)[:, :, rows]
    d2mu = d2K @ a
    term1 = d2K @ KinvK
    term2 = dKxy @ linalg.cho_solve(ka.chofac, dKxy.T)
    d2sig2 = -2.0 * varK * (term1 + term2)
    s = sig[0] if sig[0] != 0 else np.nan
    d2sig = (d2sig2 - 2.0 * np.outer(dsig[0], dsig[0])) / (2.0 * s)
    return mu, sig, dmu, dsig, d2mu[None], d2sig[None]


# ----------------------------------------------------------------------------------------------
# rescaling (base/Rescaling.py:72-125, 199-214; SURVEY appendix A)
# ----------------------------------------------------------------------------------------------

def rescale_origin(X, fval, grad, dist_set):
    """x_s = (x - x[last]) c with c = dist_set / min pairwise distance; f_s = (f - f[last]) s with
    s = 100/(max f - min f); grad_s = grad s / c."""
    from scipy.spatial.distance import pdist
    n = X.shape[0]
    c = 1.0 if n == 1 else dist_set / max(1e-14, float(np.min(pdist(X))))
    xs = (X - X[-1][None, :]) * c
    rng_f = max(1e-20, float(np.max(fval) - np.min(fval)))
    s = 1.0 if n == 1 else 100.0 / rng_f
    fs = (fval - fval[-1]) * s
    gs = grad * (s / c)
    return xs, fs, gs, c, s, fval[-1]


# ----------------------------------------------------------------------------------------------
# direct (non-adjoint) likelihood form, lkd_use_adj_mtd = False
# ----------------------------------------------------------------------------------------------

def lkd_direct(X, fval, grad, theta, mode="precon", eta=None, mask=None, kernel=None, varK=None, noise_vec=None,
               has_var_fval=False, has_var_fgrad=False, pnlt_grad=0.0):
    """The quantities the reference only returns with lkd_use_adj_mtd = False: (ln_lkd_grad, hp_beta_grad [1, n_hp],
    hp_varK_grad or None, ln_det_Kmat_grad).  Noise-free (varK None): optz/CalcLkd.py:64-85 with calc_lkd_opt_varK
    (:104-116), calc_detKmat (:349-367), calc_lkd_w_Kern_mtd_direct (:135-147) and the beta gradient of
    eval/GpMeanFun.py:110-120.  Noisy: optz/CalcLkd.py:206-207, 238-241, 253-265."""
    n, d = X.shape
    if eta is None:
        eta = nugget(n, d, mode, kernel=kernel)[1]
    noisy = varK is not None
    ka = all_K_w_chofac(X, theta, mode, eta, noise_vec if noisy else None, varK if noisy else 1.0, mask, kernel=kernel)
    g = _sel(n, mask).size
    y = make_data_vec(fval, grad)
    N = y.size
    H = aug_vand(n, g, d)
    if noisy:
        D = kcov_grad_hp_noisy(X, theta, ka.Kern, mode, eta, varK, has_var_fval, has_var_fgrad, mask, kernel=kernel)
    else:
        D = kerngrad_hp(X, theta, mode, eta, mask, kernel=kernel)
    invK_H = linalg.cho_solve(ka.chofac, H)
    term1 = np.linalg.solve(H.T @ invK_H, invK_H.T)
    beta = term1 @ y
    term2 = invK_H @ beta - linalg.cho_solve(ka.chofac, y)
    beta_grad = np.einsum("ij,kjl,l->ik", term1, D, term2)
    model_grad = H @ beta_grad
    res = y - H @ beta
    a = linalg.cho_solve(ka.chofac, res)
    ln_det_grad = np.array([np.trace(linalg.cho_solve(ka.chofac, D[i])) for i in range(D.shape[0])])
    if noisy:
        lkd_grad = -0.5 * ln_det_grad + 0.5 * np.einsum("i,kij,j", a, D, a) + a @ model_grad
        return lkd_grad, beta_grad, None, ln_det_grad
    vK = max(1e-32, float(res @ a) / N)
    varK_grad = (-2.0 * a @ model_grad - np.einsum("i,kij,j", a, D, a)) / N
    lkd_grad = -0.5 * (N * (varK_grad / vK) + ln_det_grad) - pnlt_grad * varK_grad
    return lkd_grad, beta_grad, varK_grad, ln_det_grad
