"""CPU: the batched surrogate Hessians without a device -- the batched reference (tests/hess_batch_oracle.py) against
the oracle's one-point eval_model_hess at every point, the argument codes of gegp_predict_hess_batch, and the d2sig/dx2 helper that
GaussianProcess.eval_model and eval_model_hess_batch share."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))   # tests/hess_batch_oracle.py, whatever the import mode
from oracle import gegp_oracle as O  # noqa: E402
from hess_batch_oracle import eval_model_hess_batch  # noqa: E402

KERNELS = {"SqExp": None, "Ma5f2": "Ma5f2", "RatQu": ("RatQu", 0.7)}


def _problem(n, d, seed, kernel, *, masked=False, noisy=False, mode="precon"):
    x, f, g = O.synthetic_problem(n, d, seed)
    mask = None
    if masked:
        mask = np.random.default_rng(seed + 1).uniform(size=n) > 0.3
        mask[0], mask[1] = False, True
    gin = g if mask is None else g[mask]
    ng = n if mask is None else int(np.sum(mask))
    N = n + ng * d
    noise = np.concatenate([np.linspace(1e-4, 1e-2, n), np.linspace(1e-3, 3e-2, N - n)]) if noisy else None
    th = np.linspace(0.4, 0.9, d)
    eta = O.nugget(n, d, mode, kernel=kernel)[1]
    return (x, f, gin, th, 2.5, np.array([float(np.mean(f))])), dict(mode=mode, eta=eta, kernel=kernel, noise_vec=noise,
                                                                      mask=mask)


CASES = [("SqExp", False, False, "precon"), ("SqExp", True, True, "base"), ("Ma5f2", True, False, "precon"),
         ("Ma5f2", False, True, "base"), ("RatQu", True, True, "precon"), ("RatQu", False, False, "base")]


@pytest.mark.parametrize("kname,masked,noisy,mode", CASES)
def test_oracle_batch_is_the_one_point_hessian_at_every_point(kname, masked, noisy, mode):
    args, kw = _problem(16, 3, 4, KERNELS[kname], masked=masked, noisy=noisy, mode=mode)
    xs = np.random.default_rng(5).uniform(-1.8, 1.8, (6, 3))
    xs[-1] = args[0][3]                                   # exactly on a training point (sig ~ sqrt(nugget))
    got = eval_model_hess_batch(*args, xs, **kw)
    refs = [O.eval_model_hess(*args, xs[i], **kw) for i in range(xs.shape[0])]
    on = xs.shape[0] - 1
    for k in range(6):
        ref = np.stack([np.asarray(r[k])[0] for r in refs])
        # mu and its derivatives to rounding at every point; sigma is sqrt(1 - k*^T K^-1 k*), whose cancellation the two
        # summation orders resolve differently: the sigma-derived outputs to the project's 1e-6 of their largest entry,
        # away from the data (on a training point d sigma / d x divides by sigma ~ sqrt(nugget))
        a, b = (got[k], ref) if k in (0, 2, 4) else (got[k][:on], ref[:on])
        tol = 1e-12 if k in (0, 2, 4) else 1e-6
        assert a.shape == b.shape
        assert np.max(np.abs(a - b)) <= tol * np.max(np.abs(b)), k


def test_oracle_batch_of_no_points():
    args, kw = _problem(10, 2, 1, None)
    out = eval_model_hess_batch(*args, np.zeros((0, 2)), **kw)
    assert [o.shape for o in out] == [(0,), (0,), (0, 2), (0, 2), (0, 2, 2), (0, 2, 2)]


def test_argument_codes_and_dimension_bound_without_touching_the_gpu():
    from gpgradpy_b200 import _lib
    lib = _lib.load()
    f = lib.gegp_predict_hess_batch
    P = 16   # any non-NULL, 16-byte aligned value: every call below returns before touching memory

    def call(**over):
        a = dict(n=4, n_g=4, d=3, X=P, slot=0, theta=P, kernel=_lib.KERNEL_SQEXP, khp=0.0, A=P, lda=16, dinv=P, p=P,
                 alpha=P, mode=_lib.MODE_PRECON, beta=0.0, varK=1.0, Xs=P, nx=2, mu=P, sig=P, sig2=0, dmu=P, dsig=P,
                 h3=P, nneg=0, work=P, wbytes=1 << 30, stream=0)
        a.update(over)
        return f(*a.values())

    assert call(n=0) == -1 and call(n_g=5) == -1 and call(d=0) == -1
    # the contraction's shared-memory tiles fit up to d = 421; nx = 0 returns after the checks
    assert call(d=422, lda=1696) == -3
    assert call(d=64, lda=320, nx=0) == 0 and call(d=421, lda=1696, nx=0) == 0
    assert call(kernel=7) == -50 and call(kernel=_lib.KERNEL_RATQUAD, khp=0.0) == -50
    assert call(X=0) == -4
    assert call(n_g=2, slot=0) == -5
    assert call(theta=0) == -6
    assert call(A=0) == -7
    assert call(lda=15) == -8 and call(lda=17) == -8
    assert call(dinv=0) == -9
    assert call(p=0) == -10
    assert call(alpha=0) == -11
    assert call(Xs=0) == -15
    assert call(nx=-1) == -16
    assert call(mu=0) == -17
    assert call(sig=0) == -18
    assert call(dmu=0) == -20
    assert call(dsig=0) == -21
    assert call(h3=0) == -22
    assert call(work=0) == -24 and call(work=8) == -24
    # N = 16, ld 16: gegp_dinv_doubles(16) * 8 bytes fixed, then ((d + 1) * 16 + 128) * 8 bytes per point
    fixed, per = lib.gegp_dinv_doubles(16) * 8, (4 * 16 + 128) * 8
    assert call(wbytes=fixed + per - 8) == -25 and call(wbytes=fixed) == -25


def test_d2sig_helper_matches_the_one_point_formula():
    """eval_model and eval_model_hess_batch share _d2sigdx2; for one point it is the reference's formula
    (eval/GpEvalModel.py:366-375) bit for bit, and a point with sig = 0 gets a NaN slab."""
    from gpgradpy_b200.gp import _d2sigdx2
    rng = np.random.default_rng(3)
    d, varK = 4, 2.5
    h3 = rng.normal(size=(3, 3, d, d))
    h3 = h3 + h3.transpose(0, 1, 3, 2)
    sig = np.array([0.7, 0.0, 1.3])
    dsig = rng.normal(size=(3, d))
    got = _d2sigdx2(h3, sig, dsig, varK)
    for i in range(3):
        d2sig2 = -2.0 * varK * (h3[i, 1] + h3[i, 2])
        s = np.nan if sig[i] == 0 else sig[i]
        ref = (d2sig2 - 2.0 * np.outer(dsig[i], dsig[i])) / (2.0 * s)
        if sig[i] == 0:
            assert np.all(np.isnan(got[i]))
        else:
            assert np.array_equal(got[i], ref)
            assert np.array_equal(got[i], got[i].T)
