"""CPU checks of the oracle's posterior Hessians (oracle/gegp_oracle.py: eval_model_hess) with masked gradients and
observation noise.  tests/test_gpu_posterior.py holds the CUDA Hessian kernel to this reference, so the reference is
checked on its own here: an all-True mask changes nothing, and d2mu / d2sig are the x-derivatives of eval_model_grad's
dmu / dsig (central differences)."""
import numpy as np
import pytest

from oracle import gegp_oracle as O

KERNELS = {"SqExp": None, "Ma5f2": "Ma5f2", "RatQu": ("RatQu", 0.7)}


def _problem(n, d, seed, kernel, *, mask=None, noisy=False, mode="precon"):
    x, f, g = O.synthetic_problem(n, d, seed)
    th = np.linspace(0.4, 0.9, d)
    eta = O.nugget(n, d, mode, kernel=kernel)[1]
    gin = g if mask is None else g[mask]
    ng = n if mask is None else int(np.sum(mask))
    N = n + ng * d
    noise = None
    if noisy:       # heteroscedastic: values and gradients with different, varying variances (already divided by varK)
        noise = np.concatenate([np.linspace(1e-4, 1e-2, n), np.linspace(1e-3, 3e-2, N - n)])
    return dict(X=x, fval=f, grad=gin, theta=th, varK=2.5, beta=np.array([float(np.mean(f))]), mode=mode, eta=eta,
                kernel=kernel, noise_vec=noise, mask=mask)


def _hess(p, xs):
    return O.eval_model_hess(p["X"], p["fval"], p["grad"], p["theta"], p["varK"], p["beta"], xs, p["mode"], p["eta"],
                             kernel=p["kernel"], noise_vec=p["noise_vec"], mask=p["mask"])


def _grad(p, xs):
    return O.eval_model_grad(p["X"], p["fval"], p["grad"], p["theta"], p["varK"], p["beta"], np.atleast_2d(xs), p["mode"],
                             p["eta"], p["noise_vec"], p["mask"], kernel=p["kernel"])


@pytest.mark.parametrize("kname", list(KERNELS))
@pytest.mark.parametrize("noisy", [False, True])
def test_all_true_mask_is_the_unmasked_hessian(kname, noisy):
    p = _problem(14, 3, 2, KERNELS[kname], noisy=noisy)
    xs = np.array([0.3, -0.7, 1.1])
    ref = _hess(p, xs)
    got = _hess(dict(p, mask=np.ones(14, dtype=bool)), xs)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)


def _masked(n):
    m = np.zeros(n, dtype=bool)
    m[[0, 2, 3, 7, 8, 11, 13]] = True     # scattered: neither a prefix nor a suffix
    return m


CASES = [("SqExp", False, False, "precon"), ("SqExp", True, False, "base"), ("SqExp", True, True, "precon"),
         ("Ma5f2", False, True, "base"), ("Ma5f2", True, False, "precon"), ("Ma5f2", True, True, "base"),
         ("RatQu", False, False, "base"), ("RatQu", True, True, "precon"), ("RatQu", False, True, "precon")]


@pytest.mark.parametrize("kname,masked,noisy,mode", CASES)
def test_hessian_is_the_derivative_of_the_gradient(kname, masked, noisy, mode):
    """Central differences of (dmu, dsig) in x, step h = 1e-4 (truncation ~ h^2 |f'''|, rounding ~ eps cond(K) / h)."""
    n, d = 14, 3
    p = _problem(n, d, 4, KERNELS[kname], mask=_masked(n) if masked else None, noisy=noisy, mode=mode)
    xs = np.array([0.35, -0.6, 0.9])          # between the training points: sigma well away from 0
    mu, sig, dmu, dsig, d2mu, d2sig = _hess(p, xs)
    assert sig[0] > 1e-3 * np.sqrt(p["varK"])
    h = 1e-4
    fd_mu, fd_sig = np.zeros((d, d)), np.zeros((d, d))
    for k in range(d):
        e = np.zeros(d)
        e[k] = h
        _, _, dmu_p, dsig_p = _grad(p, xs + e)
        _, _, dmu_m, dsig_m = _grad(p, xs - e)
        fd_mu[k] = (dmu_p[0] - dmu_m[0]) / (2 * h)
        fd_sig[k] = (dsig_p[0] - dsig_m[0]) / (2 * h)
    e_mu = np.max(np.abs(d2mu[0] - fd_mu)) / np.max(np.abs(fd_mu))
    e_sig = np.max(np.abs(d2sig[0] - fd_sig)) / np.max(np.abs(fd_sig))
    print(f"{kname} masked={masked} noisy={noisy} {mode}: d2mu {e_mu:.2e} d2sig {e_sig:.2e}")
    assert e_mu < 1e-6 and e_sig < 1e-6
    assert np.allclose(d2mu[0], d2mu[0].T, rtol=0, atol=1e-12 * np.max(np.abs(d2mu)))
    # the first-order outputs are eval_model_grad's at the same point
    ref = _grad(p, xs)
    assert np.array_equal(mu, ref[0]) and np.array_equal(sig, ref[1])
    assert np.array_equal(dmu, ref[2]) and np.array_equal(dsig, ref[3])


def test_masked_hessian_differs_from_the_unmasked_one():
    """A mask changes the data the posterior conditions on: the masked Hessian must not coincide with the full one
    (guards against a mask that is silently ignored)."""
    n, d = 14, 3
    xs = np.array([0.35, -0.6, 0.9])
    full = _problem(n, d, 4, None)
    m = _masked(n)
    part = dict(full, mask=m, grad=full["grad"][m])
    a, b = _hess(full, xs), _hess(part, xs)
    assert np.max(np.abs(a[4] - b[4])) > 1e-3 * np.max(np.abs(a[4]))
