"""The dense reference of tests/lml_dense_ref.py against the oracle's own matrices (no GPU needed): cov() against the
covariance of all_K_w_chofac in each build mode, dcov_hp() / contract() against the dense stacks kerngrad_hp,
kcov_grad_hp_noisy and kern_grad_dalpha, for all three kernel families, prefix and scatter masks, noise, base and
precon.  And the tolerance rule the GPU tests use, |g - g_ref| <= 1e-12 sum(|W .* dKcov/dhp|), is shown to be sharp
enough: a reference that drops one point pair, or perturbs one entry of one pair's block by 1e-9 relative, fails it."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))   # tests/lml_dense_ref.py, whatever the import mode
import lml_dense_ref as R  # noqa: E402
from gpgradpy_b200._lib import MODE_BASE, MODE_PRECON, MODE_PRECON_COV  # noqa: E402
from oracle import gegp_oracle as O  # noqa: E402

KERNELS = [None, "Ma5f2", ("RatQu", 0.7)]
MASKS = {"all": None, "prefix": np.arange(9) < 5, "scatter": np.array([1, 0, 1, 1, 0, 0, 1, 0, 1], dtype=bool)}


def _problem(n=9, d=3, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1.0, 1.0, (n, d))
    theta = rng.uniform(0.5, 2.5, d)
    return X, theta


def _noise(n, g, d, seed=1):
    rng = np.random.default_rng(seed)
    return np.hstack((rng.uniform(1e-4, 1e-2, n), rng.uniform(1e-3, 5e-2, g * d)))


@pytest.mark.parametrize("kernel", KERNELS, ids=["SqExp", "Ma5f2", "RatQu"])
@pytest.mark.parametrize("mask", list(MASKS), ids=list(MASKS))
@pytest.mark.parametrize("noisy", [False, True], ids=["free", "noise"])
def test_cov_matches_the_oracle_matrices(kernel, mask, noisy):
    X, th = _problem()
    n, d = X.shape
    m = MASKS[mask]
    g = O._sel(n, m).size
    N = n + g * d
    eta, varK = 3e-7, (1.7 if noisy else 1.0)
    noise = _noise(n, g, d) if noisy else None
    K = O.kern_grad(X, X, th, m, m, kernel=kernel)
    Kw = K + (np.diag(noise) if noisy else 0.0)
    base, _ = R.cov(X, th, MODE_BASE, eta, m, kernel, noise, varK)
    assert np.max(np.abs(base - varK * (Kw + eta * np.eye(N)))) <= 1e-15 * np.max(np.abs(base))
    Kt, p = R.cov(X, th, MODE_PRECON, eta, m, kernel, noise, varK)
    assert np.max(np.abs(p - np.sqrt(np.diag(Kw)))) <= 1e-15 * np.max(p)
    Kcor = Kw / p[:, None] / p[None, :]
    assert np.max(np.abs(Kt - varK * (Kcor + eta * np.eye(N)))) <= 1e-14 * np.max(np.abs(Kt))
    assert np.allclose(np.diag(Kt), varK * (1.0 + eta), rtol=1e-15, atol=0)
    pc, _ = R.cov(X, th, MODE_PRECON_COV, eta, m, kernel, noise, varK)
    assert np.max(np.abs(pc - varK * (Kw + eta * np.diag(np.diag(Kw))))) <= 1e-15 * np.max(np.abs(pc))
    assert np.max(np.abs(pc - p[:, None] * Kt * p[None, :])) <= 1e-14 * np.max(np.abs(pc))
    for M in (base, Kt, pc):
        assert np.max(np.abs(M - M.T)) <= 1e-15 * np.max(np.abs(M))


def _oracle_stack(X, th, mode, eta, m, kernel, noisy, varK):
    ms = "precon" if mode == MODE_PRECON else "base"
    if noisy:
        Kern = O.kern_grad(X, X, th, m, m, kernel=kernel)
        return O.kcov_grad_hp_noisy(X, th, Kern, ms, eta, varK, True, True, m, kernel=kernel)
    return O.kerngrad_hp(X, th, ms, eta, m, kernel=kernel)


@pytest.mark.parametrize("kernel", KERNELS, ids=["SqExp", "Ma5f2", "RatQu"])
@pytest.mark.parametrize("mask", list(MASKS), ids=list(MASKS))
@pytest.mark.parametrize("mode", [MODE_BASE, MODE_PRECON], ids=["base", "precon"])
@pytest.mark.parametrize("noisy", [False, True], ids=["free", "noise"])
def test_contract_matches_the_oracle_stacks(kernel, mask, mode, noisy):
    X, th = _problem(seed=2)
    n, d = X.shape
    m = MASKS[mask]
    eta, varK = 2e-6, (0.6 if noisy else 1.0)
    stack = _oracle_stack(X, th, mode, eta, m, kernel, noisy, varK)
    slots = R.hp_slots(d, kernel, noisy)
    assert stack.shape[0] == len(slots)
    mine = list(R.dcov_hp(X, th, mode, eta, m, kernel, noisy, varK))
    assert [k for k, _ in mine] == slots
    for (k, D), S in zip(mine, stack):
        assert np.max(np.abs(D - S)) <= 1e-14 * max(np.max(np.abs(S)), 1e-300), k
    if kernel is not None and O._kernel_spec(kernel)[0] == "RatQu":
        Da = O.kern_grad_dalpha(X, th, kernel, m) * (varK if noisy else 1.0)
        assert np.max(np.abs(dict(mine)[R.OUT_DKERN] - Da)) <= 1e-14 * np.max(np.abs(Da))
    N = stack.shape[1]
    rng = np.random.default_rng(3)
    W = rng.standard_normal((N, N))
    W = W + W.T
    v = rng.standard_normal(N)
    for w, ref in ((W, np.einsum("ijk,jk->i", stack, W)), (v, np.einsum("ijk,j,k->i", stack, v, v))):
        g, sc = R.contract(X, th, w, mode, eta, m, kernel, noisy, varK)
        assert R.contract_err(g, np.zeros_like(g), sc, slots) > 0.0
        gr = np.zeros_like(g)
        gr[slots] = ref
        assert R.contract_err(g, gr, sc, slots) <= 1e-13


def _pair_index(n, g, d, slot, a):
    """Rows (or columns) of point a in the dimension-major order: its value and its gradient entries."""
    idx = [a]
    if slot[a] >= 0:
        idx += [n + i * g + slot[a] for i in range(d)]
    return np.array(idx)


@pytest.mark.parametrize("kernel", KERNELS, ids=["SqExp", "Ma5f2", "RatQu"])
@pytest.mark.parametrize("mask", ["all", "scatter"])
def test_tolerance_rule_catches_one_dropped_pair_and_one_perturbed_entry(kernel, mask):
    """For every hyper-parameter: the contraction with the pair (a, b) that contributes most left out, and the contraction
    with the largest entry of W .* dKcov/dhp scaled by 1 + 1e-9, both miss the reference by more than 1e-12 of the scale."""
    X, th = _problem(seed=4)
    n, d = X.shape
    m = MASKS[mask]
    sel = O._sel(n, m)
    g = sel.size
    slot = -np.ones(n, dtype=int)
    slot[sel] = np.arange(g)
    eta = 1e-6
    N = n + g * d
    rng = np.random.default_rng(5)
    W = rng.standard_normal((N, N))
    W = W + W.T
    blocks = [_pair_index(n, g, d, slot, a) for a in range(n)]
    for k, D in R.dcov_hp(X, th, MODE_PRECON, eta, m, kernel, True, 1.3):
        gk, sk = R.weigh(D, W)
        P = W * D
        contrib = np.array([[np.sum(P[np.ix_(blocks[a], blocks[b])]) for b in range(n)] for a in range(n)])
        a, b = np.unravel_index(np.argmax(np.abs(contrib)), contrib.shape)
        Dd = D.copy()
        Dd[np.ix_(blocks[a], blocks[b])] = 0.0
        assert abs(R.weigh(Dd, W)[0] - gk) > 1e-12 * sk, (k, "dropped pair", a, b)
        e = np.unravel_index(np.argmax(np.abs(P)), P.shape)
        Dp = D.copy()
        Dp[e] *= 1.0 + 1e-9
        assert abs(R.weigh(Dp, W)[0] - gk) > 1e-12 * sk, (k, "perturbed entry", e)
