"""GPU: batched surrogate Hessians (gegp_predict_hess_batch, backend.predict_hess_batch,
GaussianProcess.eval_model_hess_batch) against the CPU oracle (tests/hess_batch_oracle.py, built on oracle/gegp_oracle.py), against the
one-point path (gegp_predict_hess / eval_model(calc_hess=True)) and against gegp_predict_grad.

Tolerances are the project's: mu, dmu/dx, d2mu/dx2 1e-8 relative to their largest entry; sigma-derived outputs (sig,
dsig/dx, d2sig/dx2) 1e-6 of their largest entry, compared away from the data (they divide by sigma); 1e-6 for the
ill-conditioned configuration-1 case; 1e-12 between the batched and the one-point path and between chunkings."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))   # tests/hess_batch_oracle.py, whatever the import mode

pytestmark = pytest.mark.gpu

KERNELS = {"SqExp": "SqExp", "Ma5f2": "Ma5f2", "RatQu": ("RatQu", 0.7)}
VARK = 2.5


def _theta(n, d, c=2.0):
    s = 4.0 / n ** (1.0 / d)
    return c * np.linspace(0.6, 1.4, d) / s ** 2


def _mask(n, seed, p=0.2):
    m = np.random.default_rng(seed).uniform(size=n) > p
    m[0], m[1] = False, True
    return m


def _problem(n, d, kname="SqExp", *, masked=False, noisy=False, mode="precon", seed=0, c=2.0, no_grad=False, eta=None):
    from gpgradpy_b200 import backend as bk, _lib as L
    from oracle import gegp_oracle as O
    x, f, g = O.synthetic_problem(n, d, seed)
    kern = KERNELS[kname]
    mask = np.zeros(n, bool) if no_grad else (_mask(n, seed + 100) if masked else None)
    gin = g if mask is None else g[mask]
    slot, ng = bk.slot_from_mask(mask, n)
    N = n + ng * d
    noise = None
    if noisy:
        rng = np.random.default_rng(seed + 7)
        noise = np.concatenate([rng.uniform(1e-4, 1e-2, n), rng.uniform(1e-3, 3e-2, N - n)]) / VARK
    th = _theta(n, d, c)
    if eta is None:
        eta = O.nugget(n, d, mode, kernel=kern)[1]
    beta = float(np.mean(f))
    y = O.make_data_vec(f, gin) if ng else f.copy()
    st = bk.predict_setup(x, y, th, beta, n_g=ng, slot=slot, noise=noise,
                          mode=L.MODE_PRECON if mode == "precon" else L.MODE_BASE, eta=eta, kernel=kern)
    assert int(st.info.item()) == 0
    oargs = (x, f, gin if ng else np.zeros((0, d)), th, VARK, np.array([beta]))
    okw = dict(mode=mode, eta=eta, kernel=kern, noise_vec=noise, mask=mask)
    return dict(st=st, x=x, n=n, d=d, N=N, oargs=oargs, okw=okw)


def _points(p, nx, seed, lo=-2.0, hi=2.0):
    return np.random.default_rng(seed).uniform(lo, hi, (nx, p["d"]))


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


def _batch(p, xs, **kw):
    from gpgradpy_b200 import backend as bk
    return _np(*bk.predict_hess_batch(p["st"], xs, VARK, **kw))


def _derived(out):
    """(mu, sig, dmu, dsig, d2mu, d2sig) from the raw outputs, with the formula GaussianProcess uses."""
    from gpgradpy_b200.gp import _d2sigdx2
    mu, sig, sig2, dmu, dsig, h3, nneg = out
    return mu, sig, dmu, dsig, h3[:, 0], _d2sigdx2(h3, sig, dsig, VARK)


def _err(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(b)))


def _check_oracle(p, xs, got, tol_sig=1e-6):
    from hess_batch_oracle import eval_model_hess_batch
    ref = eval_model_hess_batch(*p["oargs"], xs, **p["okw"])
    far = ref[1] > 1e-3 * np.sqrt(VARK)                  # away from the data: the sigma-derived outputs are defined
    assert far.sum() > 0
    e = {k: _err(g, r) for k, g, r in zip(("mu", "dmu", "d2mu"), (got[0], got[2], got[4]), (ref[0], ref[2], ref[4]))}
    for k, i in (("sig", 1), ("dsig", 3), ("d2sig", 5)):
        e[k] = _err(got[i][far], ref[i][far])
    print({k: f"{v:.1e}" for k, v in e.items()})
    assert e["mu"] < 1e-8 and e["dmu"] < 1e-8 and e["d2mu"] < 1e-8
    assert e["sig"] < tol_sig and e["dsig"] < tol_sig and e["d2sig"] < tol_sig
    return ref


def _close(got, ref, tol=1e-12):
    """Raw outputs (mu, sig, sig2, dmu, dsig, hess3) equal to rounding: each to tol of its largest entry; dsig (which
    divides by sigma) where sigma is above a tenth of its largest value."""
    far = ref[1] > 0.1 * np.max(ref[1])
    for k in range(6):
        a, b = (got[k][far], ref[k][far]) if k == 4 else (got[k], ref[k])
        assert a.shape == b.shape and np.max(np.abs(a - b)) <= tol * np.max(np.abs(b)), k


SMALL, LARGE = (20, 2), (250, 3)     # N = 60 (one leaf) and N = 1000 (recursive solves with GEMM updates)
CASES = [  # kernel, masked, noisy, mode, size
    ("SqExp", False, False, "precon", SMALL), ("SqExp", True, True, "base", LARGE), ("SqExp", True, True, "precon", SMALL),
    ("Ma5f2", True, False, "base", SMALL), ("Ma5f2", False, True, "precon", LARGE), ("Ma5f2", True, False, "precon", LARGE),
    ("RatQu", False, True, "base", SMALL), ("RatQu", True, False, "precon", LARGE), ("RatQu", True, True, "base", LARGE)]


def _case_id(c):
    return f"{c[0]}-{'mask' if c[1] else 'full'}-{'noisy' if c[2] else 'exact'}-{c[3]}-N{c[4][0] * (c[4][1] + 1)}"


# ---------------------------------------------------------------------------------------------------------------------
# 1. parity with the oracle at every point
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_vs_oracle(case):
    kname, masked, noisy, mode, (n, d) = case
    p = _problem(n, d, kname, masked=masked, noisy=noisy, mode=mode, seed=1)
    xs = _points(p, 23, 2)
    _check_oracle(p, xs, _derived(_batch(p, xs)))


def test_vs_oracle_gradient_free_gp():
    """n_g = 0: only value rows; every G_p is zero (slot -1 everywhere)."""
    p = _problem(40, 3, "Ma5f2", no_grad=True, mode="base", seed=3)
    assert p["N"] == 40
    xs = _points(p, 17, 4)
    _check_oracle(p, xs, _derived(_batch(p, xs)))


def test_vs_oracle_c2_size():
    """Configuration-2 size: n = 500, d = 10 (N = 5500), 64 points in one chunk."""
    p = _problem(500, 10, "SqExp", seed=5)
    xs = _points(p, 64, 6, -1.5, 1.5)
    _check_oracle(p, xs, _derived(_batch(p, xs)))


def test_vs_oracle_d_above_the_thread_count():
    """d = 24: 300 upper-triangle pairs, more than the 256 threads of a CTA (two pairs for some threads)."""
    p = _problem(30, 24, "RatQu", masked=True, seed=7)
    xs = _points(p, 5, 8, -1.0, 1.0)
    _check_oracle(p, xs, _derived(_batch(p, xs)))


def test_config1_conditioning():
    """Configuration 1 (d = 2, n = 20, base mode) with long length scales: cond(K) ~ 5e9.  The back substitution of
    K^-1 k* multiplies with explicit inverses of the factor's diagonal blocks; with its refinement step term1 =
    (d2 k*/dx2) . K^-1 k* and term2 match the oracle to 1e-6, d2mu to 1e-8.  (sigma itself is ~1e-2 sqrt(varK) here, the
    size of the rounding of 1 - k*^T K^-1 k* at this conditioning, so the sigma-derived outputs are not compared.)"""
    from scipy import linalg
    from oracle import gegp_oracle as O
    p = _problem(20, 2, "SqExp", mode="base", seed=9, c=0.2)
    x, f, g, th, _, beta = p["oargs"]
    eta = p["okw"]["eta"]
    K = O.kern_grad(x, x, th) + eta * np.eye(p["N"])
    assert np.linalg.cond(K) > 1e9
    xs = _points(p, 31, 10)
    out = _batch(p, xs)
    cf = linalg.cho_factor(K, lower=True)
    a = linalg.cho_solve(cf, O.make_data_vec(f, g) - O.aug_vand(20, 20, 2) @ beta)
    ref = np.zeros((31, 3, 2, 2))
    for i in range(31):
        Kg = O.kern_grad(x, xs[i:i + 1], th)
        k, dK = Kg[:, 0], Kg[:, 1:].T
        d2K = O.kern_hess_x(x, xs[i], th)
        ref[i] = d2K @ a, d2K @ linalg.cho_solve(cf, k), dK @ linalg.cho_solve(cf, dK.T)
    e = [_err(out[5][:, m], ref[:, m]) for m in range(3)]
    print("config1 d2mu, term1, term2:", [f"{v:.1e}" for v in e])
    assert e[0] < 1e-8 and e[1] < 1e-6 and e[2] < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# 2. agreement with the one-point path and with gegp_predict_grad
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [SMALL, LARGE], ids=["N60", "N1000"])
def test_agrees_with_the_one_point_path(size):
    from gpgradpy_b200 import backend as bk
    p = _problem(*size, "Ma5f2", masked=True, noisy=True, seed=11)
    xs = _points(p, 9, 12)
    out = _batch(p, xs)
    ones = [_np(*bk.predict_hess(p["st"], xs[i], VARK)) for i in range(xs.shape[0])]
    one = [np.stack([o[k].reshape(np.shape(out[k][0])) for o in ones]) for k in range(6)]
    _close(out, one)
    # mu, sig, sig2, dmu, dsig: gegp_predict_grad's for the same chunk, bit for bit
    grad = _np(*bk.predict_grad(p["st"], xs, VARK))
    for k in range(5):
        assert np.array_equal(out[k], grad[k]), k
    assert int(out[6][0]) == int(grad[5][0])


WIDE = [  # kernel, masked, noisy, mode, n, d: 2, 3 and 7 pages of upper-triangle pairs; tiles of 32 training points at d = 160
    ("SqExp", True, True, "precon", 6, 64), ("RatQu", False, True, "base", 5, 100), ("Ma5f2", True, False, "precon", 4, 160)]


@pytest.mark.parametrize("case", WIDE, ids=lambda c: f"{c[0]}-d{c[5]}")
def test_wide_vs_oracle_and_one_point(case):
    """d > 63: the batched and the one-point call against the oracle, and against each other to 1e-12.  Each test point
    lies at s = 0.5 from one training point: in this many dimensions the rest of the data is out of reach."""
    from gpgradpy_b200 import backend as bk
    kname, masked, noisy, mode, n, d = case
    p = _problem(n, d, kname, masked=masked, noisy=noisy, mode=mode, seed=27)
    z = np.random.default_rng(28).normal(size=(n, d))
    xs = p["x"] + z * np.sqrt(0.5 / np.sum(_theta(n, d) * z * z, axis=1))[:, None]
    out = _batch(p, xs)
    ones = [_np(*bk.predict_hess(p["st"], xs[i], VARK)) for i in range(n)]
    one = [np.stack([o[k].reshape(np.shape(out[k][0])) for o in ones]) for k in range(6)]
    _close(out, one)
    _check_oracle(p, xs, _derived(out))
    _check_oracle(p, xs, _derived(one + [None]))


def test_gaussian_process_batch_is_the_stacked_one_point_calls():
    """GaussianProcess.eval_model_hess_batch(X)[k][i] == eval_model(X[i:i+1], calc_grad=True, calc_hess=True)[k][0] to
    1e-12, in a rescale mode (rescale_origin: inputs, outputs and derivatives go through data_scl_2_init)."""
    from gpgradpy_b200.gp import GaussianProcess
    from oracle import gegp_oracle as O
    n, d = 24, 3
    x, f, g = O.synthetic_problem(n, d, 13)
    GP = GaussianProcess(d, True, "SqExp", "rescale_origin")
    GP.set_data(x, f, np.zeros(n), g, np.zeros(g.shape))
    assert GP.b_use_data_scl
    GP.set_hpara("set", 1, GP.make_hp_class(theta=np.linspace(0.5, 1.5, d), varK=VARK, beta=np.array([0.3])))
    xs = np.random.default_rng(14).uniform(-2, 2, (8, d))
    got = GP.eval_model_hess_batch(xs)
    assert got[4].shape == (8, d, d) and got[5].shape == (8, d, d)
    ones = [GP.eval_model(xs[i:i + 1], calc_grad=True, calc_hess=True) for i in range(8)]
    far = got[1] > 0.1 * np.max(got[1])
    for k in range(6):
        ref = np.stack([np.asarray(o[k])[0] for o in ones])
        a, b = (got[k][far], ref[far]) if k in (3, 5) else (got[k], ref)
        assert np.max(np.abs(a - b)) <= 1e-12 * np.max(np.abs(b)), k
    with pytest.raises(Exception):
        GP.hp_vals = GP.make_hp_class(theta=np.ones(d), varK=VARK, beta=np.array([0.3]))
        GP.eval_model_hess_batch(xs)


# ---------------------------------------------------------------------------------------------------------------------
# 3. chunking and symmetry
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [SMALL, LARGE], ids=["N60", "N1000"])
def test_chunk_invariance(size):
    from gpgradpy_b200 import backend as bk
    p = _problem(*size, "RatQu", masked=True, seed=15)
    nx = 29
    xs = _points(p, nx, 16)
    fixed = bk.predict_hess_batch_bytes(p["N"], p["d"], 0)
    per = bk.predict_hess_batch_bytes(p["N"], p["d"], 1) - fixed
    full = _batch(p, xs, chunk_bytes=fixed + nx * per)
    for pts in (1, 7, nx - 1):
        got = _batch(p, xs, chunk_bytes=fixed + pts * per)
        assert int(got[6][0]) == int(full[6][0])
        _close(got, full)
    _check_oracle(p, xs, _derived(_batch(p, xs, chunk_bytes=fixed + 7 * per)))


def test_exact_symmetry():
    from gpgradpy_b200.gp import _d2sigdx2
    for kname, size in (("SqExp", LARGE), ("Ma5f2", (30, 24))):
        p = _problem(*size, kname, masked=True, noisy=True, seed=17)
        out = _batch(p, _points(p, 11, 18, -1.0, 1.0))
        h3 = out[5]
        assert np.array_equal(h3, h3.transpose(0, 1, 3, 2))
        d2sig = _d2sigdx2(h3, out[1], out[4], VARK)
        assert np.array_equal(d2sig, d2sig.transpose(0, 2, 1))


# ---------------------------------------------------------------------------------------------------------------------
# 4. finite differences
# ---------------------------------------------------------------------------------------------------------------------
def test_d2mu_is_the_derivative_of_dmu():
    """N = 1000 with a mask and noise: central differences of gegp_predict_grad's dmu/dx."""
    from gpgradpy_b200 import backend as bk
    p = _problem(250, 3, "SqExp", masked=True, noisy=True, seed=19)
    xs = _points(p, 6, 20, -1.5, 1.5)
    h = 1e-5
    d2mu = _batch(p, xs)[5][:, 0]
    for j in range(3):
        e = np.zeros(3)
        e[j] = h
        dp = _np(*bk.predict_grad(p["st"], xs + e, VARK))[3]
        dm = _np(*bk.predict_grad(p["st"], xs - e, VARK))[3]
        fd = (dp - dm) / (2 * h)                                       # column j of the Hessian
        assert np.max(np.abs(fd - d2mu[:, :, j])) <= 1e-6 * np.max(np.abs(d2mu)), j


# ---------------------------------------------------------------------------------------------------------------------
# 5. edge cases
# ---------------------------------------------------------------------------------------------------------------------
def test_points_on_the_data():
    """Training points as test points, noise-free base mode without nugget: sigma^2 = 1 - k*^T K^-1 k* is zero up to
    rounding, so sig = 0 where it rounds to <= 0.  There d2sig is NaN (the one-point path's convention), d2mu stays finite,
    and n_negative counts exactly the negative sig2 entries."""
    from gpgradpy_b200 import backend as bk
    p = _problem(12, 2, "SqExp", mode="base", seed=21, c=1.0, eta=0.0)
    xs = np.vstack([p["x"], _points(p, 4, 22)])
    out = _batch(p, xs)
    mu, sig, sig2, dmu, dsig, h3, nneg = out
    d2sig = _derived(out)[5]
    assert int(nneg[0]) == int(np.sum(sig2 < 0))
    zero = sig == 0
    assert zero.sum() > 0
    assert np.all(np.isnan(d2sig[zero])) and np.all(np.isfinite(d2sig[~zero]))
    assert np.all(np.isfinite(h3[:, 0]))
    for i in np.flatnonzero(zero)[:3]:
        one = _np(*bk.predict_hess(p["st"], xs[i], VARK))
        assert one[1][0] == 0
        assert np.max(np.abs(h3[i, 0] - one[5][0])) <= 1e-12 * np.max(np.abs(one[5][0]))


def test_negative_variance_assertion(monkeypatch):
    """GaussianProcess.eval_model_hess_batch asserts on negative variances like eval_model."""
    import torch
    from gpgradpy_b200 import backend as bk
    from gpgradpy_b200.gp import GaussianProcess
    from oracle import gegp_oracle as O
    n, d = 12, 2
    x, f, g = O.synthetic_problem(n, d, 23)
    GP = GaussianProcess(d, True, "SqExp", "precon")
    GP.set_data(x, f, np.zeros(n), g, np.zeros(g.shape))
    GP.set_hpara("set", 1, GP.make_hp_class(theta=np.ones(d), varK=VARK, beta=np.array([0.0])))
    real = bk.predict_hess_batch

    def one_negative(*a, **k):
        out = list(real(*a, **k))
        out[6] = torch.ones_like(out[6])
        return tuple(out)

    GP.eval_model_hess_batch(x[:3])
    monkeypatch.setattr(bk, "predict_hess_batch", one_negative)
    with pytest.raises(AssertionError):
        GP.eval_model_hess_batch(x[:3])


def test_nx_zero_writes_nothing():
    import torch
    from gpgradpy_b200 import backend as bk, _lib as L
    p = _problem(20, 2, seed=25)
    st, d = p["st"], 2
    G, fill = 16, 12345.5
    bufs = {k: torch.full((G + m + G,), fill, dtype=torch.float64, device="cuda")
            for k, m in (("mu", 4), ("sig", 4), ("sig2", 4), ("dmu", 4 * d), ("dsig", 4 * d), ("h3", 4 * 3 * d * d))}
    nneg = torch.full((3,), 7, dtype=torch.int32, device="cuda")
    ws = torch.full((1 << 20,), fill, dtype=torch.float64, device="cuda")
    Xs = torch.zeros((1, d), dtype=torch.float64, device="cuda")
    c = lambda k: bufs[k][G:].data_ptr()
    rc = L.load().gegp_predict_hess_batch(st.n, st.n_g, st.d, bk._p(st.X), bk._p(st.slot), bk._p(st.theta), st.kid, st.khp,
                                          bk._p(st.A), st.A.stride(0), bk._p(st.dinv), bk._p(st.p), bk._p(st.alpha),
                                          int(st.mode), st.beta, VARK, Xs.data_ptr(), 0, c("mu"), c("sig"), c("sig2"),
                                          c("dmu"), c("dsig"), c("h3"), nneg[1:].data_ptr(), ws.data_ptr(), 8 * ws.numel(),
                                          bk._stream())
    torch.cuda.synchronize()
    assert rc == 0
    for k, b in bufs.items():
        assert bool((b == fill).all()), k
    assert bool((nneg == 7).all()) and bool((ws == fill).all())
    out = bk.predict_hess_batch(st, np.zeros((0, d)), VARK)
    assert [tuple(t.shape) for t in out[:6]] == [(0,), (0,), (0,), (0, d), (0, d), (0, 3, d, d)]


def test_n_negative_counts_across_chunks():
    """The counter accumulates over chunks: the same count for one chunk and for chunks of one point."""
    from gpgradpy_b200 import backend as bk
    p = _problem(12, 2, "SqExp", mode="base", seed=21, c=1.0, eta=0.0)
    xs = np.vstack([p["x"], p["x"]])
    fixed = bk.predict_hess_batch_bytes(p["N"], 2, 0)
    per = bk.predict_hess_batch_bytes(p["N"], 2, 1) - fixed
    a = _batch(p, xs)
    b = _batch(p, xs, chunk_bytes=fixed + per)
    assert int(a[6][0]) == int(np.sum(a[2] < 0)) == int(b[6][0])
