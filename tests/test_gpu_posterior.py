"""GPU: the posterior path (gegp_cross_cov, gegp_predict, gegp_predict_grad, gegp_predict_hess) against the CPU oracle
(oracle/gegp_oracle.py), across the three kernel families, masked gradients, heteroscedastic noise, both conditioning
modes, leaf-only (N <= 128) and recursive (GEMM) solves, chunked evaluation and test sets longer than one launch's
65,535 grid rows.

Tolerances (as in tests/test_gpu_gp.py and tests/test_gpu_kernels.py): cross covariance 1e-12 of the block scale;
mu, dmu/dx, d2mu/dx2 1e-8 relative to their largest entry; |d sig^2| <= 1e-8 varK; dsig/dx 1e-6 relative where
sig > 1e-3 max sig; d2sig/dx2 1e-5 relative."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KERNELS = {"SqExp": "SqExp", "Ma5f2": "Ma5f2", "RatQu": ("RatQu", 0.7)}
VARK = 2.5


def _theta(n, d, c=2.0):
    """Length scales matched to the point spacing of n uniform points in [-2, 2]^d: cond(K) stays below ~1e8."""
    s = 4.0 / n ** (1.0 / d)
    return c * np.linspace(0.6, 1.4, d) / s ** 2


def _mask(n, seed):
    """Scattered gradient mask: about one point in five without a gradient, never a prefix."""
    m = np.random.default_rng(seed).uniform(size=n) > 0.2
    m[0], m[1] = False, True
    return m


def _problem(n, d, kname="SqExp", *, masked=False, noisy=False, mode="precon", seed=0, c=2.0):
    """Seeded data, the device factor (predict_setup) and the matching oracle arguments."""
    from gpgradpy_b200 import backend as bk, _lib as L
    from oracle import gegp_oracle as O
    x, f, g = O.synthetic_problem(n, d, seed)
    kern = KERNELS[kname]
    mask = _mask(n, seed + 100) if masked else None
    gin = g if mask is None else g[mask]
    slot, ng = bk.slot_from_mask(mask, n)
    N = n + ng * d
    noise = None
    if noisy:   # heteroscedastic, divided by varK (include/gegp.h: the factor is built with varK := 1)
        rng = np.random.default_rng(seed + 7)
        noise = np.concatenate([rng.uniform(1e-4, 1e-2, n), rng.uniform(1e-3, 3e-2, N - n)]) / VARK
    th = _theta(n, d, c)
    eta = O.nugget(n, d, mode, kernel=kern)[1]
    beta = float(np.mean(f))
    y = O.make_data_vec(f, gin)
    st = bk.predict_setup(x, y, th, beta, n_g=ng, slot=slot, noise=noise,
                          mode=L.MODE_PRECON if mode == "precon" else L.MODE_BASE, eta=eta, kernel=kern)
    assert int(st.info.item()) == 0
    oargs = (x, f, gin, th, VARK, np.array([beta]))
    okw = dict(mode=mode, eta=eta, noise_vec=noise, mask=mask, kernel=kern)
    return dict(st=st, x=x, n=n, d=d, N=N, oargs=oargs, okw=okw, kern=kern, mask=mask, slot=slot, ng=ng, th=th)


def _test_points(p, nx, seed, n_on_data=0):
    """nx - n_on_data uniform points over (and a little beyond) the data, then n_on_data training points exactly."""
    xs = np.random.default_rng(seed).uniform(-2.2, 2.2, (nx - n_on_data, p["d"]))
    return np.vstack([xs, p["x"][:n_on_data]])


def _ref(p, xs, grad):
    from oracle import gegp_oracle as O
    fn = O.eval_model_grad if grad else O.eval_model
    return fn(*p["oargs"], xs, p["okw"]["mode"], p["okw"]["eta"], p["okw"]["noise_vec"], p["okw"]["mask"],
              kernel=p["kern"])


def _ref_sig2(p, xs):
    return _ref(p, xs, False)[2]


def _err(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(b)))


def _check_values(mu, sig, sig2, nneg, ref):
    mu_r, sig_r, sig2_r = ref[:3]           # the oracle's (mu, sig, sig2[, n_negative])
    assert _err(mu, mu_r) < 1e-8
    assert np.max(np.abs(sig2 - sig2_r)) < 1e-8          # sig2 is normalised by varK
    assert np.max(np.abs(sig ** 2 - sig_r ** 2)) < 1e-8 * VARK
    # sig is sqrt(max(sig2, 0)) sqrt(varK) of the very sig2 returned, and the counter counts its negative entries
    assert np.array_equal(sig, np.sqrt(np.maximum(sig2, 0.0)) * np.sqrt(VARK))
    assert nneg == int(np.sum(sig2 < 0))


def _check_grads(sig, dmu, dsig, ref):
    _, sig_r, dmu_r, dsig_r = ref
    assert _err(dmu, dmu_r) < 1e-8
    far = sig_r > 1e-3 * np.max(sig_r)          # d sigma / d x divides by sigma: compare away from the data
    assert far.sum() > 0
    assert np.max(np.abs(dsig[far] - dsig_r[far])) < 1e-6 * np.max(np.abs(dsig_r[far]))


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


# ---------------------------------------------------------------------------------------------------------------------
# 1. gegp_cross_cov
# ---------------------------------------------------------------------------------------------------------------------
CROSS_CASES = [  # kernel, masked, pinv, n, d, nx
    ("SqExp", False, False, 37, 1, 1), ("SqExp", True, True, 300, 12, 13), ("Ma5f2", False, True, 300, 3, 13),
    ("Ma5f2", True, False, 37, 12, 1), ("RatQu", True, True, 37, 3, 13), ("RatQu", False, False, 300, 1, 13)]


@pytest.mark.parametrize("kname,masked,use_pinv,n,d,nx", CROSS_CASES)
def test_cross_cov_vs_oracle(kname, masked, use_pinv, n, d, nx):
    """n = 300: two 256-wide blocks of training points; nx = 13: a partial 8-point tail; d = 12: long column loops."""
    from gpgradpy_b200 import backend as bk
    from oracle import gegp_oracle as O
    x, _, _ = O.synthetic_problem(n, d, 3)
    xs = np.random.default_rng(4).uniform(-2, 2, (nx, d))
    th = _theta(n, d)
    kern = KERNELS[kname]
    mask = _mask(n, 5) if masked else None
    slot, ng = bk.slot_from_mask(mask, n)
    diag = np.diag(O.kern_grad(x, x, th, mask, mask, kernel=kern))      # p^2 of the preconditioner (noise-free)
    pinv = 1.0 / np.sqrt(diag) if use_pinv else None
    got = bk.cross_cov(x, xs, th, n_g=ng, slot=slot, pinv=pinv, kernel=kern).cpu().numpy()
    ref = O.kern_grad(x, xs, th, mask, None, kernel=kern)[:, :nx].T
    colscale = np.sqrt(diag)                        # |k*| <= sqrt(k(x*, x*) K_cc) = sqrt(K_cc) in every column c
    if pinv is not None:
        ref, colscale = ref * pinv[None, :], colscale * pinv
    assert got.shape == ref.shape
    scale = np.maximum(np.abs(ref), 1e-3 * colscale[None, :])
    e = float(np.max(np.abs(got - ref) / scale))
    print(f"cross_cov {kname} mask={masked} pinv={use_pinv} n={n} d={d} nx={nx}: {e:.2e}")
    assert e < 1e-12


def test_cross_cov_nx_zero_writes_nothing():
    import torch
    from gpgradpy_b200 import backend as bk, _lib as L
    from oracle import gegp_oracle as O
    n, d = 37, 3
    x, _, _ = O.synthetic_problem(n, d, 3)
    X, th = bk.to_dev(x), bk.to_dev(_theta(n, d))
    ld = bk.ld_of(n * (d + 1))
    out = torch.full((4, ld), 12345.5, dtype=torch.float64, device=bk.device())
    Xs = torch.zeros((1, d), dtype=torch.float64, device=bk.device())
    rc = L.load().gegp_cross_cov(n, n, d, X.data_ptr(), 0, Xs.data_ptr(), 0, th.data_ptr(), L.KERNEL_SQEXP, 0.0, 0,
                                 out.data_ptr(), ld, bk._stream())
    torch.cuda.synchronize()
    assert rc == 0
    assert bool((out == 12345.5).all())


# ---------------------------------------------------------------------------------------------------------------------
# 2. / 3. gegp_predict and gegp_predict_grad
# ---------------------------------------------------------------------------------------------------------------------
SMALL, LARGE = (20, 2), (250, 3)     # N = 60 (one leaf: no GEMM) and N = 1000 (recursive solve with GEMM updates)
PRED_CASES = [  # kernel, masked, noisy, mode, size
    ("SqExp", False, False, "precon", SMALL), ("SqExp", True, True, "base", LARGE), ("SqExp", True, True, "precon", SMALL),
    ("Ma5f2", True, False, "base", SMALL), ("Ma5f2", False, True, "precon", LARGE), ("Ma5f2", False, False, "base", LARGE),
    ("RatQu", False, True, "base", SMALL), ("RatQu", True, False, "precon", LARGE)]


def _case_id(c):
    return f"{c[0]}-{'mask' if c[1] else 'full'}-{'noisy' if c[2] else 'exact'}-{c[3]}-N{c[4][0] * (c[4][1] + 1)}"


@pytest.mark.parametrize("case", PRED_CASES, ids=_case_id)
def test_predict_vs_oracle(case):
    from gpgradpy_b200 import backend as bk
    kname, masked, noisy, mode, (n, d) = case
    p = _problem(n, d, kname, masked=masked, noisy=noisy, mode=mode, seed=1)
    xs = _test_points(p, 45, 2, n_on_data=5)           # the last five sit exactly on training points
    mu, sig, sig2, nneg = bk.predict(p["st"], xs, VARK)
    mu, sig, sig2, nneg = _np(mu, sig, sig2, nneg)
    _check_values(mu, sig, sig2, int(nneg[0]), _ref(p, xs, False))


@pytest.mark.parametrize("case", PRED_CASES, ids=_case_id)
def test_predict_grad_vs_oracle(case):
    from gpgradpy_b200 import backend as bk
    kname, masked, noisy, mode, (n, d) = case
    p = _problem(n, d, kname, masked=masked, noisy=noisy, mode=mode, seed=1)
    xs = _test_points(p, 45, 3, n_on_data=5)
    mu, sig, sig2, dmu, dsig, nneg = _np(*bk.predict_grad(p["st"], xs, VARK))
    ref = _ref(p, xs, True)
    _check_values(mu, sig, sig2, int(nneg[0]), (ref[0], ref[1], _ref_sig2(p, xs)))
    _check_grads(sig, dmu, dsig, ref)
    # the value outputs are those of gegp_predict (the same solved row, the same reduction)
    mu0, sig0, sig20, _ = _np(*bk.predict(p["st"], xs, VARK))
    assert _err(mu, mu0) < 1e-12 and np.max(np.abs(sig2 - sig20)) < 1e-12


@pytest.fixture
def force_tma():
    """Route every GEMM with M, N >= 128 through the TMA kernel (normally only >= 400 tiles of 128 x 128)."""
    from gpgradpy_b200 import _lib
    lib = _lib.load()
    old = lib.gegp_set_option(_lib.OPT_TMA_MIN_TILES, 1)
    assert old >= 1
    yield
    lib.gegp_set_option(_lib.OPT_TMA_MIN_TILES, old)


def _tall_solve():
    """n = 100, d = 9 (N = 1000), 1100 test points in one chunk: 11,000 solved rows, above the 148 * 64 rows where the
    leaf solve switches to 16-warp strips and the K = 128 panel updates leave the single-wave kernel."""
    from gpgradpy_b200 import backend as bk
    p = _problem(100, 9, "SqExp", seed=2)
    xs = _test_points(p, 1100, 4, n_on_data=4)
    assert 1100 * 10 > 148 * 64
    mu, sig, sig2, dmu, dsig, nneg = _np(*bk.predict_grad(p["st"], xs, VARK))
    ref = _ref(p, xs, True)
    _check_values(mu, sig, sig2, int(nneg[0]), (ref[0], ref[1], _ref_sig2(p, xs)))
    _check_grads(sig, dmu, dsig, ref)


def test_predict_grad_tall_solve():
    _tall_solve()


def test_predict_grad_tall_solve_tma(force_tma):
    _tall_solve()


# ---------------------------------------------------------------------------------------------------------------------
# 4. chunk invariance
# ---------------------------------------------------------------------------------------------------------------------
def _chunked(p, xs, grad, points):
    from gpgradpy_b200 import backend as bk
    per = bk.ld_of(p["N"]) * 8 * ((p["d"] + 1) if grad else 1)
    fn = bk.predict_grad if grad else bk.predict
    out = _np(*fn(p["st"], xs, VARK, chunk_bytes=points * per))
    return out[:-1], int(out[-1][0])


@pytest.mark.parametrize("grad", [False, True])
@pytest.mark.parametrize("size", [SMALL, LARGE], ids=["N60", "N1000"])
def test_chunk_invariance(grad, size):
    """The test set in chunks of 1, 7, nx - 1 and nx points.  N = 60: one leaf solve per chunk, the same arithmetic per
    row whatever the chunk, so bit-identical.  N = 1000: the GEMM tiling follows the chunk's row count: equal to
    rounding (1e-12), and each chunking matches the oracle."""
    kname, masked = ("Ma5f2", True) if size == SMALL else ("SqExp", False)
    p = _problem(*size, kname, masked=masked, seed=5)
    nx = 37
    xs = _test_points(p, nx, 6, n_on_data=3)
    ref = _ref(p, xs, grad)
    full, nneg_full = _chunked(p, xs, grad, nx)
    for pts in (1, 7, nx - 1):
        got, nneg = _chunked(p, xs, grad, pts)
        assert nneg == nneg_full
        if size == SMALL:
            for a, b in zip(got, full):
                assert np.array_equal(a, b), pts
        else:
            mu, sig, sig2 = got[:3]
            assert _err(mu, full[0]) < 1e-12 and np.max(np.abs(sig2 - full[2])) < 1e-12
            if grad:
                far = full[1] > 1e-1 * np.max(full[1])
                assert _err(got[3], full[3]) < 1e-12
                assert np.max(np.abs(got[4][far] - full[4][far])) < 1e-12 * np.max(np.abs(full[4][far]))
        mu, sig, sig2 = got[:3]
        sig2_r = _ref_sig2(p, xs) if grad else ref[2]
        _check_values(mu, sig, sig2, nneg, (ref[0], ref[1], sig2_r))
        if grad:
            _check_grads(sig, got[3], got[4], ref)


# ---------------------------------------------------------------------------------------------------------------------
# 5. test sets longer than one launch's 65,535 grid rows
# ---------------------------------------------------------------------------------------------------------------------
def _slices(nx, centre):
    return [np.arange(512), np.arange(centre - 2048, centre + 2048), np.arange(nx - 512, nx)]


def test_predict_grad_70k_points_one_chunk():
    """n = 20, d = 2 (N = 60): 1 GiB holds ~700k gradient points, so 70,000 points are one chunk and one
    cross-covariance launch with a test point per grid row."""
    from gpgradpy_b200 import backend as bk
    p = _problem(20, 2, seed=8)
    nx = 70_000
    xs = np.random.default_rng(9).uniform(-2.5, 2.5, (nx, 2))
    mu, sig, sig2, dmu, dsig, nneg = _np(*bk.predict_grad(p["st"], xs, VARK))
    assert int(nneg[0]) == int(np.sum(sig2 < 0))
    for idx in _slices(nx, 65_535):
        ref = _ref(p, xs[idx], True)
        _check_values(mu[idx], sig[idx], sig2[idx], int(np.sum(sig2[idx] < 0)),
                      (ref[0], ref[1], _ref_sig2(p, xs[idx])))
        _check_grads(sig[idx], dmu[idx], dsig[idx], ref)


def test_predict_600k_points_one_chunk():
    """600,000 points (more than 8 x 65,535: eight test points per grid row) in one chunk at N = 60."""
    from gpgradpy_b200 import backend as bk
    p = _problem(20, 2, seed=8)
    nx = 600_000
    xs = np.random.default_rng(10).uniform(-2.5, 2.5, (nx, 2))
    mu, sig, sig2, nneg = _np(*bk.predict(p["st"], xs, VARK))
    assert int(nneg[0]) == int(np.sum(sig2 < 0))
    for idx in _slices(nx, 8 * 65_535):
        _check_values(mu[idx], sig[idx], sig2[idx], int(np.sum(sig2[idx] < 0)), _ref(p, xs[idx], False))


def test_gaussian_process_eval_model_on_a_300x300_grid():
    """End to end: GaussianProcess.eval_model(x, calc_grad=True) on a 90,000-point plotting grid (n = 20, d = 2)."""
    from gpgradpy_b200.gp import GaussianProcess
    from oracle import gegp_oracle as O
    n, d = 20, 2
    x, f, g = O.synthetic_problem(n, d, 8)
    th = _theta(n, d)
    GP = GaussianProcess(d, True, "SqExp", "precon")
    GP.set_data(x, f, np.zeros(n), g, np.zeros(g.shape))
    assert not GP.b_use_data_scl
    beta = float(np.mean(f))
    GP.set_hpara("set", 1, GP.make_hp_class(theta=th, varK=VARK, beta=np.array([beta])))
    t = np.linspace(-2.0, 2.0, 300)
    grid = np.stack(np.meshgrid(t, t), axis=-1).reshape(-1, 2)
    mu, sig, dmu, dsig = GP.eval_model(grid, calc_grad=True)[:4]
    assert mu.shape == (90_000,) and dmu.shape == (90_000, 2)
    for idx in _slices(90_000, 65_535):
        ref = O.eval_model_grad(x, f, g, th, VARK, np.array([beta]), grid[idx], "precon", GP._etaK)
        assert _err(mu[idx], ref[0]) < 1e-8
        assert np.max(np.abs(sig[idx] ** 2 - ref[1] ** 2)) < 1e-8 * VARK
        _check_grads(sig[idx], dmu[idx], dsig[idx], ref)


# ---------------------------------------------------------------------------------------------------------------------
# 6. gegp_predict_hess
# ---------------------------------------------------------------------------------------------------------------------
HESS_CASES = [  # kernel, masked, noisy, mode, n, d
    ("SqExp", False, False, "precon", 14, 3), ("SqExp", True, True, "base", 14, 3), ("Ma5f2", True, False, "base", 14, 3),
    ("Ma5f2", False, True, "precon", 14, 3), ("RatQu", False, True, "base", 14, 3), ("RatQu", True, False, "precon", 14, 3),
    ("SqExp", True, False, "precon", 300, 2),     # n > 256: the per-point loop strides
    ("Ma5f2", False, False, "base", 20, 12),      # 144 CTAs
    ("RatQu", True, True, "precon", 20, 12)]


def _hess_id(c):
    return f"{c[0]}-{'mask' if c[1] else 'full'}-{'noisy' if c[2] else 'exact'}-{c[3]}-n{c[4]}-d{c[5]}"


@pytest.mark.parametrize("case", HESS_CASES, ids=_hess_id)
def test_predict_hess_vs_oracle(case):
    from gpgradpy_b200 import backend as bk
    from oracle import gegp_oracle as O
    kname, masked, noisy, mode, n, d = case
    p = _problem(n, d, kname, masked=masked, noisy=noisy, mode=mode, seed=11)
    xs = np.random.default_rng(12).uniform(-1.5, 1.5, d)
    mu, sig, sig2, dmu, dsig, h3, nneg = _np(*bk.predict_hess(p["st"], xs, VARK))
    h = O.eval_model_hess(*p["oargs"], xs, p["okw"]["mode"], p["okw"]["eta"], kernel=p["kern"],
                          noise_vec=p["okw"]["noise_vec"], mask=p["mask"])
    assert h[1][0] > 1e-3 * np.sqrt(VARK)                  # away from the data: d2sig is well defined
    d2mu = h3[0]
    d2sig2 = -2.0 * VARK * (h3[1] + h3[2])                  # eval/GpEvalModel.py:366-371, as GaussianProcess.eval_model
    d2sig = (d2sig2 - 2.0 * np.outer(dsig, dsig)) / (2.0 * sig[0])
    e = {"mu": _err(mu, h[0]), "dmu": _err(dmu, h[2][0]), "dsig": _err(dsig, h[3][0]), "d2mu": _err(d2mu, h[4][0]),
         "d2sig": _err(d2sig, h[5][0])}
    print(_hess_id(case), {k: f"{v:.1e}" for k, v in e.items()})
    assert e["mu"] < 1e-8 and e["dmu"] < 1e-8 and e["d2mu"] < 1e-8
    assert e["dsig"] < 1e-6 and e["d2sig"] < 1e-5
    assert np.array_equal(sig, np.sqrt(np.maximum(sig2, 0.0)) * np.sqrt(VARK)) and int(nneg[0]) == int(sig2[0] < 0)
    assert np.array_equal(h3, h3.transpose(0, 2, 1))         # each slab exactly symmetric
