"""GPU: batched 2-norm condition numbers -- the batched restarted Lanczos (backend.extreme_eig_batch), the kappa columns
of GaussianProcess.calc_lkd_batch(calc_cond=True) and the condition-number-constrained lock-step multi-start fits.
A candidate's kappa must not depend on the batch it is evaluated in: every comparison with the one-candidate path is
bit for bit."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _load(golden_dir, name):
    z = np.load(os.path.join(golden_dir, name + ".npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def _spd(N, seed, w):
    Q = np.linalg.qr(np.random.default_rng(seed).standard_normal((N, N)))[0]
    M = (Q * w) @ Q.T
    return 0.5 * (M + M.T)


def test_extreme_eig_batch_equals_single():
    """Five SPD matrices of order 300 in one batch: one breaks down after two steps (c I + rank one), one needs
    restarts (no gap at the top of the spectrum), one is warm-started.  Each candidate's (lambda, v, residual, matvecs)
    equals extreme_eig on that matrix alone bit for bit, and eigh to 1e-11."""
    import torch
    from gpgradpy_b200 import backend as bk
    N = 300
    rng = np.random.default_rng(7)
    u = rng.standard_normal(N)
    mats = [_spd(N, 1, np.sort(10.0 ** rng.uniform(-4, 2, N))),
            3.0 * np.eye(N) + np.outer(u, u),
            _spd(N, 2, np.linspace(1.0, 2.0, N)),
            _spd(N, 3, np.sort(10.0 ** rng.uniform(-2, 0, N))),
            _spd(N, 4, np.sort(rng.uniform(0.5, 50.0, N)))]
    ld = bk.ld_of(N)
    Md = torch.zeros((len(mats), N + 3, ld), dtype=torch.float64, device="cuda")   # a stride other than N * ld
    for c, M in enumerate(mats):
        Md[c, :N, :N] = bk.to_dev(M)
    warm = [None, None, None, bk.to_dev(np.linalg.eigh(mats[3])[1][:, -1] + 1e-3 * rng.standard_normal(N)), None]
    lam, vec, res, mv = bk.extreme_eig_batch(Md, N, v0=warm)
    for c, M in enumerate(mats):
        l1, v1, r1, m1 = bk.extreme_eig(Md[c], N, v0=warm[c])
        assert lam[c] == l1 and res[c] == r1 and mv[c] == m1 and torch.equal(vec[c], v1), c
        wr = np.linalg.eigh(M)[0]
        assert abs(lam[c] - wr[-1]) < 1e-11 * wr[-1], c
    assert mv[1] <= 8                  # breakdown: the Krylov space of c I + u u^T has dimension 2
    assert abs(lam[1] - (3.0 + u @ u)) < 1e-11 * lam[1]
    assert mv[2] > 40                  # restarted (k = 40)
    # a subset of the candidates, in any composition: the same results
    lam2, vec2, res2, mv2 = bk.extreme_eig_batch(Md, N, v0=warm, rows=[4, 2])
    assert lam2[0] is None and lam2[4] == lam[4] and lam2[2] == lam[2] and torch.equal(vec2[2], vec[2])
    assert mv2[4] == mv[4] and res2[2] == res[2]


def _gp(kind, mode, kernel="SqExp", n=16, d=2, seed=0):
    from gpgradpy_b200.gp import GaussianProcess
    from oracle import gegp_oracle as O
    x, f, g = O.synthetic_problem(n, d, seed)
    GP = GaussianProcess(d, True, kernel, mode)
    GP.cond_warm_start = False
    std_f, std_g = (0.05, 0.1) if kind == "noisy" else (0.0, 0.0)
    mask = None
    if kind == "mask":
        mask = np.random.default_rng(4).uniform(size=n) < 0.6
        mask[0] = True
    if kind == "eta0":
        GP.cond_eta_set_mtd, GP.cond_eta_dflt = "dflt_eta", 0.0
    gm = g if mask is None else g[mask]
    GP.set_data(x, f, std_f * np.ones(n), gm, std_g * np.ones(gm.shape), bvec_use_grad=mask)
    return GP


def _rows(GP, B, seed=1, lo=-1.0, hi=1.0):
    hi_ = GP.hp_info_optz_lkd
    rng = np.random.default_rng(seed)
    rows = np.zeros((B, hi_.n_hp))
    rows[:, hi_.idx_theta] = rng.uniform(lo, hi, (B, GP.dim))
    if hi_.has_kernel:
        rows[:, hi_.idx_kernel[0]] = rng.uniform(-0.5, 0.8, B)
    if hi_.has_varK:
        rows[:, hi_.idx_varK] = rng.uniform(-0.5, 0.5, B)
    return rows


def _hp_of_rows(GP, rows):
    """The hyper-parameter classes calc_lkd_batch forms from its rows (10 ** of the same arrays)."""
    hi = GP.hp_info_optz_lkd
    th = 10 ** rows[:, hi.idx_theta].copy()
    kh = 10 ** rows[:, hi.idx_kernel[0]].copy() if hi.has_kernel else [None] * len(rows)
    vk = 10 ** rows[:, hi.idx_varK].copy() if hi.has_varK else [None] * len(rows)
    return [GP.make_hp_class(theta=th[i], kernel=kh[i], varK=vk[i]) for i in range(len(rows))]


def _check_rows(GP, rows, tab, calc_grad):
    from gpgradpy_b200 import _lib as L
    d, ol = GP.dim, L.out_len(GP.dim)
    with_grad = calc_grad and GP.wellcond_mtd != "precon"
    assert tab.shape == (len(rows), ol + 1 + (GP.hp_info_optz_lkd.n_hp if with_grad else 0))
    n_bad = 0
    for i, hp in enumerate(_hp_of_rows(GP, rows)):
        info, ok = GP.calc_lkd_all(hp, calc_cond=True, calc_grad=calc_grad)
        assert tab[i, ol] == info.cond, (i, tab[i, ol], info.cond)
        if with_grad:
            assert np.array_equal(tab[i, ol + 1:], info.cond_grad), i
        if ok:
            assert tab[i, L.OUT_INFO] == 0 and tab[i, L.OUT_LML] == info.ln_lkd, i
        else:
            n_bad += 1
            assert tab[i, L.OUT_INFO] != 0 or np.isnan(tab[i, L.OUT_LML]), i
    return n_bad


CASES = [("plain", "base", "SqExp"), ("plain", "rescale_origin", "Ma5f2"), ("plain", "precon", "RatQu"),
         ("mask", "base", "RatQu"), ("noisy", "base", "SqExp"), ("plain", "precon", "SqExp")]


@pytest.mark.parametrize("calc_grad", [False, True])
@pytest.mark.parametrize("kind,mode,kernel", CASES)
def test_calc_lkd_batch_cond_equals_calc_lkd_all(kind, mode, kernel, calc_grad):
    """calc_lkd_batch(calc_cond=True) row by row against calc_lkd_all(calc_cond=True) (cond_warm_start off): kappa and
    dkappa/dhp bit for bit, in base, rescale_origin and precon mode (both branches of the precon quirk), with the three
    kernel families, a scattered gradient mask and known noise with a varK column; outside precon mode one row has
    kappa > cond_max_abs."""
    GP = _gp(kind, mode, kernel)
    rows = _rows(GP, 6)
    tab = GP.calc_lkd_batch(rows, calc_grad=calc_grad, calc_cond=True)
    from gpgradpy_b200 import _lib as L
    ol = L.out_len(GP.dim)
    assert np.array_equal(tab[:, :ol][:, [L.OUT_INFO]], np.zeros((6, 1)))
    if mode != "precon":   # cond_max_abs below the largest kappa: that row reports no likelihood
        GP.cond_max_abs = 0.5 * float(np.max(tab[:, ol]))
        tab = GP.calc_lkd_batch(rows, calc_grad=calc_grad, calc_cond=True)
        assert np.isnan(tab[np.argmax(tab[:, ol]), L.OUT_LML])
        assert _check_rows(GP, rows, tab, calc_grad) >= 1
    else:
        assert _check_rows(GP, rows, tab, calc_grad) == 0
    base = GP.calc_lkd_batch(rows, calc_grad=calc_grad)       # without calc_cond: the table of before
    assert base.shape == (6, ol)


@pytest.mark.parametrize("calc_grad", [False, True])
def test_failed_cholesky_row_and_workspace_chunks(calc_grad):
    """Base mode without a nugget, 7 rows of which one is numerically singular: its kappa comes from the shifted
    refactorisation (_cond_on_failure) as in calc_lkd_all; a workspace cap that forces three candidate chunks gives the
    same table bit for bit."""
    from gpgradpy_b200 import _lib as L, backend as bk
    GP = _gp("eta0", "base", n=30)
    rows = _rows(GP, 7, seed=3, lo=0.0, hi=1.0)
    rows[4, :] = -9.0
    tab = GP.calc_lkd_batch(rows, calc_grad=calc_grad, calc_cond=True)
    assert tab[4, L.OUT_INFO] != 0 and tab[4, L.out_len(2)] > 1e12
    assert _check_rows(GP, rows, tab, calc_grad) >= 1
    lib = L.load()
    per = lib.gegp_workspace_bytes(L.OP_LML_GRAD, 30, 30, 2, 2) - lib.gegp_workspace_bytes(L.OP_LML_GRAD, 30, 30, 2, 1)
    GP.lml_ws_max_bytes = 256 + 4 * 7 + 256 + 3 * per
    assert bk.lml_chunk_rows(30, 30, 2, 7, max_ws_bytes=GP.lml_ws_max_bytes) == 3      # chunks of 3, 3, 1
    tab3 = GP.calc_lkd_batch(rows, calc_grad=calc_grad, calc_cond=True)
    assert np.array_equal(tab3, tab, equal_nan=True)


def test_cond_batch_vs_oracle():
    """n = 150, d = 3 (N = 600): kappa and dkappa/dtheta of three rows (kappa 3e6 .. 2e8) against the NumPy oracle, with
    the rule behind the tolerances of test_cond_and_grad_through_the_api: lambda_min is only defined to an absolute
    eps * lambda_max in either implementation, so kappa agrees to ~eps * kappa (tolerance 1e-14 kappa, at least 1e-9)
    and the gradient to 20 times that."""
    from gpgradpy_b200.gp import GaussianProcess
    from gpgradpy_b200 import _lib as L
    from oracle import gegp_oracle as O
    n, d = 150, 3
    x, f, g = O.synthetic_problem(n, d, 5)
    GP = GaussianProcess(d, True, "SqExp", "base")
    GP.set_data(x, f, np.zeros(n), g, np.zeros((n, d)))
    th = np.vstack([O.bench_theta(d) * s for s in (16.0, 32.0, 64.0)])
    tab = GP.calc_lkd_batch(np.log10(th), calc_grad=True, calc_cond=True)
    ol = L.out_len(d)
    for i in range(3):
        c, cg = O.cond_wo_noise(x, 10 ** np.log10(th[i]), "base", GP._etaK)
        tol = max(1e-9, 1e-14 * c)
        assert abs(tab[i, ol] - c) < tol * c, (i, tab[i, ol], c)
        assert np.max(np.abs(tab[i, ol + 1:] - cg)) < 20 * tol * np.max(np.abs(cg)), i


@pytest.mark.parametrize("mode", ["base", "precon", "rescale_origin"])
def test_config1_grid_as_one_call(golden_dir, mode):
    """BASELINE configs[0] (tests/golden/c1_plt_cond_grid.npz) as ONE calc_lkd_batch(calc_cond=True) call per mode,
    with the rules of test_config1_plt_cond_grid."""
    from gpgradpy_b200.gp import GaussianProcess
    from gpgradpy_b200 import _lib as L
    g = _load(golden_dir, "c1_plt_cond_grid")
    x, f, gr, tv = g["x"], g["fval"], g["grad"], g["theta_vec"]
    GP = GaussianProcess(2, True, "SqExp", mode)
    GP.cond_eta_is_const = True
    GP.set_data(x, f, np.zeros(20), gr, np.zeros(gr.shape))
    GP._etaK = float(g["nugget"])
    GP._eta_Kgrad = float(g["nugget"])
    GP.cond_max = 1e10
    ii, jj = np.meshgrid(np.arange(tv.size), np.arange(tv.size), indexing="ij")
    rows = np.log10(np.stack([tv[ii.ravel()], tv[jj.ravel()]], axis=1))
    tab = GP.calc_lkd_batch(rows, calc_cond=True)
    ol = L.out_len(2)
    n_cmp = 0
    for r, (i, j) in enumerate(zip(ii.ravel(), jj.ravel())):
        cond, lml = tab[r, ol], tab[r, L.OUT_LML]
        ok = tab[r, L.OUT_INFO] == 0 and np.isfinite(lml)
        ref_l, ref_c = g[mode + "_lkd"][i, j], g[mode + "_cond"][i, j]
        if ref_c > 1e13:
            assert cond > 1e11
            continue
        assert ok == bool(np.isfinite(ref_l)), (i, j, ok, ref_l, ref_c)
        if not ok:
            assert cond > 1e12
            continue
        tol = max(1e-8, 1e-15 * ref_c)
        assert abs(lml - ref_l) < tol * max(1.0, abs(ref_l)), (i, j, lml, ref_l, ref_c)
        if ref_c < 1e12:
            assert abs(cond - ref_c) < max(1e-8, 1e-15 * ref_c) * ref_c, (i, j, cond, ref_c)
            n_cmp += 1
    assert n_cmp >= 10


def _fit_gp(golden_dir, mode):
    from gpgradpy_b200.gp import GaussianProcess
    g = _load(golden_dir, "fit_d2_n20_" + mode)
    x, f, gr = g["x"], g["fval"], g["grad"]
    n, d = x.shape
    GP = GaussianProcess(d, True, "SqExp", mode)
    GP.init_optz_surr(3)
    GP.set_data(x[:1], f[:1], np.zeros(1), gr[:1], np.zeros((1, d)))
    GP.set_hpara("optz", 0)
    GP.set_data(x, f, np.zeros(n), gr, np.zeros((n, d)))
    hp_x0, bounds = GP.get_hp_x0_lhs_median(1, GP.hp_info_optz_lkd, 5)
    return GP, hp_x0, bounds


@pytest.mark.parametrize("mode", ["base", "rescale_origin"])
def test_constrained_lockstep_fit(golden_dir, mode):
    """A 5-start lhs fit with the kappa <= cond_max constraint: with warm start off the lock step equals the sequential
    loop bit for bit (solution, objective, info); with warm start on every start equals that start fitted alone from
    the same GP state; the chosen optimum satisfies the constraint."""
    GP, hp_x0, bounds = _fit_gp(golden_dir, mode)
    assert GP._can_batch_fit()
    GP.cond_warm_start = False
    best, cond, info = GP.optz_hp_max_lkd(hp_x0, bounds)
    table = GP._multistart_table.copy()
    assert GP._lockstep_stats["batch_sizes"][0] == 5 and GP._lockstep_stats["n_batches"] < GP._lockstep_stats["n_evals"]
    GP.lockstep_multistart = False
    best_s, cond_s, info_s = GP.optz_hp_max_lkd(hp_x0, bounds)
    assert np.array_equal(best, best_s) and cond == cond_s and info == info_s
    assert cond < 1.01 * GP.cond_max and info["hp_optz_con_good"] > 0
    n_hp = GP.hp_info_optz_lkd.n_hp
    GP.lockstep_multistart = True
    GP.cond_warm_start = True
    state = GP._last_cond
    GP.optz_hp_max_lkd(hp_x0, bounds)
    table_w = GP._multistart_table.copy()
    for i in range(5):
        GP._last_cond = state
        b1, _, info1 = GP.optz_hp_max_lkd(hp_x0[i:i + 1], bounds)
        assert np.array_equal(table_w[i, :n_hp], b1) and table_w[i, n_hp + 2] == info1["hp_optz_iter_mean"], i
    # warm start moves kappa only within the Lanczos tolerance: same solutions to rounding
    assert np.allclose(table_w[:, :n_hp], table[:, :n_hp], rtol=1e-6, atol=1e-8)
