"""The likelihood path's two on-the-fly generators against the dense reference of tests/lml_dense_ref.py, at every kernel
variant and tile edge:

* the covariance build (build_cov_fast_kernel / build_cov_kernel), entry by entry at 1e-12 of the block scale, across
  the 8-row / 16-row point tiles and the 64-column tiles, both sides of each shared-memory opt-in, the fast -> generic
  switch, every build mode, uplo 0 / 1, noise and varK, into NaN-poisoned padded outputs; and the batched build;
* the dKcov/dhp contraction (lml_grad_kernel<quad, WIDE, GAUSS>) through gegp_weighted_grad (quad 2),
  gegp_quad_grad (quad 1), gegp_lml_eval (quad 0) and gegp_lml_direct_terms (quad 1 and 2), with the tolerance rule
  |g - g_ref| <= 1e-12 sum(|W .* dKcov/dhp|), which a dropped point pair or one entry off by 1e-9 fails
  (tests/test_lml_dense_ref_cpu.py); the d = 112 / 113 limit; n = 70,000 points (more than gridDim.y holds).

Which case reaches which kernel instantiation is listed beside each case table."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))   # tests/lml_dense_ref.py, whatever the import mode
import lml_dense_ref as R  # noqa: E402
from oracle import gegp_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu

TOL = 1e-12
RQ = ("RatQu", 0.8)


def _block_scale_err(Kg, Kr):
    s = np.sqrt(np.abs(np.diag(Kr)))
    scale = np.maximum(np.abs(Kr), 1e-3 * s[:, None] * s[None, :])
    return float(np.max(np.abs(Kg - Kr) / scale))


def _mask(kind, n, ng, seed):
    if kind is None:
        return None
    m = np.zeros(n, dtype=bool)
    if kind == "prefix":
        m[:ng] = True
    else:
        m[np.random.default_rng(seed).choice(n, ng, replace=False)] = True
    return m


def _problem(n, d, seed, lo=-1.0, hi=1.0):
    rng = np.random.default_rng(seed)
    X = rng.uniform(lo, hi, (n, d))
    theta = rng.uniform(0.5, 1.5, d) * (3.0 / d)
    return X, theta


def _slot(mask, n):
    from gpgradpy_b200 import backend as bk
    return bk.slot_from_mask(mask, n)


# ---------------------------------------------------------------------------------------------------------------------
# covariance build
# ---------------------------------------------------------------------------------------------------------------------
# fast path: Gaussian kernel, every point with a gradient, even n.  n crosses the 8-row a-tile and the 64-column b-tile;
# d = 81 / 82 are the two sides of its shared-memory opt-in; d = 342 no longer fits it and takes the generic kernel.
FAST = [(2, 1), (64, 1), (66, 1), (130, 1), (258, 1), (66, 8), (130, 8), (10, 81), (2, 82), (18, 82), (2, 342)]
# generic kernel: odd n, masks, the other families.  n crosses the 16-row a-tile and the 64-column b-tile; d = 74 / 75
# are the two sides of its opt-in, d = 353 its largest.   (kernel, n, d, mask kind, n_g)
GENERIC = [(None, 17, 3, None, 17), ("Ma5f2", 66, 8, None, 66), (RQ, 65, 5, "scatter", 30), (None, 130, 4, "prefix", 70),
           ("Ma5f2", 17, 74, None, 17), (RQ, 17, 75, None, 17), (None, 33, 75, "scatter", 5), ("Ma5f2", 17, 353, "scatter", 2),
           (None, 16, 353, "prefix", 1)]
MODES = [(0, 0, False), (1, 1, True), (2, 0, True), (0, 1, True), (1, 0, False), (2, 1, False)]   # (mode, uplo, noisy)


def _check_build(X, th, kernel, mask, mode, uplo, noisy, eta=3e-7, seed=0, out_offset=0):
    """gegp_build_cov into a NaN-poisoned buffer of 3 extra rows and 8 extra columns (optionally starting one double
    into it, so that the output base is only 8-byte aligned): entries against cov(); with uplo = 1 the strict upper
    triangle, and always the padding, stays NaN.  Returns the built matrix."""
    from gpgradpy_b200 import backend as bk
    n, d = X.shape
    slot, ng = _slot(mask, n)
    N = n + ng * d
    rng = np.random.default_rng(seed)
    varK = 1.7 if noisy else 1.0
    noise = np.hstack((rng.uniform(1e-4, 1e-2, n), rng.uniform(1e-3, 5e-2, ng * d))) if noisy else None
    ld = bk.ld_of(N) + 8
    buf = torch.full((N + 3, ld + 2), float("nan"), dtype=torch.float64, device="cuda")
    out = buf[:, out_offset:out_offset + ld]
    _, p = bk.build_cov(X, th, n_g=ng, slot=slot, noise=noise, mode=mode, eta=eta, varK=varK, uplo=uplo, out=out,
                        kernel=kernel)
    Kg = out.cpu().numpy()
    Kr, pr = R.cov(X, th, mode, eta, mask, kernel, noise, varK)
    Km = Kg[:N, :N]
    if uplo:
        iu = np.triu_indices(N, 1)
        assert np.all(np.isnan(Km[iu]))
        Km = np.tril(Km) + np.tril(Km, -1).T
    assert np.all(np.isfinite(Km))
    assert np.all(np.isnan(Kg[N:])) and np.all(np.isnan(Kg[:, N:]))
    full = buf.cpu().numpy()
    assert np.all(np.isnan(np.delete(full, np.s_[out_offset:out_offset + N], axis=1)[:N]))
    e = _block_scale_err(Km, Kr)
    assert e < TOL, e
    if mode == 1:
        pg = p.cpu().numpy()
        assert np.max(np.abs(pg[:N] / pr - 1.0)) < 1e-15
        assert np.max(np.abs(pg[N:] * pr - 1.0)) < 1e-15
    return Km


@pytest.mark.parametrize("n,d", FAST)
def test_build_fast_path_vs_dense_reference(n, d):
    X, th = _problem(n, d, seed=n + d)
    for i, (mode, uplo, noisy) in enumerate(MODES if n * (d + 1) <= 600 else MODES[(n + d) % 6:][:2]):
        _check_build(X, th, None, None, mode, uplo, noisy, seed=i)


@pytest.mark.parametrize("kernel,n,d,mk,ng", GENERIC)
def test_build_generic_path_vs_dense_reference(kernel, n, d, mk, ng):
    X, th = _problem(n, d, seed=3 * n + d)
    mask = _mask(mk, n, ng, seed=d)
    N = n + ng * d
    for i, (mode, uplo, noisy) in enumerate(MODES if N <= 600 else MODES[(n + d) % 6:][:2]):
        _check_build(X, th, kernel, mask, mode, uplo, noisy, seed=i)


@pytest.mark.parametrize("n,d", [(66, 3), (130, 8), (2, 82)])
def test_build_fast_path_agrees_with_generic_kernel(n, d):
    """The same fast-eligible problem built by the fast kernel and, into an output whose base is only 8-byte aligned, by
    the generic kernel: agreement to rounding in every mode.  The two order their products differently, so an entry where
    its terms cancel (the (i, i) blocks: (2 th_i - 4 th_i^2 r_i^2) k) differs by a few ulps of the terms, which are
    bounded by sqrt(K_ii K_jj): measured against that, not against the entry."""
    X, th = _problem(n, d, seed=7)
    for mode, uplo, noisy in MODES:
        Kf = _check_build(X, th, None, None, mode, uplo, noisy)
        Kg = _check_build(X, th, None, None, mode, uplo, noisy, out_offset=1)
        s = np.sqrt(np.diag(Kf))
        assert np.max(np.abs(Kg - Kf) / (s[:, None] * s[None, :])) < 1e-14


def test_build_rejects_d_354_and_writes_nothing():
    from gpgradpy_b200 import _lib as L
    lib = L.load()
    for n, d, ng in ((3, 354, 3), (4, 354, 1)):
        X, th = _problem(n, d, seed=1)
        slot, ng = _slot(_mask("prefix", n, ng, 0) if ng < n else None, n)
        N = n + ng * d
        Xd, thd = torch.as_tensor(X, device="cuda"), torch.as_tensor(th, device="cuda")
        out = torch.full((N, N + N % 2), float("nan"), dtype=torch.float64, device="cuda")
        rc = lib.gegp_build_cov(n, ng, d, Xd.data_ptr(), 0 if slot is None else slot.data_ptr(), thd.data_ptr(), 0, 0.0, 0,
                                0, 1e-8, 1.0, out.data_ptr(), out.stride(0), 0, 0, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert rc == -907
        assert torch.isnan(out).all()


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_build_cov_batch_rows_vs_reference_and_single_builds(mode):
    """Three rows with their own theta, varK and rational-quadratic alpha into a strided, NaN-poisoned output: each row
    matches cov() of that row and is bit-identical to gegp_build_cov of that row."""
    from gpgradpy_b200 import backend as bk
    n, d, ng = 67, 5, 40
    X, th0 = _problem(n, d, seed=11)
    mask = _mask("scatter", n, ng, 5)
    slot, ng = _slot(mask, n)
    N = n + ng * d
    rng = np.random.default_rng(12)
    th = th0[None, :] * rng.uniform(0.6, 1.6, (3, d))
    vk = np.array([0.7, 1.0, 2.3])
    al = np.array([0.6, 1.5, 4.0])
    noise = np.hstack((rng.uniform(1e-4, 1e-2, n), rng.uniform(1e-3, 5e-2, ng * d)))
    ld = bk.ld_of(N) + 4
    buf = torch.full((3, N + 2, ld), float("nan"), dtype=torch.float64, device="cuda")
    bk.build_cov_batch(X, th, n_g=ng, slot=slot, noise=bk.to_dev(noise), varK_rows=vk, mode=mode, eta=2e-7, out=buf,
                       kernel="RatQu", kernel_hp_rows=al)
    got = buf.cpu().numpy()
    for z in range(3):
        assert np.all(np.isnan(got[z, N:])) and np.all(np.isnan(got[z, :, N:]))
        Kr, _ = R.cov(X, th[z], mode, 2e-7, mask, ("RatQu", al[z]), noise / vk[z], vk[z])
        assert _block_scale_err(got[z, :N, :N], Kr) < TOL
        Ks, _ = bk.build_cov(X, th[z], n_g=ng, slot=slot, noise=noise / vk[z], mode=mode, eta=2e-7, varK=vk[z],
                             kernel=("RatQu", al[z]))
        assert np.array_equal(Ks.cpu().numpy(), got[z, :N, :N])


# ---------------------------------------------------------------------------------------------------------------------
# contraction, quad 1 (gegp_quad_grad) and quad 2 (gegp_weighted_grad)
# ---------------------------------------------------------------------------------------------------------------------
# (kernel, n, d, mask kind, n_g, noisy).  Narrow (d < 8) and wide (d >= 8) instantiations of both families' kernels;
# d mod 4 = 1, 3 (wide remainder loop) and 0; d = 23 / 24 the two sides of the wide kernels' opt-in, d = 112 the largest;
# n = 1, 127, 128, 129, 300 (CTAs with b >= n; the diagonal CTA and the ones off it); scatter masks at n > 128.
CONTRACT = [(None, 129, 5, None, 129, False), ("Ma5f2", 127, 5, "scatter", 60, True), (RQ, 300, 7, "scatter", 30, False),
            (None, 128, 8, None, 128, True), ("Ma5f2", 129, 9, "scatter", 40, False), (RQ, 40, 11, None, 40, True),
            (None, 1, 23, None, 1, False), ("Ma5f2", 60, 23, None, 60, False), (RQ, 57, 24, None, 57, True),
            (None, 300, 24, "scatter", 20, False), ("Ma5f2", 20, 40, "scatter", 12, True), (None, 13, 40, None, 13, True),
            (("RatQu", 2.0), 3, 112, None, 3, False), (None, 1, 112, None, 1, True), ("Ma5f2", 130, 112, "scatter", 2, True)]


@pytest.mark.parametrize("kernel,n,d,mk,ng,noisy", CONTRACT)
def test_quad_and_weighted_contraction_vs_dense_reference(kernel, n, d, mk, ng, noisy):
    from gpgradpy_b200 import backend as bk
    X, th = _problem(n, d, seed=n * 7 + d)
    mask = _mask(mk, n, ng, seed=n)
    slot, ng = _slot(mask, n)
    N = n + ng * d
    rng = np.random.default_rng(d)
    v = rng.standard_normal(N)
    W = rng.standard_normal((N, N))
    W = W + W.T
    eta, varK = 3e-6, (2.1 if noisy else 1.0)
    Wd = torch.zeros((N, bk.ld_of(N)), dtype=torch.float64, device="cuda")
    Wd[:, :N] = torch.as_tensor(W, device="cuda")
    g1 = bk.quad_grad(X, th, v, n_g=ng, slot=slot, eta=eta, noisy=noisy, varK=varK, kernel=kernel).cpu().numpy()
    g2 = bk.weighted_grad(X, th, Wd, n_g=ng, slot=slot, eta=eta, noisy=noisy, varK=varK, kernel=kernel).cpu().numpy()
    r1, s1, r2, s2 = (np.zeros_like(g1) for _ in range(4))
    for k, D in R.dcov_hp(X, th, 0, eta, mask, kernel, noisy, varK):
        r1[k], s1[k] = R.weigh(D, v)
        r2[k], s2[k] = R.weigh(D, W)
    slots = R.hp_slots(d, kernel, noisy)
    e1, e2 = R.contract_err(g1, r1, s1, slots), R.contract_err(g2, r2, s2, slots)
    print(f"quad 1: {e1:.2e}  quad 2: {e2:.2e}")
    assert e1 <= TOL and e2 <= TOL, (e1, e2)
    others = [k for k in range(len(g1)) if k not in slots]
    assert not np.any(g1[others]) and not np.any(g2[others])


def test_contraction_d113_returns_an_error_and_leaves_out_unwritten():
    """d = 112 is the largest dimension the contraction's shared memory holds (run above); at d = 113 every entry point
    that reaches it returns -907 instead of a launch error, and gegp_quad_grad / gegp_weighted_grad leave out unwritten."""
    from gpgradpy_b200 import _lib as L, backend as bk
    lib = L.load()
    n, d = 2, 113
    N = n * (d + 1)
    X, th = _problem(n, d, seed=3)
    Xd, thd = bk.to_dev(X), bk.to_dev(th)
    v = bk.to_dev(np.ones(N))
    W = torch.eye(N, dtype=torch.float64, device="cuda")
    vk = bk.to_dev(np.array([1.0]))
    st = torch.cuda.current_stream().cuda_stream
    out = torch.full((L.out_len(d),), float("nan"), dtype=torch.float64, device="cuda")
    nb = int(lib.gegp_quad_grad_work_bytes(n, n, d)) + 8 * (N + 2)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    rc = lib.gegp_quad_grad(n, n, d, Xd.data_ptr(), 0, thd.data_ptr(), 0, 0.0, v.data_ptr(), 0, 1e-6, 1, vk.data_ptr(),
                            out.data_ptr(), ws.data_ptr(), nb, st)
    torch.cuda.synchronize()
    assert rc == -907 and torch.isnan(out).all()
    rc = lib.gegp_weighted_grad(n, n, d, Xd.data_ptr(), 0, thd.data_ptr(), 1, 0.0, W.data_ptr(), W.stride(0), 0, 1e-6, 0,
                                0, out.data_ptr(), ws.data_ptr(), nb, st)
    torch.cuda.synchronize()
    assert rc == -907 and torch.isnan(out).all()
    y = np.random.default_rng(0).standard_normal(N)
    with pytest.raises(RuntimeError, match="code -907"):
        bk.lml_eval(X, y, th[None, :], mode=L.MODE_PRECON, eta=1e-6, want_grad=True)
    o, _ = bk.lml_eval(X, y, th[None, :], mode=L.MODE_PRECON, eta=1e-6, want_grad=False)
    assert o.cpu().numpy()[0, L.OUT_INFO] == 0


def test_quad_grad_70000_points_gradient_free():
    """A gradient-free GP of n = 70,000 points puts more points a on the contraction's grid than gridDim.y holds
    (65,535): the launch is sliced.  Reference: sum_ab v_a v_b dk(x_a, x_b)/dtheta_m = -sum_ab v_a v_b r_m^2 k in fp64
    torch, chunked over a."""
    from gpgradpy_b200 import backend as bk
    n, d = 70000, 2
    rng = np.random.default_rng(70)
    X = rng.uniform(-3.0, 3.0, (n, d))
    th = np.array([0.8, 2.5])
    v = rng.standard_normal(n)
    slot = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    g = bk.quad_grad(X, th, v, n_g=0, slot=slot, eta=0.0, kernel=None).cpu().numpy()
    Xd, vd, thd = bk.to_dev(X), bk.to_dev(v), bk.to_dev(th)
    ref, scale = torch.zeros(d, dtype=torch.float64, device="cuda"), torch.zeros(d, dtype=torch.float64, device="cuda")
    for a0 in range(0, n, 2048):
        Rm = Xd[a0:a0 + 2048, None, :] - Xd[None, :, :]                  # [ta, n, d]
        R2 = Rm * Rm
        k = torch.exp(-(R2 @ thd))
        vv = (vd[a0:a0 + 2048, None] * vd[None, :]) * k
        for m in range(d):
            t = vv * R2[:, :, m]
            ref[m] -= t.sum()
            scale[m] += t.abs().sum()
        del Rm, R2, k, vv, t
    ref, scale = ref.cpu().numpy(), scale.cpu().numpy()
    from gpgradpy_b200 import _lib as L
    e = float(np.max(np.abs(g[L.OUT_GRAD:L.OUT_GRAD + d] - ref) / scale))
    print(f"n = 70000: {e:.2e}")
    assert e <= TOL, e


# ---------------------------------------------------------------------------------------------------------------------
# contraction, quad 0 (gegp_lml_eval with the gradient) and the direct terms
# ---------------------------------------------------------------------------------------------------------------------
# (kernel, n, d, mask kind, n_g, noisy, mode).  Wide non-Gaussian quad 0 at d = 8, 10, 24 (d = 24: its opt-in), the
# narrow and the Gaussian ones (wide at d = 8 and, past its opt-in, 24) beside them; n across 128.
LML = [("Ma5f2", 130, 8, "scatter", 40, False, 1), (RQ, 129, 10, None, 129, True, 0), ("Ma5f2", 129, 24, "scatter", 30, True, 1),
       (("RatQu", 1.3), 130, 24, "scatter", 20, False, 0), (None, 131, 8, "scatter", 50, True, 1),
       ("Ma5f2", 140, 5, "prefix", 90, False, 1), (None, 129, 5, None, 129, False, 0), (None, 50, 24, "scatter", 20, False, 1)]


def _lml_case(kernel, n, d, mk, ng, noisy, mode, seed):
    x, f, gr = O.synthetic_problem(n, d, seed)
    th = np.random.default_rng(seed).uniform(0.5, 1.5, d) * (1.0 / d)
    mask = _mask(mk, n, ng, seed)
    gr = gr[O._sel(n, mask)]                  # the gradients the GP is given (the oracle takes them already masked)
    y = O.make_data_vec(f, gr)
    ng = gr.shape[0]
    noise = np.hstack((np.full(n, 1e-4), np.full(ng * d, 1e-3))) if noisy else None
    eta = O.nugget(n, d, "precon" if mode == 1 else "base", kernel=kernel)[1]
    return x, f, gr, th, mask, y, noise, eta


@pytest.mark.parametrize("kernel,n,d,mk,ng,noisy,mode", LML)
def test_lml_gradient_contraction_vs_dense_reference_and_oracle(kernel, n, d, mk, ng, noisy, mode):
    """W = P^-1 (c1 alpha alpha^T - K~^-1 / 2) P^-1 built from the evaluation's own K~^-1 and p^-1 (the workspace) and
    alpha (alpha_out = P^-1 alpha~ = Kcov^-1 (y - H beta), the un-preconditioned one), c1 = 1 / (2 sigma^2) noise-free and
    1/2 noisy: the gradient row (with the precon term c eta DG and the noisy rows) meets the tolerance rule.  End to end
    the evaluation agrees with oracle.lkd_wo_noise / lkd_w_noise at 1e-8."""
    from gpgradpy_b200 import _lib as L, backend as bk
    x, f, gr, th, mask, y, noise, eta = _lml_case(kernel, n, d, mk, ng, noisy, mode, seed=n + d)
    slot, ng = _slot(mask, n)
    varK = 1.9
    out, alpha = bk.lml_eval(x, y, th[None, :], n_g=ng, slot=slot, mode=mode, eta=eta, noise=noise,
                             varK_batch=np.array([varK]) if noisy else None, want_grad=True, want_alpha=True, kernel=kernel)
    o = out.cpu().numpy()[0]
    assert o[L.OUT_INFO] == 0
    v = bk.lml_views(n, ng, x.shape[1])
    N = y.size
    Kinv = v["Kinv"][:, :N].cpu().numpy()
    pinv = v["pinv"].cpu().numpy()
    a = alpha.cpu().numpy()[0]
    c1 = 0.5 if noisy else 1.0 / (2.0 * o[L.OUT_SIGMA2])
    W = c1 * np.outer(a, a) - 0.5 * (pinv[:, None] * Kinv * pinv[None, :])
    g, sc = R.contract(x, th, W, mode, eta, mask, kernel, noisy, varK)
    slots = R.hp_slots(d, kernel, noisy)
    e = R.contract_err(o, g, sc, slots)
    print(f"quad 0 vs contract: {e:.2e}")
    assert e <= TOL, e
    if noisy:
        ref = O.lkd_w_noise(x, f, gr, th, varK, noise, "precon" if mode == 1 else "base", eta, mask, kernel=kernel)
        got = np.hstack((o[L.OUT_GRAD:L.OUT_GRAD + d], [o[L.OUT_DKERN]] if isinstance(kernel, tuple) else [],
                         [o[L.OUT_DVARK]]))
    else:
        ref = O.lkd_wo_noise(x, f, gr, th, "precon" if mode == 1 else "base", eta, mask, kernel=kernel)
        got = np.hstack((o[L.OUT_GRAD:L.OUT_GRAD + d], [o[L.OUT_DKERN]] if isinstance(kernel, tuple) else []))
        assert abs(o[L.OUT_SIGMA2] - ref.hp_varK) <= 1e-8 * ref.hp_varK
    assert abs(o[L.OUT_LML] - ref.ln_lkd) <= 1e-8 * abs(ref.ln_lkd)
    assert np.max(np.abs(got - ref.ln_lkd_grad)) <= 1e-8 * np.max(np.abs(ref.ln_lkd_grad))


@pytest.mark.parametrize("mode", [0, 1])
def test_direct_terms_vs_dense_reference(mode):
    """gegp_lml_direct_terms (quad 1 for a, a + h, a - h; quad 2 for K^-1) at a wide, masked Matern-5/2 problem, against
    contract() from the same evaluation's alpha, h = K^-1 H (the call's own, read back from its scratch) and K^-1."""
    from gpgradpy_b200 import _lib as L, backend as bk
    kernel, n, d = "Ma5f2", 130, 9
    x, f, gr, th, mask, y, noise, eta = _lml_case(kernel, n, d, "scatter", 50, True, mode, seed=5)
    slot, ng = _slot(mask, n)
    varK = 0.8
    _, alpha = bk.lml_eval(x, y, th[None, :], n_g=ng, slot=slot, mode=mode, eta=eta, noise=noise,
                           varK_batch=np.array([varK]), want_grad=True, want_alpha=True, kernel=kernel)
    v = bk.lml_views(n, ng, d)
    N = y.size
    Kinv = v["Kinv"][:, :N].cpu().numpy()
    pinv = v["pinv"].cpu().numpy()
    a = alpha.cpu().numpy()[0]
    lib = L.load()
    ol = L.out_len(d)
    out = torch.zeros(4 * ol + 2, dtype=torch.float64, device="cuda")
    scratch = torch.empty(4 * bk.ld_of(N), dtype=torch.float64, device="cuda")
    ws = bk._ws_cache[torch.cuda.current_device()]
    Xd, thd, vk = bk.to_dev(x), bk.to_dev(th), bk.to_dev(np.array([varK]))
    rc = lib.gegp_lml_direct_terms(n, ng, d, Xd.data_ptr(), slot.data_ptr(), thd.data_ptr(), 1, 0.0, mode, float(eta), 1,
                                   vk.data_ptr(), ws.data_ptr(), ws.numel(), scratch.data_ptr(), out.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    rows = out.cpu().numpy()[:4 * ol].reshape(4, ol)
    h = scratch[:N].cpu().numpy() * pinv
    slots = R.hp_slots(d, kernel, True)
    for row, w in zip(rows, (a, a + h, a - h, pinv[:, None] * Kinv * pinv[None, :])):
        g, sc = R.contract(x, th, w, mode, eta, mask, kernel, True, varK)
        e = R.contract_err(row, g, sc, slots)
        print(f"direct terms: {e:.2e}")
        assert e <= TOL, e


# ---------------------------------------------------------------------------------------------------------------------
# batch invariance on the wide non-Gaussian variants
# ---------------------------------------------------------------------------------------------------------------------
def test_quad_grad_batch_rows_are_bit_identical_to_single_calls():
    from gpgradpy_b200 import backend as bk
    n, d, ng = 140, 10, 60
    X, th0 = _problem(n, d, seed=21)
    mask = _mask("scatter", n, ng, 21)
    slot, ng = _slot(mask, n)
    N = n + ng * d
    rng = np.random.default_rng(22)
    B = 5
    th = th0[None, :] * rng.uniform(0.6, 1.6, (B, d))
    vk = rng.uniform(0.5, 2.0, B)
    al = rng.uniform(0.5, 3.0, B)
    V = torch.as_tensor(rng.standard_normal((B, N)), device="cuda")
    tab = bk.quad_grad_batch(X, th, V, n_g=ng, slot=slot, eta=1e-6, noisy=True, varK_rows=vk, kernel="RatQu",
                             kernel_hp_rows=al).cpu().numpy()
    for z in range(B):
        one = bk.quad_grad(X, th[z], V[z], n_g=ng, slot=slot, eta=1e-6, noisy=True, varK=vk[z],
                           kernel=("RatQu", al[z])).cpu().numpy()
        assert np.array_equal(one, tab[z])


def test_lml_eval_batch_rows_are_bit_identical_to_single_rows():
    from gpgradpy_b200 import backend as bk
    kernel, n, d = "Ma5f2", 130, 12
    x, f, gr, th0, mask, y, noise, eta = _lml_case(kernel, n, d, "scatter", 30, True, 1, seed=9)
    slot, ng = _slot(mask, n)
    rng = np.random.default_rng(10)
    B = 5
    th = th0[None, :] * rng.uniform(0.7, 1.4, (B, d))
    vk = rng.uniform(0.5, 2.0, B)
    tab = bk.lml_eval(x, y, th, n_g=ng, slot=slot, mode=1, eta=eta, noise=noise, varK_batch=vk, want_grad=True,
                      kernel=kernel)[0].cpu().numpy()
    for z in range(B):
        one = bk.lml_eval(x, y, th[z:z + 1], n_g=ng, slot=slot, mode=1, eta=eta, noise=noise, varK_batch=vk[z:z + 1],
                          want_grad=True, kernel=kernel)[0].cpu().numpy()
        assert np.array_equal(one[0], tab[z])
