"""`GaussianProcess`: host-side mirror of GpGradPy's GP class with the hot path on the B200.

Same constructor, option attributes, method names, argument meaning and return contracts as the reference
class (gpgradpy/src/GaussianProcess.py:24-457 and its mixins) for the Gaussian ("SqExp") kernel with a
constant mean, gradient-free or gradient-enhanced data and the base / rescaling / preconditioned modes.
Everything O(N^2) or O(N^3) is done by libgegp.so (hand-written sm_100a kernels behind include/gegp.h):

  calc_all_K_w_chofac   -> gegp_build_cov + gegp_potrf        (kernel/Kernel.py:140-307)
  calc_lkd_all          -> gegp_lml_eval                      (optz/CalcLkd.py:270-346)
  select_hp_optz_x0     -> gegp_lml_eval, B candidates, sharded across ranks (optz/GpHparaX0.py:16-65)
  setup_eval_model      -> gegp_predict_setup                 (eval/GpEvalModel.py:17-57)
  eval_model            -> gegp_predict                       (eval/GpEvalModel.py:59-198; mu and sigma)

Host Python keeps what the reference keeps in Python: log10 <-> theta transforms and the chain factor
(optz/OptzLkd.py:65-70), SLSQP (optz/OptzLkd.py:265), bounds and Latin-hypercube starts, nugget
formulas, rescaling, history arrays.  There is no CPU fallback for the device work.
"""
from __future__ import annotations

import copy
import time

import numpy as np
from scipy.optimize import Bounds, NonlinearConstraint, minimize
from scipy.stats import qmc

from . import _lib as L
from . import backend as bk
from . import hpara as H
from . import parallel
from .hpara import HparaOptzInfo, HparaOptzVal, LkdInfo
from .rescaling import Rescaling


class DeviceMatrix:
    """A matrix that lives on the GPU and turns into a NumPy array on demand (np.asarray / indexing).  `t` is a device
    tensor or a zero-argument callable that produces one: the callable runs on first access, so a matrix of the
    reference's 7-tuple that nobody reads is never built (at N = 21000 each one is 3.5 GB)."""

    def __init__(self, t, symmetrize_from_lower=False, shape=None):
        self._make = t if callable(t) else None
        self._t = None if callable(t) else t
        self._shape = shape
        self._sym, self._np = symmetrize_from_lower, None

    @property
    def tensor(self):
        if self._t is None:
            self._t, self._make = self._make(), None
        return self._t

    @property
    def shape(self):
        return tuple(self._shape) if self._t is None and self._shape is not None else tuple(self.tensor.shape)

    def numpy(self):
        if self._np is None:
            a = self.tensor.cpu().numpy().copy()
            self._np = a
        return self._np

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, idx):
        return self.numpy()[idx]


class GaussianProcess:
    use_cuda_graphs = True      # replay a captured CUDA graph for repeated noise-free evaluations (not in the reference)
    cond_warm_start = True      # start the Lanczos iterations of the condition number from the previous eigenvectors
    lockstep_multistart = True  # run the SLSQP instances of a multi-start fit in lock step, objective requests batched

    # ---- options (names and defaults of gpgradpy/src/GaussianProcess.py:27-113) ----
    print_txt_data = False
    save_data_npz = False
    save_data_txt = False

    optz_mtd = "SLSQP"
    optz_n_x0 = 5
    optz_iter_max = 250
    optz_tol_obj = 1e-12
    optz_tol_x = 1e-12
    optz_log_hp_theta = True
    optz_log_hp_var = True
    optz_log_hp_kernel = True

    lkd_use_adj_mtd = True
    lkd_optz_start_avail = ["hp_best", "lhs"]
    lkd_optz_start_mtd = "hp_best"
    lkd_hp_best_n_eval = 40
    lkd_varK_pnlt_use = False
    lkd_varK_pnlt_lb_var = 0.1
    lkd_varK_pnlt_c1 = 1.0
    lkd_varK_pnlt_c2 = 10.0

    hp_const_n_eval = 1
    hp_lhs_bound_factor = 1e3
    hp_box_bound_factor = 1e5
    hp_median_n_idx = 5
    hp_theta_init = 1e-2
    hp_varK_init = 1.0
    hp_kernel_init = np.nan
    hp_var_fval_init = 0.0
    hp_var_fgrad_init = 0.0
    hp_theta_range = [1e-18, 1e24]
    hp_varK_range = [1e-24, 1e14]
    hp_kernel_range = [np.nan, np.nan]
    hp_var_fval_range = [1e-8, 1e8]
    hp_var_fgrad_range = [1e-8, 1e8]

    wellcond_mtd_avail = ["base", "precon", "rescale_origin", "rescale_eta_vary", "dflt_vmin", "dflt_vmax"]
    cond_eta_set_mtd = "Kbase_eta"
    cond_eta_is_const = True
    cond_eta_dflt = 1e-8
    cond_max_target = 1e10
    cond_max = 1e10
    cond_max_abs = 1e16
    cond_norm = 2
    cond_dist_min_dflt = 1
    cond_dist_max_dflt = 1
    cond_vreq_max_iter = 3
    vmin_rescale_eta_vary = 1.0
    cond_vreq_iter_tol = 1e-1

    b_optz_hp_kernel = True
    b_use_data_scl = None
    b_has_noisy_data = None
    b_optz_var_fval = None
    b_optz_var_fgrad = None
    bvec_use_grad = None
    _vmin_req_grad = np.nan
    _time_chofac = 0
    _save_data = False
    _last_hp_vec = None
    hp_vals = None
    kernel_has_hp = False
    hp_kernel_default = None
    dist_group = None  # torch.distributed group used to shard candidate batches (None: default group / single rank)

    HparaOptzVal = HparaOptzVal
    HparaOptzInfo = HparaOptzInfo
    LkdInfo = LkdInfo

    def __init__(self, dim, use_grad, kernel_type="SqExp", wellcond_mtd="precon", mean_fun_type="poly_ord_0",
                 path_data_surr="baye_data_surr", surr_name="obj_"):
        assert isinstance(dim, int), "dim must be an integer"
        assert isinstance(use_grad, bool), "use_grad must be of type bool"
        assert isinstance(kernel_type, str), "kernel_type must be of type str"
        if kernel_type not in L.KERNEL_IDS:
            raise Exception("Kernel type is not available")                  # kernel/Kernel.py:105-107
        if mean_fun_type != "poly_ord_0":
            raise Exception(f"mean_fun_type = {mean_fun_type} not available")
        self.dim, self.use_grad, self.kernel_type = dim, use_grad, kernel_type
        self.mean_fun_type, self.n_beta_coeff, self.beta_var_npara = mean_fun_type, 1, 1
        self.set_wellcond_mtd(wellcond_mtd)
        self.path_data_surr, self.surr_name = path_data_surr, surr_name
        # kernel family (kernel/Kernel.py:27-113): extra hyper-parameter and its range per kernel file
        # (kernel/KernelSqExp.py:577-578, kernel/KernelMatern5f2.py:649-650: none; kernel/KernelRatQuad.py:849-850: alpha)
        self._kid = L.KERNEL_IDS[kernel_type]
        if kernel_type == "RatQu":
            self.hp_kernel_default, self.hp_kernel_range = 2, [1e-3, 10]
        else:
            self.hp_kernel_default, self.hp_kernel_range = None, [np.nan, np.nan]
        self.kernel_has_hp = self.hp_kernel_default is not None
        self.hp_kernel = self.hp_kernel_default
        self._diag_coef = 5.0 / 3.0 if kernel_type == "Ma5f2" else 2.0      # gamma_i^2 = c theta_i
        self.theta2gamma = lambda theta: np.sqrt(self._diag_coef * np.asarray(theta))
        self.gamma2theta = lambda gamma: np.asarray(gamma) ** 2 / self._diag_coef
        self.calc_Kern_precon = lambda n_eval, n_grad, theta, calc_grad=False, b_return_vec=False: \
            GaussianProcess.calc_Kern_precon(n_eval, n_grad, theta, calc_grad, b_return_vec, diag_coef=self._diag_coef)
        self._pred = None

    def _kern(self, hp_vals=None):
        """(GEGP_KERNEL_* id, kernel hyper-parameter) handed to every device call."""
        hp = self.hp_kernel_default if (hp_vals is None or hp_vals.kernel is None) else hp_vals.kernel
        return self._kid, (0.0 if hp is None else float(np.ravel(hp)[0]))

    # ------------------------------------------------------------------ configuration
    def set_wellcond_mtd(self, wellcond_mtd):
        """gpgradpy/src/GaussianProcess.py:192-217."""
        assert wellcond_mtd in self.wellcond_mtd_avail, f"Requested method not available, wellcond_mtd : {wellcond_mtd}"
        if wellcond_mtd == "rescale_eta_vary":
            self.cond_eta_is_const = False
        if not self.use_grad:
            wellcond_mtd = "base"
        self.wellcond_mtd = wellcond_mtd
        self.b_use_cond_cstr = wellcond_mtd != "precon"
        if self.b_use_cond_cstr:
            self.condnum_nlc = NonlinearConstraint(self.return_cond_val, -np.inf, self.cond_max,
                                                   jac=self.return_cond_grad)
        self.b_use_data_scl = ("rescale" in wellcond_mtd) or ("dflt_v" in wellcond_mtd)

    @property
    def _mode(self):
        return L.MODE_PRECON if self.wellcond_mtd == "precon" else L.MODE_BASE

    # ------------------------------------------------------------------ small kernel-level helpers kept for API parity
    @staticmethod
    def theta2gamma(theta):
        return np.sqrt(2 * np.asarray(theta))          # kernel/KernelSqExp.py:581-583

    @staticmethod
    def gamma2theta(gamma):
        return 0.5 * np.asarray(gamma) ** 2            # kernel/KernelSqExp.py:586-588

    @staticmethod
    def calc_Kern_precon(n_eval, n_grad, theta, calc_grad=False, b_return_vec=False, diag_coef=2.0):
        """Analytic preconditioner (kernel/KernelSqExp.py:591-605, kernel/KernelMatern5f2.py:665-680,
        kernel/KernelRatQuad.py:863-877 with kernel/KernelCommon.py:14-49): p = [1_n, gamma_i (x) 1_ng],
        gamma = sqrt(c theta) with c = 2 (Gaussian, rational quadratic) or 5/3 (Matern-5/2), d gamma_i / d theta_i =
        c / (2 gamma_i).  Host helper kept for API parity (the kernels form p themselves, csrc/build.cu prep_p_kernel);
        like the reference it always returns the derivative, as an [N, d] array or a stack of diagonal matrices.
        Called on the class it is the Gaussian kernel's; instances bind their own kernel's coefficient."""
        theta = np.asarray(theta, dtype=float)
        gamma = np.sqrt(diag_coef * theta)
        pvec = np.hstack((np.ones(n_eval), np.kron(gamma, np.ones(n_grad))))
        dim, n_data = theta.size, n_eval + n_grad * theta.size
        dgam = diag_coef / (2 * gamma)
        if b_return_vec:
            grad = np.zeros((n_data, dim))
            for i in range(dim):
                grad[n_eval + i * n_grad: n_eval + (i + 1) * n_grad, i] = dgam[i]
            return pvec, 1 / pvec, grad
        grad = np.zeros((dim, n_data, n_data))
        for i in range(dim):
            v = np.zeros(n_data)
            v[n_eval + i * n_grad: n_eval + (i + 1) * n_grad] = dgam[i]
            grad[i] = np.diag(v)
        return np.diag(pvec), np.diag(1 / pvec), grad

    @staticmethod
    def make_data_vec(fval, fgrad=None):
        """base/CommonFun.py:152-173."""
        if fgrad is None:
            return np.atleast_1d(fval)
        return np.hstack((fval, fgrad.reshape(fgrad.size, order="F")))

    def calc_nugget_Kbase(self, n_eval, cond_max=None):
        return H.nugget_Kbase(n_eval, self.cond_max_target if cond_max is None else cond_max)

    def calc_mtd_rescale_origin_vreq(self, n_eval, dim=None):
        return H.vreq_rescale_origin(n_eval, self.dim if dim is None else dim)

    def calc_nugget_Kfull_vreq(self, n_eval, vmin=None):
        return H.nugget_Kfull_vreq(n_eval, self.dim, self.cond_max_target, vmin)

    def calc_nugget(self, n_eval):
        """(eta_Kbase, eta_Kgrad) -- base/GpWellCond.py:116-154."""
        if self.cond_eta_set_mtd == "dflt_eta":
            return self.cond_eta_dflt, self.cond_eta_dflt
        eta_Kbase = self.calc_nugget_Kbase(n_eval)
        if not self.use_grad:
            return eta_Kbase, np.nan
        if n_eval == 1:
            return eta_Kbase, eta_Kbase
        if self.wellcond_mtd == "precon":
            if self.kernel_type == "Ma5f2":
                return eta_Kbase, H.nugget_precon_matern52(n_eval, self.dim, self.cond_max_target)
            return eta_Kbase, H.nugget_precon_sqexp(n_eval, self.dim, self.cond_max_target)   # SqExp and RatQu share it
        if "rescale" in self.wellcond_mtd:
            return eta_Kbase, self.calc_nugget_Kfull_vreq(n_eval)
        if self.cond_eta_set_mtd == "Kbase_eta":
            return eta_Kbase, eta_Kbase
        if self.cond_eta_set_mtd == "Kbase_eta_w_dim":
            return eta_Kbase, eta_Kbase * (self.dim + 1)
        raise Exception(f"Uknown method for cond_eta_set_mtd = {self.cond_eta_set_mtd}")

    # ------------------------------------------------------------------ hyper-parameter plumbing (base/GpHpara.py)
    def make_hp_class(self, beta=None, theta=None, kernel=None, varK=None, var_fval=None, var_fgrad=None):
        return HparaOptzVal(beta, theta, kernel, varK, var_fval, var_fgrad)

    def set_custom_hp(self, beta=None, theta=None, kernel=None, varK=None, var_fval=None, var_fgrad=None):
        if varK is not None:
            assert varK > 0, f"varK must be positive but it is {varK}"
        self.hp_vals = self.make_hp_class(beta, theta, kernel, varK, var_fval, var_fgrad)

    def hp_vec2dataclass(self, hp_optz_info, hp_vec):
        """base/GpHpara.py:56-103 (10** for the log-optimised entries)."""
        v = np.array(hp_vec, dtype=float, copy=True)
        b = hp_optz_info.bvec_log_optz
        v[b] = 10 ** v[b]
        theta = v[hp_optz_info.idx_theta] if hp_optz_info.has_theta else None
        kernel = float(v[hp_optz_info.idx_kernel][0]) if hp_optz_info.has_kernel else None
        varK = float(v[hp_optz_info.idx_varK]) if hp_optz_info.has_varK else None
        var_fval = float(v[hp_optz_info.idx_var_fval]) if hp_optz_info.has_var_fval else None
        var_fgrad = float(v[hp_optz_info.idx_var_fgrad]) if hp_optz_info.has_var_fgrad else None
        return self.make_hp_class(None, theta, kernel, varK, var_fval, var_fgrad)

    def set_hp_optz_info(self, has_theta, has_kernel=False, has_varK=False, has_var_fval=False, has_var_fgrad=False):
        """optz/GpHparaOptz.py:44-138."""
        n_hp = has_theta * self.dim + has_kernel + has_varK + has_var_fval + has_var_fgrad
        blog = np.zeros(n_hp, dtype=bool)
        cnt = 0
        empty = np.array([], dtype=int)
        idx_theta = empty
        if has_theta:
            idx_theta = np.arange(cnt, cnt + self.dim, dtype=int)
            cnt += self.dim
            blog[idx_theta] = self.optz_log_hp_theta
        idx_kernel = empty
        if has_kernel:
            assert self.kernel_has_hp, "Kernel must have hyperaparamters if b_optz_hp_kernel is set to True"
            idx_kernel = np.array([cnt])
            cnt += 1
            blog[idx_kernel] = self.optz_log_hp_kernel
        idx_varK = idx_vf = idx_vg = empty
        if has_varK:
            idx_varK, cnt = cnt, cnt + 1
            blog[idx_varK] = self.optz_log_hp_var
        if has_var_fval:
            idx_vf, cnt = cnt, cnt + 1
            blog[idx_vf] = self.optz_log_hp_var
        if has_var_fgrad:
            idx_vg, cnt = cnt, cnt + 1
            blog[idx_vg] = self.optz_log_hp_var
        return HparaOptzInfo(n_hp=n_hp, has_theta=has_theta, idx_theta=idx_theta, has_kernel=bool(has_kernel),
                             idx_kernel=idx_kernel,
                             has_varK=has_varK, idx_varK=idx_varK, has_var_fval=has_var_fval, idx_var_fval=idx_vf,
                             has_var_fgrad=has_var_fgrad, idx_var_fgrad=idx_vg, bvec_log_optz=blog)

    def setup_hp_idx4optz(self):
        self.hp_info_optz_lkd = self.set_hp_optz_info(True, self.b_optz_hp_kernel and self.kernel_has_hp,
                                                      self.b_has_noisy_data, self.b_optz_var_fval, self.b_optz_var_fgrad)

    # ------------------------------------------------------------------ data
    def set_data(self, x_eval, fval, std_fval, grad=None, std_grad=None, bvec_use_grad=None):
        """gpgradpy/src/GaussianProcess.py:219-363 (validation, noise flags, nugget, scaling, device upload)."""
        x_eval = np.asarray(x_eval, dtype=float)
        fval = np.atleast_1d(np.asarray(fval, dtype=float)).ravel()
        n_eval = fval.size
        if self.use_grad:
            if bvec_use_grad is None:
                n_grad = n_eval
            else:
                bvec_use_grad = np.asarray(bvec_use_grad, dtype=bool)
                n_grad = int(np.sum(bvec_use_grad))
                assert bvec_use_grad.size == n_eval, \
                    f"Length of bvec_use_grad is {bvec_use_grad.size} but it should be n_eval = {n_eval}"
                assert grad.shape[0] == n_grad, f"No. of rows of grad is {grad.shape[0]} but it should be n_grad = {n_grad}"
        else:
            assert bvec_use_grad is None, "bvec_use_grad must be None if grads are not used for the GP"
            n_grad = 0
        self.n_eval, self.n_grad, self.n_data = n_eval, n_grad, n_eval + n_grad * self.dim
        assert x_eval.ndim == 2, f"x_eval must be a 2 array but x_eval.ndim = {x_eval.ndim}"
        assert x_eval.shape == (n_eval, self.dim), "No. of points do not match with x_eval and fval"

        if (std_fval is None) or np.any(np.isnan(std_fval)):
            self.known_eps_fval = False
        else:
            self.known_eps_fval = True
            std_fval = np.atleast_1d(np.asarray(std_fval, dtype=float)).ravel()
            assert n_eval == std_fval.size, f"Size of std_fval is {std_fval.size} while it should be {n_eval}"
        if grad is None:
            assert self.use_grad is False, "No grad info provided but use_grad was set to True"
            self.has_grad_info, self.known_eps_fgrad = False, False
        else:
            assert self.use_grad, "Grad info provided but use_grad was set to False"
            grad = np.asarray(grad, dtype=float)
            self.has_grad_info = True
            assert grad.ndim == 2 and grad.shape == (n_grad, self.dim), "Shape of grad does not match x_eval"
            if (std_grad is None) or np.any(np.isnan(std_grad)):
                self.known_eps_fgrad = False
            else:
                std_grad = np.asarray(std_grad, dtype=float)
                self.known_eps_fgrad = True
                assert grad.shape == std_grad.shape, "Shape of grad does not match std_grad"

        self._x_eval_in, self._fval_in, self._grad_in = x_eval, fval, grad
        self._std_fval_in = std_fval if self.known_eps_fval else None
        self._std_grad_in = std_grad if self.known_eps_fgrad else None
        self.bvec_use_grad = bvec_use_grad

        if self.known_eps_fval:
            self.b_optz_var_fval, self.b_fval_zero = False, bool(np.max(std_fval) < 1e-10)
        else:
            self.b_optz_var_fval, self.b_fval_zero = True, False
        if self.use_grad is False:
            self.b_optz_var_fgrad, self.b_fgrad_zero = False, True
        elif self.known_eps_fgrad:
            self.b_optz_var_fgrad, self.b_fgrad_zero = False, bool(np.max(std_grad) < 1e-10)
        else:
            self.b_optz_var_fgrad, self.b_fgrad_zero = True, False
        self.b_has_noisy_data = not (self.b_fval_zero and self.b_fgrad_zero)

        self._eta_Kbase, self._eta_Kgrad = self.calc_nugget(n_eval)
        self._etaK = self._eta_Kgrad if self.use_grad else self._eta_Kbase
        self._vmin_init = np.nan if n_eval == 1 else float(np.min(_pdist(x_eval)))
        self.setup_hp_idx4optz()

        if self.b_use_data_scl:
            if self.wellcond_mtd == "rescale_origin":
                dist_set = self.calc_mtd_rescale_origin_vreq(n_eval, self.dim)
                self._vmin_req_grad, mtd = dist_set, "set_vmin"
            elif self.wellcond_mtd == "rescale_eta_vary":
                dist_set, mtd = self.vmin_rescale_eta_vary, "set_vmin"
            elif self.wellcond_mtd == "dflt_vmin":
                dist_set, mtd = self.cond_dist_min_dflt, "set_vmin"
            elif self.wellcond_mtd == "dflt_vmax":
                dist_set, mtd = self.cond_dist_max_dflt, "set_vmax"
            else:
                raise Exception(f"Unknown method wellcond_mtd = {self.wellcond_mtd}")
            self.DataScl = Rescaling(x_eval, x_scl_method=mtd, dist_set=dist_set)
            self.DataScl.set_obj_data(fval, std_fval, grad, std_grad)
            self.Rtensor_init = None
        else:
            # the reference caches the [d, n, n] distance tensor here (GaussianProcess.py:363) and scripts pass it back
            # into calc_all_K_w_chofac (plt/plt_nugget_1d.py:174-175); the CUDA builder reads X directly, so a
            # placeholder stands in for it (accepted and ignored wherever an Rtensor argument is taken)
            self.Rtensor_init = _DeviceRtensor(n_eval, self.dim)
        self._dev_ready = False
        self._pred = None
        self.KernEta_chofac = None        # a model set up for the previous data cannot be evaluated any more
        self.invKernEta_fdiff = None
        self._last_hp_vec = None
        self._last_cond = None

    def _ensure_device(self):
        """Put the (scaled) training data on the device (lazily): X[n,d], y[N], gradient-slot map."""
        if getattr(self, "_dev_ready", False):
            return
        x_scl = self.get_scl_x_w_dist()[0]
        fval, _, grad, _ = self.get_scl_eval_data()
        self._slot_dev, ng = bk.slot_from_mask(self.bvec_use_grad if self.use_grad else np.zeros(self.n_eval, bool),
                                               self.n_eval)
        assert ng == self.n_grad
        self._y_host = self.make_data_vec(fval, grad if self.use_grad else None)
        # host -> device through pinned staging buffers (kept, so a refresh re-uses them)
        self._x_pin = bk.pinned_like(getattr(self, "_x_pin", None), x_scl)
        self._y_pin = bk.pinned_like(getattr(self, "_y_pin", None), self._y_host)
        # device buffers are kept while the shapes stay the same, so captured CUDA graphs remain valid after a refresh
        if getattr(self, "_X_dev", None) is not None and tuple(self._X_dev.shape) == tuple(self._x_pin.shape) \
                and tuple(self._y_dev.shape) == tuple(self._y_pin.shape):
            self._X_dev.copy_(self._x_pin, non_blocking=True)
            self._y_dev.copy_(self._y_pin, non_blocking=True)
        else:
            self._X_dev = self._x_pin.to(bk.device(), non_blocking=True)
            self._y_dev = self._y_pin.to(bk.device(), non_blocking=True)
        self._dev_ready = True

    # ---- scaled / unscaled accessors (GaussianProcess.py:399-457)
    def get_scl_x_w_dist(self):
        """(x_scl, Rtensor).  The CUDA builder reads X directly, so no [d,n,n] distance tensor is kept: Rtensor is None."""
        if self.b_use_data_scl:
            return self.DataScl.get_scl_x_w_dist()
        return self._x_eval_in, None

    def x_init_2_scl(self, x):
        return self.DataScl.x_init_2_scl(x) if self.b_use_data_scl else x

    def x_scl_2_init(self, x):
        return self.DataScl.x_scl_2_init(x) if self.b_use_data_scl else x

    def get_init_eval_data(self):
        return self._fval_in, self._std_fval_in, self._grad_in, self._std_grad_in

    def get_scl_eval_data(self):
        f, sf, g, sg = self.data_init_2_scl(*self.get_init_eval_data())[:4]
        return f, (sf if self.known_eps_fval else None), g, (sg if self.known_eps_fgrad else None)

    def data_init_2_scl(self, *a):
        a = tuple(a) + (None,) * (6 - len(a))
        return self.DataScl.obj_init_2_scl(*a) if self.b_use_data_scl else a

    def data_scl_2_init(self, *a):
        a = tuple(a) + (None,) * (6 - len(a))
        return self.DataScl.obj_scl_2_init(*a) if self.b_use_data_scl else a

    # ------------------------------------------------------------------ noise
    def calc_noise_vec(self, hp_vals):
        """kernel/Kernel.py:309-357."""
        if self.b_fval_zero and self.b_fgrad_zero:
            std_fval, std_fgrad = np.zeros(self.n_eval), np.zeros((self.n_grad, self.dim))
        else:
            std_fval, _, std_fgrad = self.get_scl_eval_data()[1:]
        if not self.use_grad:
            return std_fval ** 2 if self.known_eps_fval else np.full(self.n_eval, hp_vals.var_fval)
        v = np.zeros(self.n_data)
        v[: self.n_eval] = std_fval ** 2 if self.known_eps_fval else hp_vals.var_fval
        v[self.n_eval:] = (std_fgrad ** 2).reshape(std_fgrad.size, order="F") if self.known_eps_fgrad else hp_vals.var_fgrad
        return v

    # ------------------------------------------------------------------ covariance assembly + factorisation
    def calc_Kern_w_chofac(self, Rtensor, hp_vals, noise_vec=None, calc_chofac=True, calc_cond=False):
        assert self.b_has_noisy_data is False, "This function should not be called if there is noisy data"
        return self.calc_all_K_w_chofac(Rtensor, hp_vals, noise_vec, calc_chofac, calc_cond, varK=1)

    def calc_all_K_w_chofac(self, Rtensor, hp_vals, noise_vec=None, calc_chofac=True, calc_cond=False, varK=None,
                            b_normlz_w_varK=False):
        """Same 7-tuple as kernel/Kernel.py:140-307; the matrices are device-resident DeviceMatrix objects that
        convert to NumPy on demand.  `Rtensor` is accepted for signature compatibility and ignored."""
        import torch
        self._ensure_device()
        theta = np.asarray(hp_vals.theta, dtype=float)
        if varK is None:
            assert hp_vals.varK is not None, f"varK is not provided and hp_vals.varK is None, hp_vals = {hp_vals}"
            varK = hp_vals.varK
        if b_normlz_w_varK:
            varK = 1.0
        else:
            assert varK > 0, f"varK must be positive but varK = {varK}"
        assert np.sum(np.isnan(theta)) == 0, f"There are nan values theta = {theta}"
        if noise_vec is None:
            noise_vec = self.calc_noise_vec(hp_vals)
        noise = None if not np.any(noise_vec) else bk.to_dev(np.asarray(noise_vec, dtype=float) / varK)
        X, slot, ng, N = self._X_dev, self._slot_dev, self.n_grad, self.n_data
        kw = dict(n_g=ng, slot=slot, kernel=self._kern(hp_vals))
        # Only the matrix that is factored / whose condition number is asked for is built here; the other members of
        # the tuple are built by the same kernel when (if) they are read.
        Kern = DeviceMatrix(lambda: bk.build_cov(X, theta, mode=L.MODE_BASE, eta=0.0, **kw)[0], shape=(N, N))
        idx_etaK_argmax = None
        precon = self.wellcond_mtd == "precon"
        if precon:
            assert self.use_grad is True, "self.wellcond_mtd should be base if use_grad is False"
        if self.cond_eta_is_const:
            etaK = self._etaK
        else:
            etaK, idx_etaK_argmax = self._variable_eta(theta, noise, None if precon else Kern.tensor,
                                                       kernel=self._kern(hp_vals))
        fac_src = pvec = None
        need_fac = calc_chofac or calc_cond
        if precon:
            if need_fac:
                fac_src, p = bk.build_cov(X, theta, noise=noise, mode=L.MODE_PRECON, eta=etaK, varK=varK, **kw)
                pvec = p[:N]

            def make_kcor(Kt=fac_src):
                if Kt is None:
                    Kt = bk.build_cov(X, theta, noise=noise, mode=L.MODE_PRECON, eta=etaK, varK=varK, **kw)[0]
                out = Kt / varK
                out.diagonal().sub_(etaK)
                return out
            Kcor = DeviceMatrix(make_kcor, shape=(N, N))
            Kcov = DeviceMatrix(lambda: bk.build_cov(X, theta, noise=noise, mode=L.MODE_PRECON_COV, eta=etaK, varK=varK,
                                                     **kw)[0], shape=(N, N))
        else:
            if need_fac:
                fac_src = bk.build_cov(X, theta, noise=noise, mode=L.MODE_BASE, eta=etaK, varK=varK, **kw)[0]
                Kcov = DeviceMatrix(fac_src)
            else:
                Kcov = DeviceMatrix(lambda: bk.build_cov(X, theta, noise=noise, mode=L.MODE_BASE, eta=etaK, varK=varK,
                                                         **kw)[0], shape=(N, N))
            Kcor = None
        condK = None
        if calc_cond:   # condition number of the matrix that is factored (kernel/Kernel.py:240,280)
            if self.cond_norm == 2:       # device Lanczos
                self._last_cond = bk.cond2_of_matrix(fac_src, N)
                condK = float(self._last_cond["cond"])
            elif self.cond_norm == "fro":
                condK = bk.cond_fro_of_matrix(fac_src, N)
            else:
                raise Exception(f'cond_norm must be either 2 or "fro" but it is {self.cond_norm}')
            if (not precon) and condK > self.cond_max_abs:
                calc_chofac = False
        Kcov_chofac = None
        t0 = time.time()
        if calc_chofac:
            ld = bk.ld_of(N)
            A = torch.empty((N, ld), dtype=fac_src.dtype, device=fac_src.device)
            A[:, :N] = fac_src
            info, _dinv = bk.potrf(A, N, 0)
            if int(info.item()) == 0:
                # the factor in the reference's convention, produced from the device factor when it is read
                if precon:
                    Kcov_chofac = (DeviceMatrix(lambda: torch.tril(A[:, :N]).mul_(pvec[:, None]), shape=(N, N)),
                                   True)                                          # (P @ L, lower=True)  :252
                else:
                    Kcov_chofac = (DeviceMatrix(lambda: torch.tril(A[:, :N]).T.contiguous(), shape=(N, N)),
                                   False)                                         # scipy default: upper     :291
        self._time_chofac += time.time() - t0
        return Kern, Kcor, Kcov, Kcov_chofac, condK, etaK, idx_etaK_argmax

    def _variable_eta(self, theta, noise_div, Kern=None, kernel=None):
        """Variable nugget from the Gershgorin row sums of Kcor (precon) or of the noise-free Kern (otherwise):
        eta = max_row sum|.| / (cond_max_target - 1)  (kernel/Kernel.py:229-234, 269-274) -> (eta, argmax row)."""
        self._ensure_device()
        kw = dict(n_g=self.n_grad, slot=self._slot_dev, kernel=kernel if kernel is not None else self._kern())
        if self.wellcond_mtd == "precon":
            M = bk.build_cov(self._X_dev, theta, noise=noise_div, mode=L.MODE_PRECON, eta=0.0, **kw)[0]
        else:
            M = Kern if Kern is not None else bk.build_cov(self._X_dev, theta, mode=L.MODE_BASE, eta=0.0, **kw)[0]
        rs = bk.row_abs_sum(M, self.n_data).cpu().numpy()
        idx = int(np.argmax(rs))
        return float(rs[idx]) / (self.cond_max_target - 1), idx

    def _eta_for(self, hp_vals):
        """The nugget the likelihood uses at these hyper-parameters (constant, or Gershgorin-based)."""
        if self.cond_eta_is_const:
            return self._etaK
        theta, noise_div, _ = self._cond_matrix_args(hp_vals)
        return self._variable_eta(theta, noise_div, kernel=self._kern(hp_vals))[0]

    # ------------------------------------------------------------------ likelihood
    def calc_lkd_varK_pnlt(self, varK, fval_vec):
        """optz/CalcLkd.py:118-133."""
        if not self.lkd_varK_pnlt_use:
            return 0, 0
        var_fval = max(np.var(fval_vec), self.lkd_varK_pnlt_lb_var)
        mx = max(varK - self.lkd_varK_pnlt_c2 * var_fval, 0)
        return self.lkd_varK_pnlt_c1 * var_fval * mx ** 2, 2 * self.lkd_varK_pnlt_c1 * var_fval * mx

    def _eval_rows(self, theta_rows, *, want_grad, varK_rows=None, noise_vec=None, pnlt_grad=0.0, eta=None,
                   khp_rows=None):
        """Device evaluation of B candidate rows -> torch [B, 9+d] (see GEGP_OUT_* in include/gegp.h).

        Noise-free evaluations of a fixed data set replay a captured CUDA graph (the optimiser repeats the same-shaped
        evaluation hundreds of times); everything else goes through the plain stream path."""
        self._ensure_device()
        kw = dict(n_g=self.n_grad, slot=self._slot_dev, mode=self._mode, eta=self._etaK if eta is None else eta,
                  pnlt_grad=pnlt_grad, want_grad=want_grad, kernel=self._kern())
        if self.kernel_has_hp:        # one kernel hyper-parameter per candidate row (default: the kernel's default value)
            nrow = int(np.prod(tuple(theta_rows.shape))) // self.dim
            kw["kernel_hp_batch"] = (np.full(nrow, float(self.hp_kernel_default)) if khp_rows is None
                                     else np.asarray(khp_rows, dtype=float).reshape(-1))
        single = int(np.prod(tuple(theta_rows.shape))) == self.dim   # one candidate: the optimiser's inner loop
        if self.use_cuda_graphs and single and noise_vec is None and pnlt_grad == 0.0 and eta is None:
            th = theta_rows if hasattr(theta_rows, "is_cuda") else np.asarray(theta_rows, dtype=float)
            return bk.lml_eval_graphed(self._X_dev, self._y_dev, th, **kw)
        out, _ = bk.lml_eval(self._X_dev, self._y_dev, theta_rows, noise=noise_vec, varK_batch=varK_rows, **kw)
        return out

    def _direct_form(self, hp_vals, info, varK_scale, pn_grad=0.0):
        """lkd_use_adj_mtd = False (optz/CalcLkd.py:64-85 noise-free, :238-241 noisy): fill hp_beta_grad, hp_varK_grad,
        ln_det_Kmat_grad and the direct-form ln_lkd_grad from three on-the-fly contractions over dKcov/dhp
        (gegp_lml_direct_terms) of the evaluation that has just run."""
        noisy = self.b_has_noisy_data
        t = bk.lml_direct_terms(self._X_dev, np.asarray(hp_vals.theta, dtype=float), n_g=self.n_grad, slot=self._slot_dev,
                                mode=self._mode, eta=getattr(self, "_eta_used", self._etaK), noisy=noisy,
                                varK=float(hp_vals.varK) if noisy else 1.0, kernel=self._kern(hp_vals))
        aDa, hDa, tr = (self._hp_row_to_grad(t[k]) for k in ("aDa", "hDa", "trKinvD"))
        N = self.n_data
        beta_grad = -hDa / t["HKH"]                              # eval/GpMeanFun.py:110-117 (term2 = -alpha)
        info.hp_beta_grad = beta_grad[None, :]
        info.ln_det_Kmat_grad = tr                               # optz/CalcLkd.py:349-367
        if noisy:                                                # optz/CalcLkd.py:253-265
            info.ln_lkd_grad = -0.5 * tr + 0.5 * aDa + t["Ha"] * beta_grad
        else:                                                    # optz/CalcLkd.py:104-116, 135-147
            varK_grad = (-2.0 * t["Ha"] * beta_grad - aDa) / N
            info.hp_varK_grad = varK_grad
            info.ln_lkd_grad = -0.5 * (N * varK_grad / varK_scale + tr) - pn_grad * varK_grad
        return info

    def calc_lkd_all(self, hp_vals, calc_lkd=True, calc_cond=False, calc_grad=False, lkd_use_adj_mtd=None):
        """(LkdInfo, b_chofac_good) -- optz/CalcLkd.py:270-346.  lkd_use_adj_mtd (default: the class option, True) picks
        the adjoint form (:149-181) or the direct one (:135-147), which also returns hp_beta_grad, hp_varK_grad and
        ln_det_Kmat_grad; the two gradients agree to rounding.

        With calc_cond the 2-norm condition number of the factored matrix (and, outside precon mode, its
        hyper-parameter gradient, optz/GpHparaCon.py:161-235) is computed on the device from the factor and the
        explicit inverse this very evaluation leaves in the workspace."""
        theta = np.asarray(hp_vals.theta, dtype=float)
        d = self.dim
        need_inv = calc_grad or calc_cond      # the condition number iterates with the explicit inverse
        # variable nugget (rescale_eta_vary): eta follows the matrix; like the reference, its theta-dependence is not
        # differentiated (optz/GpHparaGrad.py:40-50 uses the constant _etaK, and only in precon mode)
        eta = None if self.cond_eta_is_const else self._eta_for(hp_vals)
        self._eta_used = self._etaK if eta is None else eta
        hi = self.hp_info_optz_lkd
        use_adj = self.lkd_use_adj_mtd if lkd_use_adj_mtd is None else lkd_use_adj_mtd
        khp = np.array([self._kern(hp_vals)[1]]) if self.kernel_has_hp else None
        if self.b_has_noisy_data:
            noise = self.calc_noise_vec(hp_vals)
            o = self._eval_rows(theta[None, :], want_grad=need_inv, varK_rows=np.array([hp_vals.varK]),
                                noise_vec=noise, eta=eta, khp_rows=khp).cpu().numpy()[0]
            if o[L.OUT_INFO] != 0:
                cond, cond_grad = self._cond_on_failure(hp_vals, calc_grad)
                return LkdInfo(cond=cond, cond_grad=cond_grad), False
            info = LkdInfo(hp_beta=np.array([o[L.OUT_BETA]]), ln_det_Kmat=o[L.OUT_LOGDET], ln_lkd=o[L.OUT_LML],
                           data_vec=self._y_host)
            if calc_grad:
                g = np.zeros(hi.n_hp)
                g[hi.idx_theta] = o[L.OUT_GRAD:L.OUT_GRAD + d]
                if hi.has_kernel:
                    g[hi.idx_kernel] = o[L.OUT_DKERN]
                if hi.has_varK:
                    g[hi.idx_varK] = o[L.OUT_DVARK]
                if hi.has_var_fval:
                    g[hi.idx_var_fval] = o[L.OUT_DVARF]
                if hi.has_var_fgrad:
                    g[hi.idx_var_fgrad] = o[L.OUT_DVARG]
                info.ln_lkd_grad = g
                if not use_adj:
                    info = self._direct_form(hp_vals, info, float(hp_vals.varK))
            if calc_cond:
                info.cond, info.cond_grad = self._cond_from_workspace(hp_vals, calc_grad)
                if self.wellcond_mtd != "precon" and info.cond > self.cond_max_abs:
                    return LkdInfo(cond=info.cond, cond_grad=info.cond_grad), False      # kernel/Kernel.py:282-283
            return info, True
        pn_val = pn_grad = 0.0
        if self.lkd_varK_pnlt_use:   # the penalty slope depends on sigma^2: one value-only pass first
            o0 = self._eval_rows(theta[None, :], want_grad=False, eta=eta, khp_rows=khp).cpu().numpy()[0]
            pn_val, pn_grad = self.calc_lkd_varK_pnlt(o0[L.OUT_SIGMA2], self.get_scl_eval_data()[0])
        o = self._eval_rows(theta[None, :], want_grad=need_inv, pnlt_grad=pn_grad, eta=eta, khp_rows=khp).cpu().numpy()[0]
        if o[L.OUT_INFO] != 0:
            cond, cond_grad = self._cond_on_failure(hp_vals, calc_grad)
            return LkdInfo(cond=cond, cond_grad=cond_grad), False
        info = LkdInfo(hp_beta=np.array([o[L.OUT_BETA]]), hp_varK=o[L.OUT_SIGMA2], ln_det_Kmat=o[L.OUT_LOGDET])
        if calc_lkd:
            info.ln_lkd = o[L.OUT_LML] - pn_val
            if calc_grad:       # hyper-parameter order of the optimiser: theta_1..d, then the kernel's own (RatQu alpha)
                g = np.zeros(hi.n_hp)
                g[hi.idx_theta] = o[L.OUT_GRAD:L.OUT_GRAD + d]
                if hi.has_kernel:
                    g[hi.idx_kernel] = o[L.OUT_DKERN]
                info.ln_lkd_grad = g
                if not use_adj:
                    info = self._direct_form(hp_vals, info, float(o[L.OUT_SIGMA2]), pn_grad)
        if calc_cond:
            info.cond, info.cond_grad = self._cond_from_workspace(hp_vals, calc_grad)
            if self.wellcond_mtd != "precon" and info.cond > self.cond_max_abs:
                # the reference does not attempt the factorisation then (kernel/Kernel.py:282-283): no likelihood
                return LkdInfo(cond=info.cond, cond_grad=info.cond_grad), False
        return info, True

    # ------------------------------------------------------------------ condition number (optz/GpHparaCon.py:139-235)
    def _cond_matrix_args(self, hp_vals):
        """(theta, noise / varK or None, varK) of the matrix the likelihood factors (kernel/Kernel.py:128-138,213-237)."""
        theta = np.asarray(hp_vals.theta, dtype=float)
        if self.b_has_noisy_data:
            varK = float(hp_vals.varK)
            nv = self.calc_noise_vec(hp_vals)
            return theta, (bk.to_dev(nv / varK) if np.any(nv) else None), varK
        return theta, None, 1.0

    def _cond_grad_from_vectors(self, hp_vals, res, varK):
        """dkappa/dhp = (v_max^T dKcov v_max - kappa v_min^T dKcov v_min) / max(lambda_min, 1e-16)
        (optz/GpHparaCon.py:178-193), the quadratic forms evaluated with dKcov/dhp generated on the fly."""
        return self._cond_grads([hp_vals], [res], [varK])[0]

    def _cond_grads(self, hp_list, res_list, varK_list):
        """_cond_grad_from_vectors for many rows: the 2 quadratic forms of every row in one gegp_quad_grad_batch call."""
        if self.wellcond_mtd == "precon":
            return [None] * len(hp_list)   # the reference has no condition-number gradient in precon mode (:171-173)
        out = [np.zeros(self.hp_info_optz_lkd.n_hp) for _ in hp_list]
        live = [i for i, r in enumerate(res_list) if r.get("v_max") is not None]
        if not live:
            return out
        import torch
        th = np.vstack([np.asarray(hp_list[i].theta, dtype=float) for i in live])
        V = torch.stack([res_list[i]["v_max"] for i in live] + [res_list[i]["v_min"] for i in live])
        vk = np.array([float(varK_list[i]) for i in live])
        khp = np.array([self._kern(hp_list[i])[1] for i in live])
        q = bk.quad_grad_batch(self._X_dev, np.vstack([th, th]), V, n_g=self.n_grad, slot=self._slot_dev,
                               eta=getattr(self, "_eta_used", self._etaK), noisy=self.b_has_noisy_data,
                               varK_rows=np.hstack([vk, vk]), kernel=self._kern(), kernel_hp_rows=np.hstack([khp, khp])
                               ).cpu().numpy()
        for k, i in enumerate(live):
            r = res_list[i]
            out[i] = self._hp_row_to_grad((q[k] - r["cond"] * q[len(live) + k]) / max(r["lam_min"], 1e-16))
        return out

    def _hp_row_to_grad(self, q):
        """GEGP_OUT_* row of per-hyper-parameter sums -> vector in the optimiser's hyper-parameter order."""
        hi, d = self.hp_info_optz_lkd, self.dim
        g = np.zeros(hi.n_hp)
        if hi.has_theta:
            g[hi.idx_theta] = q[L.OUT_GRAD:L.OUT_GRAD + d]
        if hi.has_kernel:
            g[hi.idx_kernel] = q[L.OUT_DKERN]
        if self.b_has_noisy_data:
            if hi.has_varK:
                g[hi.idx_varK] = q[L.OUT_DVARK]
            if hi.has_var_fval:
                g[hi.idx_var_fval] = q[L.OUT_DVARF]
            if hi.has_var_fgrad:
                g[hi.idx_var_fgrad] = q[L.OUT_DVARG]
        return g

    def _rebuild_in_workspace(self, hp_list, calc_grad):
        """Views of the len(hp_list) candidates whose factor, L^-T and explicit inverse the likelihood evaluation that
        has just run left in the workspace, with each candidate's matrix rebuilt into its (no longer needed) L^-T buffer
        for the lambda_max products (lambda_min comes from products with the inverse).  Every row shares the noise
        vector of hp_list[0]."""
        B, N, mode = len(hp_list), self.n_data, self._mode
        v = bk.lml_views_batch(self.n_eval, self.n_grad, self.dim, B)
        if self.wellcond_mtd == "precon" and calc_grad:
            # reference quirk (optz/CalcLkd.py:341-343): with calc_grad the number returned in precon mode is kappa of
            # the UN-preconditioned Kcov = P Kt P, whose inverse is P^-1 Kt^-1 P^-1
            mode = L.MODE_PRECON_COV
            v["Kinv"][:, :, :N].mul_(v["pinv"][:, :, None]).mul_(v["pinv"][:, None, :])
        noise = varK = None
        if self.b_has_noisy_data:      # the device divides the noise by each row's varK (kernel/Kernel.py:218)
            nv = self.calc_noise_vec(hp_list[0])
            noise = bk.to_dev(nv) if np.any(nv) else None
            varK = np.array([float(h.varK) for h in hp_list])
        bk.build_cov_batch(self._X_dev, np.vstack([np.asarray(h.theta, dtype=float) for h in hp_list]), n_g=self.n_grad,
                           slot=self._slot_dev, noise=noise, varK_rows=varK, mode=mode,
                           eta=getattr(self, "_eta_used", self._etaK), out=v["U"], kernel=self._kern(),
                           kernel_hp_rows=np.array([self._kern(h)[1] for h in hp_list]))
        return v

    def _cond2_from_workspace(self, hp_list, calc_grad, warm, rows=None):
        """kappa_2 (+ gradient) of every candidate of the evaluation that has just run (_rebuild_in_workspace), the
        Lanczos iterations of all candidates batched (backend.cond2_batch); warm: one earlier result or None per row;
        rows: the candidates to evaluate (default all; the others get None throughout).
        -> (list of kappa, list of gradient or None, list of cond2 results)."""
        v = self._rebuild_in_workspace(hp_list, calc_grad)
        res = bk.cond2_batch(v["U"], v["Kinv"], self.n_data, warm=warm, rows=rows)
        idx = [i for i, r in enumerate(res) if r is not None]
        vk = [float(h.varK) if self.b_has_noisy_data else 1.0 for h in hp_list]
        grads = [None] * len(hp_list)
        if calc_grad:
            for i, g in zip(idx, self._cond_grads([hp_list[i] for i in idx], [res[i] for i in idx], [vk[i] for i in idx])):
                grads[i] = g
        return [None if r is None else float(r["cond"]) for r in res], grads, res

    def _cond_from_workspace(self, hp_vals, calc_grad):
        """Condition number (+ gradient) of the matrix the likelihood evaluation that has just run factored."""
        if self.cond_norm not in (2, "fro"):
            raise Exception(f'cond_norm must be either 2 or "fro" but it is {self.cond_norm}')
        if self.cond_norm == "fro":   # optz/GpHparaCon.py:237-261
            v = self._rebuild_in_workspace([hp_vals], calc_grad)
            theta, _, varK = self._cond_matrix_args(hp_vals)
            want_w = calc_grad and self.wellcond_mtd != "precon"
            cond, W = bk.cond_fro(v["U"][0], v["Kinv"][0], self.n_data, want_w)
            if not want_w:
                return cond, None
            q = bk.weighted_grad(self._X_dev, theta, W, n_g=self.n_grad, slot=self._slot_dev,
                                 eta=getattr(self, "_eta_used", self._etaK), noisy=self.b_has_noisy_data,
                                 varK=varK, kernel=self._kern(hp_vals)).cpu().numpy()
            return cond, self._hp_row_to_grad(q)
        warm = getattr(self, "_last_cond", None) if self.cond_warm_start else None
        cond, grad, res = self._cond2_from_workspace([hp_vals], calc_grad, [warm])
        self._last_cond = res[0]
        return cond[0], grad[0]

    def _cond_on_failure(self, hp_vals, calc_grad=False):
        """Failed Cholesky: the reference substitutes -cond (and -cond_grad) for the objective (optz/OptzLkd.py:75-77).
        The matrix is numerically singular; it is factored once more with a tiny diagonal shift (backend.cond2_of_matrix)."""
        try:
            theta, noise, varK = self._cond_matrix_args(hp_vals)
            K = bk.build_cov(self._X_dev, theta, n_g=self.n_grad, slot=self._slot_dev, noise=noise, mode=self._mode,
                             eta=getattr(self, "_eta_used", self._etaK), varK=varK, kernel=self._kern(hp_vals))[0]
            res = bk.cond2_of_matrix(K, self.n_data)
            self._last_cond = res
            return float(res["cond"]), (self._cond_grad_from_vectors(hp_vals, res, varK) if calc_grad else None)
        except Exception:
            return np.inf, (np.zeros(self.hp_info_optz_lkd.n_hp) if calc_grad else None)

    def calc_lkd_batch(self, hp_vec_rows, calc_grad=False, calc_cond=False):
        """LML (and d/dtheta) of many candidate rows at once, sharded over the process group.

        hp_vec_rows: [B, n_hp] in optimiser coordinates (log10 where bvec_log_optz).  Returns a NumPy table
        [B, 9+d] laid out as GEGP_OUT_* -- identical on every rank.  This is the batched form of the loops at
        optz/GpHparaX0.py:39-45 and optz/OptzLkd.py:249-270.

        calc_cond=True appends the 2-norm condition number kappa of the factored matrix as column 9+d and, with calc_grad
        outside precon mode, dkappa/dhp in the optimiser's hyper-parameter order (n_hp columns more): row i holds what
        calc_lkd_all(row i, calc_cond=True, calc_grad=calc_grad) returns as cond / cond_grad (a failed Cholesky takes
        kappa from the shifted refactorisation of _cond_on_failure).  The likelihood columns then come from the
        gradient-path evaluation calc_lkd_all runs for kappa; where kappa > cond_max_abs outside precon mode,
        calc_lkd_all reports no likelihood and OUT_LML is NaN.  The Lanczos iterations of all rows run batched and are
        not warm-started, so every row is bit-identical to calc_lkd_all with cond_warm_start = False.  Needs
        cond_norm = 2 and a constant nugget."""
        rows = np.atleast_2d(np.asarray(hp_vec_rows, dtype=float))
        hi = self.hp_info_optz_lkd
        assert not (hi.has_var_fval or hi.has_var_fgrad), "rows with their own noise variance are evaluated one by one"
        if calc_cond and (self.cond_norm != 2 or not self.cond_eta_is_const):
            raise Exception("calc_lkd_batch(calc_cond=True) needs cond_norm = 2 and a constant nugget, but cond_norm = "
                            f"{self.cond_norm} and cond_eta_is_const = {self.cond_eta_is_const}")
        th = rows[:, hi.idx_theta].copy()
        if self.optz_log_hp_theta:
            th = 10 ** th
        cols = [th]
        if self.kernel_has_hp:      # the kernel's own hyper-parameter rides along as one more candidate column
            kh = rows[:, hi.idx_kernel[0]].copy() if hi.has_kernel else np.full(rows.shape[0], float(self.hp_kernel_default))
            if hi.has_kernel and self.optz_log_hp_kernel:
                kh = 10 ** kh
            cols.append(kh[:, None])
        noise = None
        if self.b_has_noisy_data:   # known noise: one vector for every row; varK is a column of the candidate table
            vk = rows[:, hi.idx_varK].copy()
            cols.append((10 ** vk if self.optz_log_hp_var else vk)[:, None])
            noise = self.calc_noise_vec(self.make_hp_class(theta=th[0]))
        cand = bk.to_dev(np.hstack(cols))
        d = self.dim
        c_k = d if self.kernel_has_hp else None
        c_v = (d + (1 if self.kernel_has_hp else 0)) if self.b_has_noisy_data else None
        width = L.out_len(d)

        if not calc_cond:
            def eval_shard(c):
                return self._eval_rows(c[:, :d].contiguous(), want_grad=calc_grad,
                                       khp_rows=c[:, c_k].cpu().numpy() if c_k is not None else None,
                                       varK_rows=c[:, c_v].cpu().numpy() if c_v is not None else None, noise_vec=noise)
        else:
            with_grad = calc_grad and self.wellcond_mtd != "precon"
            width += 1 + (hi.n_hp if with_grad else 0)

            def eval_shard(c):
                import torch
                h = c.cpu().numpy()
                hp_list = [self.make_hp_class(theta=h[i, :d].copy(), kernel=h[i, c_k] if c_k is not None else None,
                                              varK=h[i, c_v] if c_v is not None else None) for i in range(h.shape[0])]
                out, cond, cgrad = self._lkd_cond_rows(hp_list, calc_grad, noise)[:3]
                tab = np.hstack([out, cond[:, None]] + ([cgrad] if with_grad else []))
                return torch.as_tensor(tab).to(c.device)
        table = parallel.sharded_eval(eval_shard, cand, self.dist_group, width=width)
        return table.cpu().numpy()

    lml_ws_max_bytes = None   # cap on the likelihood workspace of batched evaluations that also need kappa (None: 60% free)

    def _lkd_cond_rows(self, hp_list, calc_grad, noise=None, warm=None):
        """Likelihood rows (gradient path, GEGP_OUT_*) and kappa_2 (+ dkappa/dhp outside precon mode) of many
        hyper-parameter rows that share the nugget and the noise vector `noise`.  gegp_lml_eval reuses its workspace
        chunk by chunk, so the rows go to the device in chunks that fit it, and kappa of a chunk is computed before the
        next chunk overwrites its factors.  warm: None or one earlier cond2 result per row.
        -> (out [B, 9+d], kappa [B], dkappa [B, n_hp] or None, the warm state each row leaves behind (what
        calc_lkd_all leaves in _last_cond), b_chofac_good [B] as calc_lkd_all returns it)."""
        B, d = len(hp_list), self.dim
        n_hp = self.hp_info_optz_lkd.n_hp
        with_grad = calc_grad and self.wellcond_mtd != "precon"
        out = np.zeros((B, L.out_len(d)))
        cond = np.zeros(B)
        cgrad = np.zeros((B, n_hp)) if with_grad else None
        warm = list(warm) if warm is not None else [None] * B
        res_all = list(warm)
        good_all = np.zeros(B, dtype=bool)
        self._eta_used = self._etaK
        last_cond = getattr(self, "_last_cond", None)
        chunk = self._cond_chunk_rows(B)
        for c0 in range(0, B, chunk):
            part = hp_list[c0:c0 + chunk]
            th = np.vstack([np.asarray(h.theta, dtype=float) for h in part])
            khp = np.array([self._kern(h)[1] for h in part]) if self.kernel_has_hp else None
            vk = np.array([float(h.varK) for h in part]) if self.b_has_noisy_data else None
            o = self._eval_rows(th, want_grad=True, khp_rows=khp, varK_rows=vk, noise_vec=noise).cpu().numpy()
            out[c0:c0 + len(part)] = o
            good = [i for i in range(len(part)) if o[i, L.OUT_INFO] == 0]
            if good:
                c, g, res = self._cond2_from_workspace(part, calc_grad, warm[c0:c0 + len(part)], rows=good)
                for i in good:
                    cond[c0 + i], res_all[c0 + i] = c[i], res[i]
                    if with_grad:
                        cgrad[c0 + i] = g[i]
            for i in range(len(part)):
                if o[i, L.OUT_INFO] != 0:      # failed Cholesky: shifted refactorisation, row by row
                    self._last_cond = warm[c0 + i]
                    c, g = self._cond_on_failure(part[i], calc_grad)
                    cond[c0 + i], res_all[c0 + i] = c, self._last_cond
                    if with_grad:
                        cgrad[c0 + i] = g
                elif self.wellcond_mtd != "precon" and cond[c0 + i] > self.cond_max_abs:
                    out[c0 + i, L.OUT_LML] = np.nan       # kernel/Kernel.py:282-283: no likelihood
                else:
                    good_all[c0 + i] = True
        self._last_cond = last_cond
        return out, cond, cgrad, res_all, good_all

    def _cond_chunk_rows(self, B):
        """Rows per likelihood call of _lkd_cond_rows: as many as the workspace keeps at once (lml_ws_max_bytes)."""
        self._ensure_device()
        return bk.lml_chunk_rows(self.n_eval, self.n_grad, self.dim, B, want_grad=True, max_ws_bytes=self.lml_ws_max_bytes)

    # ------------------------------------------------------------------ optimiser callbacks (optz/OptzLkd.py:16-113)
    def calc_store_likelihood(self, hp_vec, always_calc_cond=False, calc_grad=True):
        hp_vec = np.atleast_1d(hp_vec).ravel()
        # value and gradient come from ONE fused evaluation; the cache makes the second callback free
        # (the reference never refreshes _last_hp_vec, optz/OptzLkd.py:48 vs :263, and evaluates twice).
        if not np.array_equal(hp_vec, self._last_hp_vec):
            hp_vals = self.hp_vec2dataclass(self.hp_info_optz_lkd, hp_vec)
            calc_cond = self.b_use_cond_cstr or always_calc_cond
            lkd_info, good = self.calc_lkd_all(hp_vals, calc_lkd=True, calc_cond=calc_cond, calc_grad=calc_grad)
            cond_val, cond_grad = lkd_info.cond, lkd_info.cond_grad
            if good:
                val, grad = lkd_info.ln_lkd, lkd_info.ln_lkd_grad
                if calc_grad:
                    b = self.hp_info_optz_lkd.bvec_log_optz
                    grad = grad.copy()
                    grad[b] *= 10 ** hp_vec[b] * np.log(10)
                    if self.b_use_cond_cstr and cond_grad is not None:
                        cond_grad = cond_grad.copy()
                        cond_grad[b] *= 10 ** hp_vec[b] * np.log(10)
            else:   # failed Cholesky: the condition number becomes the objective (optz/OptzLkd.py:75-77)
                val = -cond_val
                grad = -cond_grad if cond_grad is not None else np.zeros(hp_vec.size)
            self._lkd_val, self._lkd_grad, self._cond_val, self._cond_grad = val, grad, cond_val, cond_grad
            if calc_grad:
                self._last_hp_vec = hp_vec.copy()
        return self._lkd_val, self._lkd_grad, self._cond_val, self._cond_grad

    def return_optz_val(self, hp_vec):
        return -self.calc_store_likelihood(hp_vec)[0]

    def return_optz_grad(self, hp_vec):
        return -self.calc_store_likelihood(hp_vec)[1]

    def return_cond_val(self, hp_vec):
        return self.calc_store_likelihood(hp_vec)[2]

    def return_cond_grad(self, hp_vec):
        return self.calc_store_likelihood(hp_vec)[3]

    # ------------------------------------------------------------------ start points (optz/GpHparaX0.py)
    def get_hp_x0_lhs_median(self, i_optz, hp_optz_info, n_x0):
        """LHS in log10 space around the median of past hyper-parameters (optz/GpHparaX0.py:67-183)."""
        lo_i, hi_i = int(max(0, i_optz - self.hp_median_n_idx)), i_optz
        lf, bf = self.hp_lhs_bound_factor, self.hp_box_bound_factor
        n_hp = hp_optz_info.n_hp
        lhs_lb, lhs_ub, box_lb, box_ub = (np.full(n_hp, np.nan) for _ in range(4))

        def fill(idx, hist, rng):
            med = np.clip(np.median(hist, axis=0), rng[0], rng[1])
            lhs_lb[idx], lhs_ub[idx] = np.maximum(med / lf, rng[0]), np.minimum(med * lf, rng[1])
            box_lb[idx], box_ub[idx] = np.maximum(med / bf, rng[0]), np.minimum(med * bf, rng[1])

        if hp_optz_info.has_theta:
            fill(hp_optz_info.idx_theta, self.hp_theta_all[lo_i:hi_i, :], self.hp_theta_range)
        if hp_optz_info.has_kernel:     # optz/GpHparaX0.py:100-111
            fill(hp_optz_info.idx_kernel, self.hp_kernel_all[lo_i:hi_i], self.hp_kernel_range)
        if hp_optz_info.has_varK:
            fill(hp_optz_info.idx_varK, self.hp_varK_all[lo_i:hi_i], self.hp_varK_range)
        if hp_optz_info.has_var_fval:
            fill(hp_optz_info.idx_var_fval, np.maximum(self.hp_var_fval_all[lo_i:hi_i], self.hp_var_fval_range[0]),
                 self.hp_var_fval_range)
        if hp_optz_info.has_var_fgrad:
            fill(hp_optz_info.idx_var_fgrad, np.maximum(self.hp_var_fgrad_all[lo_i:hi_i], self.hp_var_fgrad_range[0]),
                 self.hp_var_fgrad_range)
        b = hp_optz_info.bvec_log_optz
        for arr in (lhs_lb, lhs_ub, box_lb, box_ub):
            arr[b] = np.log10(arr[b])
        if np.any(lhs_lb > lhs_ub) or np.any(np.isnan(lhs_lb)):
            raise Exception("Invalid bounds for lhs")
        if np.any(box_lb > box_ub):
            raise Exception("Invalid bounds for box")
        bounds = Bounds(box_lb, box_ub, keep_feasible=True)
        if n_hp == 1:
            hp_x0 = np.linspace(lhs_lb[0], lhs_ub[0], n_x0 + 2)[1:-1, None]
        else:
            hp_x0 = self._lhs(np.array([lhs_lb, lhs_ub]).T, n_x0)
        return hp_x0, bounds

    @staticmethod
    def _lhs(limits, n, seed=1):
        """Latin hypercube with random_state=1 like the reference; `smt` when importable, else scipy.stats.qmc."""
        try:
            from smt.sampling_methods import LHS  # noqa: WPS433 (optional dependency of the reference)
            return LHS(xlimits=limits, random_state=seed)(n)
        except Exception:
            unit = qmc.LatinHypercube(d=limits.shape[0], seed=seed).random(n)
            return limits[:, 0][None, :] + unit * (limits[:, 1] - limits[:, 0])[None, :]

    def select_hp_optz_x0(self, i_optz, hp_optz_info):
        """optz/GpHparaX0.py:16-65; the 40-candidate scan runs as ONE batched device call (sharded over ranks)."""
        t0 = time.time()
        if self.lkd_optz_start_mtd == "lhs":
            n_x0 = self.optz_n_x0
        elif self.lkd_optz_start_mtd == "hp_best":
            n_x0 = self.lkd_hp_best_n_eval
        else:
            raise Exception(f"Unknown lkd_optz_start_mtd: {self.lkd_optz_start_mtd}")
        hp_x0, bounds = self.get_hp_x0_lhs_median(i_optz, hp_optz_info, n_x0)
        self._scan_stats = None
        if self.lkd_optz_start_mtd == "hp_best":
            calc_cond = self.wellcond_mtd != "precon"
            if self._can_batch_scan(hp_optz_info):
                # ONE batched device call for the LML of all rows; the condition number (base / rescale modes) is only
                # needed to veto the winner, so it is computed lazily down the LML ranking: same selection as the loop
                tab = self.calc_lkd_batch(hp_x0, calc_grad=False)
                lml = np.where(tab[:, L.OUT_INFO] == 0, tab[:, L.OUT_LML], np.nan)
                n_cond = 0
                if calc_cond and np.any(np.isfinite(lml)):
                    cond_all = np.full(n_x0, np.nan)
                    order = [i for i in np.argsort(-np.where(np.isfinite(lml), lml, -np.inf)) if np.isfinite(lml[i])]
                    chosen = None
                    for i in order:
                        info, good = self.calc_lkd_all(self.hp_vec2dataclass(hp_optz_info, hp_x0[i, :]), calc_cond=True)
                        n_cond += 1
                        cond_all[i] = info.cond if info.cond is not None else np.nan
                        if good and not (cond_all[i] > 1.2 * self.cond_max):
                            chosen = i
                            break
                        lml[i] = np.nan
                    if chosen is None:      # every row is too ill-conditioned: the loop keeps the least bad one
                        lml[:] = np.nan
                        if np.any(np.isfinite(cond_all)):
                            k = int(np.nanargmin(cond_all))
                            lml[k] = tab[k, L.OUT_LML]
                self._scan_stats = dict(batched=True, n_cond_evals=n_cond)
            else:
                lml = np.full(n_x0, np.nan)
                cond_all = np.full(n_x0, np.nan)
                for i in range(n_x0):
                    info, good = self.calc_lkd_all(self.hp_vec2dataclass(hp_optz_info, hp_x0[i, :]), calc_cond=calc_cond)
                    if good:
                        lml[i], cond_all[i] = info.ln_lkd, (info.cond if info.cond is not None else np.nan)
                if calc_cond:
                    bad = cond_all > 1.2 * self.cond_max
                    if np.sum(bad) == bad.size:
                        bad[np.nanargmin(cond_all)] = False
                    lml[bad] = np.nan
                self._scan_stats = dict(batched=False, n_cond_evals=n_x0 if calc_cond else 0)
            hp_x0 = hp_x0[np.nanargmax(lml), :][None, :]
        return hp_x0, bounds, time.time() - t0

    def _can_batch_scan(self, hp_optz_info):
        """The candidate scan runs as one batched call whenever every row shares the nugget and the noise vector: constant
        eta, no varK penalty, and no noise variance among the optimised hyper-parameters (known noise is fine)."""
        return self.cond_eta_is_const and (not self.lkd_varK_pnlt_use) and (not hp_optz_info.has_var_fval) \
            and (not hp_optz_info.has_var_fgrad)

    # ------------------------------------------------------------------ fit (optz/GpHparaOptz.py, optz/OptzLkd.py:185-333)
    def get_init_hp_vals(self):
        fval = self.get_scl_eval_data()[0]
        beta = np.array([np.mean(fval)])
        vf = None if self.known_eps_fval else self.hp_var_fval_init
        vg = None if ((self.use_grad is False) or self.known_eps_fgrad) else self.hp_var_fgrad_init
        return self.make_hp_class(beta, self.hp_theta_init * np.ones(self.dim), self.hp_kernel_default, self.hp_varK_init,
                                  vf, vg)

    def optz_closed_form_hp(self, hp_vals):
        info, _ = self.calc_lkd_all(hp_vals, calc_lkd=False, calc_cond=False, calc_grad=False)
        hp_vals.beta = info.hp_beta
        if self.b_has_noisy_data is False:
            hp_vals.varK = info.hp_varK
        return hp_vals

    def optz_hp_max_lkd(self, hp_x0_all, optz_bound):
        """optz/OptzLkd.py:185-333: SLSQP from every start row, with the condition-number constraint
        kappa_2 <= cond_max outside precon mode; the best feasible solution wins."""
        if self.optz_mtd == "SLSQP":        # recommended by the reference (optz/OptzLkd.py:209)
            opt = {"ftol": self.optz_tol_obj, "eps": self.optz_tol_x, "maxiter": self.optz_iter_max, "disp": False}
        elif self.optz_mtd == "trust-constr":   # optz/OptzLkd.py:216-221
            opt = {"initial_tr_radius": 0.1, "xtol": self.optz_tol_x, "gtol": self.optz_tol_obj,
                   "maxiter": self.optz_iter_max, "disp": False}
        else:
            raise Exception(f"Unknown optz_mtd = {self.optz_mtd}")
        if hp_x0_all.ndim == 1:
            hp_x0_all = hp_x0_all[None, :]
        n_optz = hp_x0_all.shape[0]
        ok = np.zeros(n_optz, bool)
        con_good = np.zeros(n_optz, bool)
        nit = np.full(n_optz, np.nan)
        obj = np.full(n_optz, np.nan)
        cond_all = np.full(n_optz, np.nan)
        sol = np.full((n_optz, self.hp_info_optz_lkd.n_hp), np.nan)
        n_cho_fail = n_cond2big = 0
        max_init_cond = np.nan
        nlc = self.condnum_nlc if self.b_use_cond_cstr else []
        if n_optz > 1 and self.lockstep_multistart and self.optz_mtd == "SLSQP" and self._can_batch_fit():
            return self._optz_multistart_lockstep(hp_x0_all, optz_bound, opt)
        for i in range(n_optz):
            x0 = hp_x0_all[i, :]
            self._last_hp_vec = None
            if self.b_use_cond_cstr:
                lkd_val, _, cond_val = self.calc_store_likelihood(x0)[:3]
                max_init_cond = np.nanmax((max_init_cond, cond_val))
                if np.isnan(lkd_val):
                    n_cho_fail += 1
                if cond_val > self.cond_max:
                    n_cond2big += 1
            self._last_hp_vec = None
            res = minimize(self.return_optz_val, x0, method=self.optz_mtd, jac=self.return_optz_grad, bounds=optz_bound,
                           constraints=nlc, options=opt)
            sol[i, :], obj[i], ok[i], nit[i] = res.x, res.fun, res.success, res.nit
            if self.b_use_cond_cstr:
                cond_all[i] = self.return_cond_val(res.x)
                con_good[i] = cond_all[i] < 1.01 * self.cond_max
            else:
                con_good[i] = True
        if np.any(con_good):
            obj_ok, sol_ok = obj[con_good], sol[con_good, :]
        else:
            print("*** No solutions satisfy the constraints for the GP hyperparameter optimization ***")
            obj_ok, sol_ok = obj, sol
        best = sol_ok[np.nanargmin(obj_ok), :]
        info = {"hp_optz_success": float(np.mean(ok)), "hp_optz_iter_mean": float(np.mean(nit)),
                "hp_optz_iter_max": float(np.max(nit)), "hp_optz_con_good": float(np.mean(con_good)),
                "optz_n_cho_fail": n_cho_fail, "optz_n_cond2big": n_cond2big, "optz_max_init_cond": max_init_cond}
        return best, self._final_cond(best), info

    def _final_cond(self, best):
        """Condition number of the matrix the chosen solution factors (optz/OptzLkd.py:323-331; every mode: in precon
        mode it is kappa of the preconditioned matrix, kernel/Kernel.py:240) -- it ends up in Kcov_cond_all."""
        best_vals = self.hp_vec2dataclass(self.hp_info_optz_lkd, best)
        return self.calc_all_K_w_chofac(None, best_vals, calc_chofac=False, calc_cond=True,
                                        varK=None if self.b_has_noisy_data else 1)[4]

    def _can_batch_fit(self):
        """The batched objective covers the noise-free fit with a constant nugget: unconstrained (precon), or with the
        kappa_2 <= cond_max constraint of the base / rescale / dflt modes (adjoint-form gradient)."""
        cstr_ok = (not self.b_use_cond_cstr) or (self.cond_norm == 2 and self.lkd_use_adj_mtd)
        return (not self.b_has_noisy_data) and cstr_ok and self.cond_eta_is_const \
            and (not self.lkd_varK_pnlt_use) and self.optz_log_hp_theta and (not self.kernel_has_hp)

    def _optz_multistart_lockstep(self, hp_x0_all, optz_bound, opt):
        """Batch point B (optz/OptzLkd.py:249-270): every start row is its own SLSQP instance; their objective requests
        are evaluated together (multistart.minimize_lockstep), the start rows sharded over the ranks of dist_group.
        Same trajectories and the same selected optimum as the sequential loop (batched == single, bit for bit).

        With the condition-number constraint every request also returns kappa_2 and its gradient (_lkd_cond_rows, the
        Lanczos iterations of all requests batched), following calc_store_likelihood exactly, and the per-start
        bookkeeping of the sequential loop is reproduced.  Warm start: each start row begins from the GP's warm state
        on entry and then carries its own, so start i follows the trajectory it would follow as the only start row of a
        sequential fit begun in the same state (the sequential loop chains the warm vectors across start rows, so with
        cond_warm_start the two agree to the Lanczos tolerance; without it, bit for bit)."""
        import torch
        from . import multistart
        hi = self.hp_info_optz_lkd
        rank, size = parallel.world(self.dist_group)
        n_optz = hp_x0_all.shape[0]
        lo, hi_row = parallel.shard_bounds(n_optz, rank, size)
        d = self.dim
        cstr = self.b_use_cond_cstr
        warm_state = {i: getattr(self, "_last_cond", None) for i in range(lo, hi_row)}

        def batch_val_and_grad(Xlog):
            th = 10 ** Xlog[:, hi.idx_theta]
            tab = self._eval_rows(th, want_grad=True).cpu().numpy()
            ok = tab[:, L.OUT_INFO] == 0
            vals = np.empty(Xlog.shape[0])
            grads = np.zeros((Xlog.shape[0], hi.n_hp))
            for r in range(Xlog.shape[0]):
                if ok[r]:
                    vals[r] = -tab[r, L.OUT_LML]
                    g = tab[r, L.OUT_GRAD:L.OUT_GRAD + d].copy()
                    g *= 10 ** Xlog[r, hi.idx_theta] * np.log(10)     # same expression as calc_store_likelihood
                    grads[r, hi.idx_theta] = -g
                else:   # failed Cholesky: the condition number becomes the objective (optz/OptzLkd.py:75-77)
                    hp_vals = self.hp_vec2dataclass(hi, Xlog[r])
                    vals[r] = self._cond_on_failure(hp_vals, False)[0]
            return vals, grads

        def batch_cond(Xlog, ids):
            """calc_store_likelihood(x, calc_grad=True) for every request, negated for minimisation."""
            hp_list = [self.hp_vec2dataclass(hi, x) for x in Xlog]
            warm = [warm_state[i] for i in ids] if self.cond_warm_start else None
            out, cond, cgrad, res, good = self._lkd_cond_rows(hp_list, True, None, warm)
            if self.cond_warm_start:
                warm_state.update(zip(ids, res))
            b = hi.bvec_log_optz
            vals, grads, cgs = np.empty(len(ids)), np.zeros((len(ids), hi.n_hp)), np.zeros((len(ids), hi.n_hp))
            for r, hp_vec in enumerate(Xlog):
                if good[r]:
                    val = out[r, L.OUT_LML]
                    grad = np.zeros(hi.n_hp)
                    grad[hi.idx_theta] = out[r, L.OUT_GRAD:L.OUT_GRAD + d]
                    grad[b] *= 10 ** hp_vec[b] * np.log(10)
                    cg = cgrad[r].copy()
                    cg[b] *= 10 ** hp_vec[b] * np.log(10)
                else:   # failed Cholesky or kappa > cond_max_abs: -kappa is the objective (optz/OptzLkd.py:75-77)
                    val, grad, cg = -cond[r], -cgrad[r], cgrad[r]
                vals[r], grads[r], cgs[r] = -val, -grad, cg
            return vals, grads, cond.copy(), cgs

        W = hi.n_hp + (6 if cstr else 3)
        local = np.full((max(hi_row - lo, 0), W), np.nan)
        self._lockstep_stats = None
        if hi_row > lo:
            cur_dev = torch.cuda.current_device() if torch.cuda.is_available() else None
            init = (lambda: torch.cuda.set_device(cur_dev)) if cur_dev is not None else None
            if cstr:
                res, ev = multistart.minimize_lockstep(batch_cond, hp_x0_all[lo:hi_row], optz_bound, opt,
                                                       thread_init=init, with_ids=True, cond_ub=self.condnum_nlc.ub)
            else:
                res, ev = multistart.minimize_lockstep(batch_val_and_grad, hp_x0_all[lo:hi_row], optz_bound, opt,
                                                       thread_init=init)
            self._lockstep_stats = dict(n_batches=ev.n_batches, n_evals=ev.n_evals, batch_sizes=ev.batch_sizes)
            for i, r in enumerate(res):
                local[i, :hi.n_hp], local[i, hi.n_hp:hi.n_hp + 3] = r.x, (r.fun, float(r.success), r.nit)
                if cstr:   # kappa at the solution; LML and kappa at x0 (-objective is the LML, or -kappa on failure)
                    local[i, hi.n_hp + 3:] = (ev.at_solution[i][2], -ev.at_x0[i][0], ev.at_x0[i][2])
        if size > 1:
            # a rank without start rows (more ranks than rows) contributes an empty block but enters the collective
            t = torch.as_tensor(local)
            t = t.to(bk.device()) if torch.cuda.is_available() else t
            table = parallel.gather_rows(t, n_optz, self.dist_group, width=W).cpu().numpy()
        else:
            table = local
        self._multistart_table = table   # per start row: solution, objective, success, iterations (+ kappa columns)
        sol, obj, ok, nit = table[:, :hi.n_hp], table[:, hi.n_hp], table[:, hi.n_hp + 1], table[:, hi.n_hp + 2]
        if not cstr:
            best = sol[np.nanargmin(obj), :]
            info = {"hp_optz_success": float(np.mean(ok)), "hp_optz_iter_mean": float(np.mean(nit)),
                    "hp_optz_iter_max": float(np.max(nit)), "hp_optz_con_good": 1.0, "optz_n_cho_fail": 0,
                    "optz_n_cond2big": 0, "optz_max_init_cond": np.nan}
            return best, self._final_cond(best), info
        cond_sol, lkd_x0, cond_x0 = table[:, hi.n_hp + 3], table[:, hi.n_hp + 4], table[:, hi.n_hp + 5]
        n_cho_fail = n_cond2big = 0
        max_init_cond = np.nan
        for i in range(n_optz):          # the bookkeeping of the sequential loop, in its order
            max_init_cond = np.nanmax((max_init_cond, cond_x0[i]))
            if np.isnan(lkd_x0[i]):
                n_cho_fail += 1
            if cond_x0[i] > self.cond_max:
                n_cond2big += 1
        con_good = cond_sol < 1.01 * self.cond_max
        if np.any(con_good):
            obj_ok, sol_ok = obj[con_good], sol[con_good, :]
        else:
            print("*** No solutions satisfy the constraints for the GP hyperparameter optimization ***")
            obj_ok, sol_ok = obj, sol
        best = sol_ok[np.nanargmin(obj_ok), :]
        info = {"hp_optz_success": float(np.mean(ok)), "hp_optz_iter_mean": float(np.mean(nit)),
                "hp_optz_iter_max": float(np.max(nit)), "hp_optz_con_good": float(np.mean(con_good)),
                "optz_n_cho_fail": n_cho_fail, "optz_n_cond2big": n_cond2big, "optz_max_init_cond": max_init_cond}
        return best, self._final_cond(best), info

    def rescaling_data_w_theta_sol(self, X_scl_v1, xvec_scale_v1, hp_theta, tol_min_dist_x=1e-15):
        """base/GpWellCond.py:42-76: anisotropic re-scaling of x by sqrt(theta / geometric-mean theta), corrected so
        that the minimum pairwise distance is v_req again; returns the isotropic theta estimate in the new coordinates."""
        from scipy.spatial.distance import pdist
        assert X_scl_v1.shape[0] > 1, "This method should only be called if n_eval > 1"
        if self.optz_log_hp_theta:
            theta_sol, log_theta = 10 ** hp_theta, hp_theta
        else:
            theta_sol, log_theta = hp_theta, np.log10(hp_theta)
        vreq = self.calc_mtd_rescale_origin_vreq(X_scl_v1.shape[0], self.dim)
        theta_star = 10 ** np.mean(log_theta)
        scale_v2 = np.sqrt(theta_sol / theta_star)
        min_dist = max(float(np.min(pdist(X_scl_v1 * scale_v2[None, :]))), tol_min_dist_x)
        corr = vreq / min_dist
        dist2 = np.dot(log_theta, log_theta) - np.dot(log_theta, np.ones(self.dim)) ** 2 / self.dim
        est = np.ones(self.dim) * theta_star / corr ** 2
        return (np.log10(est) if self.optz_log_hp_theta else est), dist2, xvec_scale_v1 * scale_v2 * corr

    def optz_hp_max_lkd_mtd_rescale(self, i_optz, hp_x0, optz_bound):
        """optz/OptzLkd.py:116-183: optimise, re-scale x with the solution's theta, optimise again from the isotropic
        estimate -- up to cond_vreq_max_iter times or until theta is isotropic within cond_vreq_iter_tol."""
        assert "rescale" in self.wellcond_mtd
        best_hp, cond_val, info = self.optz_hp_max_lkd(hp_x0, optz_bound)
        if self.n_eval <= 1:
            return best_hp, cond_val, info
        max_iter, idx = self.cond_vreq_max_iter, self.hp_info_optz_lkd.idx_theta
        theta_all = np.full((max_iter, self.dim), np.nan)
        dist_all = np.full(max_iter, np.nan)
        scale_all = np.full((max_iter, self.dim), np.nan)
        theta_new = best_hp[idx]
        for cnt in range(max_iter):
            theta_new, dist, scale_new = self.rescaling_data_w_theta_sol(self.DataScl.x_scl, self.DataScl.xvec_scale,
                                                                         theta_new)
            theta_all[cnt, :], dist_all[cnt], scale_all[cnt, :] = theta_new, dist, scale_new
            if cnt == max_iter - 1 or dist < self.cond_vreq_iter_tol:
                break
            x0 = best_hp.copy()
            x0[idx] = theta_new
            best_hp, cond_val = self.optz_hp_max_lkd(x0, optz_bound)[:2]
        k = int(np.nanargmin(dist_all))
        self.DataScl.set_xscale_data(xvec_scale_in=scale_all[k, :])
        self._dev_ready = False          # the scaled training data changed: refresh the device copy
        self._last_hp_vec = None
        best_final = best_hp.copy()
        best_final[idx] = theta_all[k, :]
        return best_final, cond_val, info

    def optz_hp(self, i_optz):
        if self.n_eval <= self.hp_const_n_eval:
            hp_vals, info = self.get_init_hp_vals(), None
            cond_val = self.calc_all_K_w_chofac(None, hp_vals, calc_chofac=False, calc_cond=True)[4]
            t_optz = t_cho = t_x0 = 0
        else:
            self._time_chofac = 0
            hp_x0, bound, t_x0 = self.select_hp_optz_x0(i_optz, self.hp_info_optz_lkd)
            t0 = time.time()
            if "rescale" in self.wellcond_mtd and self.cond_vreq_max_iter > 1:
                hp_optz, cond_val, info = self.optz_hp_max_lkd_mtd_rescale(i_optz, hp_x0, bound)
            else:
                hp_optz, cond_val, info = self.optz_hp_max_lkd(hp_x0, bound)
            t_optz, t_cho = time.time() - t0, self._time_chofac
            hp_vals = self.optz_closed_form_hp(self.hp_vec2dataclass(self.hp_info_optz_lkd, hp_optz))
        self.store_new_para_surr(i_optz, hp_vals, info, cond_val, t_optz, t_cho, t_x0)

    # ------------------------------------------------------------------ history (base/GpParaDef.py)
    def init_optz_surr(self, n_optz_max):
        self._save_data, self.n_optz_max = True, n_optz_max
        full = lambda *s: np.full(s, np.nan)  # noqa: E731
        self.hp_beta_all, self.hp_varK_all = full(n_optz_max, self.n_beta_coeff), full(n_optz_max)
        self.hp_var_fval_all, self.hp_var_fgrad_all = full(n_optz_max), full(n_optz_max)
        self.hp_kernel_all, self.hp_theta_all = full(n_optz_max), full(n_optz_max, self.dim)
        self.min_nugget_all, self.Kcov_cond_all = full(n_optz_max), full(n_optz_max)
        self.eta_Kbase_all, self.eta_Kgrad_all = full(n_optz_max), full(n_optz_max)
        self.vmin_init_all, self.vmin_req_grad_all = full(n_optz_max), full(n_optz_max)
        self.xvec_rescaling_all = full(n_optz_max, self.dim)
        self.hp_optz_success, self.hp_optz_iter_mean, self.hp_optz_iter_max = full(n_optz_max), full(n_optz_max), full(n_optz_max)
        self.time_pick_hp0_all, self.time_hp_optz_all, self.time_chofac_all = full(n_optz_max), full(n_optz_max), full(n_optz_max)

    def store_new_para_surr(self, i_optz, hp_vals, surr_optz_info=None, cond_val=np.nan, time_hp_optz=np.nan,
                            time_chofac=np.nan, time_pick_hp0=np.nan):
        self.hp_vals = hp_vals
        if self._save_data is False:
            return
        i = i_optz
        self.time_hp_optz_all[i], self.time_chofac_all[i], self.time_pick_hp0_all[i] = time_hp_optz, time_chofac, time_pick_hp0
        self.hp_beta_all[i, :], self.hp_theta_all[i, :] = hp_vals.beta, hp_vals.theta
        self.hp_varK_all[i] = hp_vals.varK
        self.hp_kernel_all[i] = np.nan if hp_vals.kernel is None else hp_vals.kernel
        self.hp_var_fval_all[i] = np.nan if hp_vals.var_fval is None else hp_vals.var_fval
        self.hp_var_fgrad_all[i] = np.nan if hp_vals.var_fgrad is None else hp_vals.var_fgrad
        self.min_nugget_all[i] = self._eta_Kgrad if self.use_grad else self._eta_Kbase
        self.Kcov_cond_all[i] = cond_val
        self.eta_Kbase_all[i], self.eta_Kgrad_all[i] = self._eta_Kbase, self._eta_Kgrad
        self.vmin_init_all[i], self.vmin_req_grad_all[i] = self._vmin_init, self._vmin_req_grad
        if self.b_use_data_scl:
            self.xvec_rescaling_all[i] = self.DataScl.xvec_scale
        if surr_optz_info is not None:
            self.hp_optz_success[i] = surr_optz_info["hp_optz_success"]
            self.hp_optz_iter_mean[i] = surr_optz_info["hp_optz_iter_mean"]
            self.hp_optz_iter_max[i] = surr_optz_info["hp_optz_iter_max"]

    def set_hp_from_idx(self, i_optz):
        vf = None if np.isnan(self.hp_var_fval_all[i_optz]) else self.hp_var_fval_all[i_optz]
        vg = None if np.isnan(self.hp_var_fgrad_all[i_optz]) else self.hp_var_fgrad_all[i_optz]
        kh = None if np.isnan(self.hp_kernel_all[i_optz]) else self.hp_kernel_all[i_optz]
        self.hp_vals = self.make_hp_class(self.hp_beta_all[i_optz, :], self.hp_theta_all[i_optz, :], kh,
                                          self.hp_varK_all[i_optz], vf, vg)

    def set_hpara(self, method2set_hp, i_optz, hp_vals=None, calc_cond=False):
        """gpgradpy/src/GaussianProcess.py:365-395."""
        assert type(method2set_hp) is str, "method2set_hp must be a string"
        if method2set_hp == "stored":
            assert i_optz >= 0
            self.set_hp_from_idx(i_optz)
        elif method2set_hp == "optz":
            self.optz_hp(i_optz)
        elif method2set_hp == "current":
            assert i_optz > 0
            assert self.hp_vals is not None, "Cannot use current hp_vals if they have not been set yet"
        elif method2set_hp == "set":
            assert hp_vals is not None, 'If method2set_hp == "set", then the class hp_vals must be provided'
            self.hp_vals = hp_vals
        else:
            raise Exception(f"Unknown method to set GP hp: method2set_hp = {method2set_hp}")
        self.setup_eval_model(calc_cond=calc_cond)

    # ------------------------------------------------------------------ posterior (eval/GpEvalModel.py)
    def setup_eval_model(self, calc_cond=False):
        """Factor K (varK := 1) once and keep it on the device with w = L^-1 P^-1 (y - H beta)."""
        self._ensure_device()
        self._hp_vals_model_setup = copy.copy(self.hp_vals)
        hp = self.hp_vals
        noise = self.calc_noise_vec(hp)   # NOT divided by varK: the reference sets varK = 1 first (kernel/Kernel.py:196-197,218)
        noise = None if not np.any(noise) else noise
        beta = float(np.atleast_1d(hp.beta)[0])
        eta = self._etaK
        if not self.cond_eta_is_const:   # variable nugget: Gershgorin row sums with varK := 1 (kernel/Kernel.py:196-197)
            eta = self._variable_eta(np.asarray(hp.theta, dtype=float), None if noise is None else bk.to_dev(noise),
                                     kernel=self._kern(hp))[0]
        self._pred = bk.predict_setup(self._X_dev, self._y_dev, np.asarray(hp.theta, dtype=float), beta,
                                      n_g=self.n_grad, slot=self._slot_dev, noise=noise, mode=self._mode,
                                      eta=eta, kernel=self._kern(hp))
        self.data_vec = self._y_host
        self.etaK_eval = eta
        self.condK = None
        if calc_cond:
            self.condK = self.calc_all_K_w_chofac(None, hp, b_normlz_w_varK=True, calc_chofac=False, calc_cond=True)[4]
        good = int(self._pred.info.item()) == 0
        if self.condK is not None and self.wellcond_mtd != "precon" and self.condK > self.cond_max_abs:
            good = False          # the reference does not attempt the factorisation then (kernel/Kernel.py:282-283)
        self.KernEta_chofac = self._pred if good else None
        self.invKernEta_fdiff = DeviceMatrix(self._pred.alpha) if good else None

    def _test_points(self, x2model_in, squeeze_nx=False):
        """x2model_in as a [nx, dim] array, with the checks eval_model and its variants share (eval/GpEvalModel.py)."""
        x = np.asarray(x2model_in, dtype=float)
        if x.ndim == 1:
            x = x[None, :]
        elif x.ndim != 2:
            raise Exception(f"x2model_in should be a 2d array but it has shape {x.shape}")
        if squeeze_nx:
            assert x.shape[0] == 1, "If squeeze_nx is True, then x_acq must only have one point"
        if not (self.hp_vals == self._hp_vals_model_setup):
            raise Exception("Cannot change hp_vals between calling setup_eval_model() and eval_model()")
        return x

    def eval_model(self, x2model_in, calc_grad=False, calc_hess=False, squeeze_nx=False):
        """(mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2) -- eval/GpEvalModel.py:59-198.  calc_grad adds d mu / d x and
        d sig / d x [nx, dim] (:170-173, 319-354); calc_hess adds the Hessians [1, dim, dim] for ONE point per call,
        like the reference (:175-180, 356-382)."""
        assert self.KernEta_chofac is not None, "To evaluate the surr the Cholesky decomposition is required"
        if calc_hess:
            assert calc_grad, "To return the hessian calc_grad must also be set to True"
        x = self._test_points(x2model_in, squeeze_nx)
        if self.b_use_data_scl:
            x = self.DataScl.x_init_2_scl(x)
        dmudx = dsigdx = d2mudx2 = d2sigdx2 = None
        if calc_hess:
            assert x.shape[0] == 1, "calc_hess can only be used on one point per call"
            varK = float(self.hp_vals.varK)
            mu, sig, sig2, dmudx, dsigdx, h3, nneg = bk.predict_hess(self._pred, x[0], varK)
            dmudx, dsigdx, h3 = dmudx.cpu().numpy()[None, :], dsigdx.cpu().numpy()[None, :], h3.cpu().numpy()
            d2mudx2 = h3[0][None, :, :]
            d2sigdx2 = _d2sigdx2(h3[None], sig.cpu().numpy(), dsigdx, varK)
        elif calc_grad:
            mu, sig, sig2, dmudx, dsigdx, nneg = bk.predict_grad(self._pred, x, float(self.hp_vals.varK))
            dmudx, dsigdx = dmudx.cpu().numpy(), dsigdx.cpu().numpy()
        else:
            mu, sig, sig2, nneg = bk.predict(self._pred, x, float(self.hp_vals.varK))
        mu, sig = mu.cpu().numpy(), sig.cpu().numpy()
        n_bad = int(nneg.item())
        assert n_bad == 0, ("The variance of the surr should be non-negative but min(sig2_wo_sigK) = "
                            f"{float(sig2.min().item())}")
        if self.b_use_data_scl:
            mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2 = self.data_scl_2_init(mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2)
        if squeeze_nx:
            mu, sig = mu[0], sig[0]
            if calc_grad:
                dmudx, dsigdx = dmudx[0, :], dsigdx[0, :]
            if calc_hess:
                d2mudx2, d2sigdx2 = d2mudx2[0, :, :], d2sigdx2[0, :, :]
        return mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2


    def eval_model_hess_batch(self, x2model_in):
        """(mu, sig, dmudx, dsigdx, d2mudx2 [nx, dim, dim], d2sigdx2 [nx, dim, dim]) at every row of x2model_in in one
        chunked pass: what stacking eval_model(x[i:i+1], calc_grad=True, calc_hess=True) over i gives, for an optimiser
        that takes Newton or trust-region steps on the surrogate from many starts at once.  Same guards as eval_model;
        d2sigdx2 is NaN at a point where sig = 0 (eval/GpEvalModel.py:374-375)."""
        assert self.KernEta_chofac is not None, "To evaluate the surr the Cholesky decomposition is required"
        x = self._test_points(x2model_in)
        if self.b_use_data_scl:
            x = self.DataScl.x_init_2_scl(x)
        varK = float(self.hp_vals.varK)
        mu, sig, sig2, dmudx, dsigdx, h3, nneg = bk.predict_hess_batch(self._pred, x, varK)
        mu, sig, dmudx, dsigdx, h3 = (t.cpu().numpy() for t in (mu, sig, dmudx, dsigdx, h3))
        d2mudx2 = h3[:, 0]
        d2sigdx2 = _d2sigdx2(h3, sig, dsigdx, varK)
        assert int(nneg.item()) == 0, ("The variance of the surr should be non-negative but min(sig2_wo_sigK) = "
                                       f"{float(sig2.min().item())}")
        if self.b_use_data_scl:
            mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2 = self.data_scl_2_init(mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2)
        return mu, sig, dmudx, dsigdx, d2mudx2, d2sigdx2

    def eval_model_var(self, x2model_in, calc_grad=False, calc_hess=False, squeeze_nx=False):
        """(sig2, dsig2dx, None) -- eval/GpEvalModel.py:200-317: posterior variance varK (1 - k*^T K^-1 k*) and its
        x-gradient -2 varK (dk*/dx)^T K^-1 k* = 2 sig dsig/dx.  Like the reference: no rescale modes, no Hessian."""
        assert self.KernEta_chofac is not None, "To evaluate the surr the Cholesky decomposition is required"
        if self.b_use_data_scl:
            raise Exception("The method eval_model_var() is not setup for cases where data must be rescaled")
        if calc_hess:
            assert calc_grad, "To return the hessian calc_grad must also be set to True"
            raise Exception("Must add method to calculate d2sig2dx2")          # the reference's own message (:303)
        x = self._test_points(x2model_in, squeeze_nx)
        varK = float(self.hp_vals.varK)
        dsig2dx = None
        if calc_grad:
            _, sig, sig2, _, dsig, nneg = bk.predict_grad(self._pred, x, varK)
            dsig2dx = (2.0 * sig[:, None] * dsig).cpu().numpy()
        else:
            _, sig, sig2, nneg = bk.predict(self._pred, x, varK)
        sig2 = varK * sig2.cpu().numpy()
        assert int(nneg.item()) == 0, f"The variance of the surr should be non-negative but min(sig2) = {sig2.min()}"
        if squeeze_nx:
            sig2 = sig2[0]
            if calc_grad:
                dsig2dx = dsig2dx[0, :]
        return sig2, dsig2dx, None


def _d2sigdx2(h3, sig, dsigdx, varK):
    """d2sig/dx2 [nx, d, d] from the Hessian slabs h3 [nx, 3, d, d] (d2mu, term1, term2), sig [nx] and dsigdx [nx, d]
    (eval/GpEvalModel.py:366-375): d2sig2 = -2 varK (term1 + term2), d2sig = (d2sig2 - 2 dsig dsig^T) / (2 sig), NaN where
    sig = 0."""
    d2sig2 = -2.0 * varK * (h3[:, 1] + h3[:, 2])
    s = np.where(sig == 0, np.nan, sig)
    return (d2sig2 - 2.0 * (dsigdx[:, :, None] * dsigdx[:, None, :])) / (2.0 * s[:, None, None])


class _DeviceRtensor:
    """Stand-in for the reference's cached distance tensor R[d, n, n] (never materialised on the CUDA path)."""

    def __init__(self, n, d):
        self.shape = (d, n, n)

    def __repr__(self):
        return f"<Rtensor placeholder {self.shape}: the CUDA builder reads X directly>"


def _pdist(x):
    from scipy.spatial.distance import pdist
    return pdist(x)
