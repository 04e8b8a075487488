"""Thin PyTorch-side plumbing over the C ABI: device buffers, streams and workspace management.

Every function here hands raw device pointers to libgegp.so; no arithmetic of the hot path is done in
Python/PyTorch, and there is no CPU fallback (a missing CUDA device or library raises).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L

F64 = torch.float64


def device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("gpgradpy_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def to_dev(a, dtype=F64):
    """Host array / tensor -> contiguous device tensor (no copy if already there)."""
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        return a.to(device=device(), dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(device())


def pinned_like(buf, a):
    """Copy the host array `a` into a page-locked fp64 staging tensor (re-using `buf` when the shape matches)."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    if buf is None or tuple(buf.shape) != a.shape:
        buf = torch.empty(a.shape, dtype=F64, pin_memory=True)
    buf.copy_(torch.from_numpy(a))
    return buf


def _p(t) -> int:
    return 0 if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed with code {rc} (negative: bad argument index / -1000-cudaError)")


def dmma_peak_tflops(reps: int = 3) -> float:
    """gegp_dmma_peak: issue peak of DMMA.8x8x4 on the current device in TFLOP/s (the fp64 roofline denominator)."""
    lib = L.load()
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    scratch = torch.empty(512 * sms, dtype=F64, device=device())
    out = C.c_double(0.0)
    torch.cuda.synchronize()
    rc = lib.gegp_dmma_peak(_p(scratch), scratch.numel(), int(reps), C.byref(out), _stream())
    _check(rc, "gegp_dmma_peak")
    return float(out.value)


def _kern(kernel):
    """kernel = None | name | id | (name-or-id, hp)  ->  (GEGP_KERNEL_* id, hp float)."""
    if kernel is None:
        return L.KERNEL_SQEXP, 0.0
    hp = 0.0
    if isinstance(kernel, (tuple, list)):
        kernel, hp = kernel[0], (0.0 if kernel[1] is None else float(np.ravel(kernel[1])[0]))
    kid = L.KERNEL_IDS[kernel] if isinstance(kernel, str) else int(kernel)
    return kid, hp


def ld_of(N: int) -> int:
    return int(L.load().gegp_ld(N))


def slot_from_mask(mask, n):
    """bvec_use_grad (bool[n]) -> (slot int32[n] device tensor or None, n_g)."""
    if mask is None:
        return None, n
    m = np.asarray(mask, dtype=bool)
    assert m.size == n
    slot = np.where(m, np.cumsum(m) - 1, -1).astype(np.int32)
    ng = int(m.sum())
    if ng == n:
        return None, n
    return torch.as_tensor(slot).to(device()), ng


_ws_cache: dict = {}


def workspace(nbytes: int) -> torch.Tensor:
    """Grow-only byte workspace per device (torch caching allocator owns the memory)."""
    key = torch.cuda.current_device()
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        _ws_cache.pop(key, None)
        buf = None
        buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device())
        _ws_cache[key] = buf
    return buf


def free_workspace():
    _graph_cache.clear()
    _ws_cache.clear()


def build_cov(X, theta, *, n_g=None, slot=None, noise=None, mode=L.MODE_BASE, eta=0.0, varK=1.0, uplo=0, out=None,
              kernel=None):
    """gegp_build_cov -> (K [N, N] strided view over an [N, ld] buffer, p [2N] or None)."""
    lib = L.load()
    X = to_dev(X)
    n, d = X.shape
    n_g = n if n_g is None else n_g
    N = n + n_g * d
    theta = to_dev(theta)
    noise = to_dev(noise)
    ld = ld_of(N)
    if out is None:
        out = torch.empty((N, ld), dtype=F64, device=device())
    p = torch.empty(2 * N, dtype=F64, device=device()) if mode == L.MODE_PRECON else None
    kid, khp = _kern(kernel)
    rc = lib.gegp_build_cov(n, n_g, d, _p(X), _p(slot), _p(theta), kid, khp, _p(noise), mode, float(eta), float(varK),
                            _p(out), out.stride(0), _p(p), int(uplo), _stream())
    _check(rc, "gegp_build_cov")
    return out[:, :N], p


def cross_cov(X, Xs, theta, *, n_g=None, slot=None, pinv=None, kernel=None):
    lib = L.load()
    X, Xs, theta, pinv = to_dev(X), to_dev(Xs), to_dev(theta), to_dev(pinv)
    n, d = X.shape
    n_g = n if n_g is None else n_g
    N = n + n_g * d
    nx = Xs.shape[0]
    ld = ld_of(N)
    out = torch.empty((nx, ld), dtype=F64, device=device())
    kid, khp = _kern(kernel)
    rc = lib.gegp_cross_cov(n, n_g, d, _p(X), _p(slot), _p(Xs), nx, _p(theta), kid, khp, _p(pinv), _p(out), ld, _stream())
    _check(rc, "gegp_cross_cov")
    return out[:, :N]


def dinv_buffer(N: int) -> torch.Tensor:
    """Device buffer for the inverse-transposed diagonal blocks that belong to a factor of order N."""
    return torch.empty(int(L.load().gegp_dinv_doubles(N)), dtype=F64, device=device())


def potrf(A: torch.Tensor, N: int, n_extra: int = 0, dinv: torch.Tensor | None = None):
    """In-place trapezoid Cholesky of A[(N+n_extra), ld]; returns (device info int tensor, dinv blocks)."""
    lib = L.load()
    assert A.is_cuda and A.dtype == F64 and A.stride(1) == 1 and A.shape[0] >= N + n_extra
    info = torch.zeros(1, dtype=torch.int32, device=A.device)
    if dinv is None:
        dinv = dinv_buffer(N)
    rc = lib.gegp_potrf(N, n_extra, _p(A), A.stride(0), _p(dinv), _p(info), _stream())
    _check(rc, "gegp_potrf")
    return info, dinv


def trsm_rows(Lfac: torch.Tensor, dinv: torch.Tensor, N: int, B: torch.Tensor):
    lib = L.load()
    rc = lib.gegp_trsm_rows(N, _p(Lfac), Lfac.stride(0), _p(dinv), _p(B), B.stride(0), B.shape[0], _stream())
    _check(rc, "gegp_trsm_rows")
    return B


def potri(Lfac: torch.Tensor, dinv: torch.Tensor, N: int, U: torch.Tensor | None = None,
          Kinv: torch.Tensor | None = None):
    """Explicit inverse from the factor -> (U = L^-T in its upper triangle, Kinv full symmetric), [N, ld] buffers."""
    lib = L.load()
    ld = ld_of(N)
    if U is None:
        U = torch.empty((N, ld), dtype=F64, device=device())
    if Kinv is None:
        Kinv = torch.empty((N, ld), dtype=F64, device=device())
    rc = lib.gegp_potri(N, _p(Lfac), Lfac.stride(0), _p(dinv), _p(U), U.stride(0), _p(Kinv), Kinv.stride(0), _stream())
    _check(rc, "gegp_potri")
    return U, Kinv


def dgemm(A: torch.Tensor, B: torch.Tensor, C: torch.Tensor, *, transb: bool, alpha=1.0, beta=0.0):
    """C = alpha * A @ (B.T if transb else B) + beta * C on the DMMA engine (row-major 2-D device tensors)."""
    lib = L.load()
    M, K = A.shape
    N = B.shape[0] if transb else B.shape[1]
    assert (B.shape[1] if transb else B.shape[0]) == K and tuple(C.shape) == (M, N)
    rc = lib.gegp_dgemm(int(transb), M, N, K, float(alpha), _p(A), A.stride(0), _p(B), B.stride(0), float(beta), _p(C),
                        C.stride(0), _stream())
    _check(rc, "gegp_dgemm")
    return C


def _lml_workspace(lib, op, n, n_g, d, B, max_ws_bytes):
    """Workspace for B candidates (or the largest chunk of them that fits); cudaMemGetInfo only when it must grow."""
    need_all = int(lib.gegp_workspace_bytes(op, n, n_g, d, B)) + 4 * B + 256
    cached = _ws_cache.get(torch.cuda.current_device())
    if cached is not None and cached.numel() >= need_all and (max_ws_bytes is None or need_all <= max_ws_bytes):
        return cached
    per1 = int(lib.gegp_workspace_bytes(op, n, n_g, d, 1))
    if max_ws_bytes is None:
        free, _total = torch.cuda.mem_get_info()
        max_ws_bytes = int(0.6 * (free + (cached.numel() if cached is not None else 0)))
    if per1 + 4096 + 4 * B > max_ws_bytes:
        raise MemoryError(f"one candidate of this size needs a {per1 / 2**30:.1f} GiB workspace (N = {n + n_g * d}, "
                          f"{'with' if op == L.OP_LML_GRAD else 'without'} gradient) but only {max_ws_bytes / 2**30:.1f} GiB "
                          "may be used on this device")
    chunk = max(1, min(B, (max_ws_bytes - 4096 - 4 * B) // per1))
    return workspace(int(lib.gegp_workspace_bytes(op, n, n_g, d, chunk)) + 4 * B + 256)


def lml_eval(X, y, theta_batch, *, n_g=None, slot=None, mode=L.MODE_PRECON, eta=0.0, noise=None, varK_batch=None,
             pnlt_grad=0.0, want_grad=True, want_alpha=False, max_ws_bytes=None, out=None, kernel=None, kernel_hp_batch=None):
    """gegp_lml_eval for B candidate rows -> (out [B, 9+d] device tensor, alpha [B, N] or None)."""
    lib = L.load()
    X, y = to_dev(X), to_dev(y)
    n, d = X.shape
    n_g = n if n_g is None else n_g
    N = n + n_g * d
    th = to_dev(theta_batch).reshape(-1, d)
    B = th.shape[0]
    noisy = noise is not None
    noise = to_dev(noise)
    vk = to_dev(varK_batch).reshape(-1) if noisy else None
    if noisy:
        assert vk.numel() == B
    if out is None:
        out = torch.empty((B, L.out_len(d)), dtype=F64, device=device())
    alpha = torch.empty((B, N), dtype=F64, device=device()) if want_alpha else None
    op = L.OP_LML_GRAD if want_grad else L.OP_LML
    ws = _lml_workspace(lib, op, n, n_g, d, B, max_ws_bytes)
    kid, khp = _kern(kernel)
    khp_dev = None
    if kid == L.KERNEL_RATQUAD:      # one alpha per candidate row (a scalar is broadcast)
        khp_dev = to_dev(kernel_hp_batch).reshape(-1) if kernel_hp_batch is not None else torch.full(
            (B,), khp, dtype=F64, device=device())
        assert khp_dev.numel() == B
    rc = lib.gegp_lml_eval(B, _p(th), _p(vk), kid, _p(khp_dev), n, n_g, d, _p(X), _p(slot), _p(y), _p(noise), int(mode),
                           float(eta), int(noisy), float(pnlt_grad), int(bool(want_grad)), _p(out), _p(alpha), _p(ws),
                           ws.numel(), _stream())
    _check(rc, "gegp_lml_eval")
    return out, alpha


class LmlGraph:
    """One captured CUDA graph of gegp_lml_eval for a fixed problem (data, shapes, mode, flags).

    The ~300 kernel launches of one evaluation are recorded once and replayed with new hyper-parameters, which
    are written into static device buffers before the replay.  Used for the optimiser's inner loop, where the
    same-shaped evaluation is repeated hundreds of times (optz/OptzLkd.py:249-270).
    """

    def __init__(self, X, y, B, *, n_g, slot, mode, eta, noise, noisy, pnlt_grad, want_grad, kernel=None):
        n, d = X.shape
        self.key_tensors = (X, y, slot, noise)          # keep the captured buffers alive
        self.theta = torch.empty((B, d), dtype=F64, device=device())
        self.varK = torch.ones(B, dtype=F64, device=device()) if noisy else None
        kid = _kern(kernel)[0]
        self.khp = torch.full((B,), 2.0, dtype=F64, device=device()) if kid == L.KERNEL_RATQUAD else None
        self.out = torch.empty((B, L.out_len(d)), dtype=F64, device=device())
        kw = dict(n_g=n_g, slot=slot, mode=mode, eta=eta, noise=noise if noisy else None, varK_batch=self.varK,
                  pnlt_grad=pnlt_grad, want_grad=want_grad, out=self.out, kernel=kid, kernel_hp_batch=self.khp)
        self.theta.fill_(1.0)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                   # warm-up: function attributes, tensor maps, workspace growth
            lml_eval(X, y, self.theta, **kw)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        L.profile_begin(False)
        with torch.cuda.graph(self.graph):
            lml_eval(X, y, self.theta, **kw)
        self.n_launches = L.profile_end()["launches"]          # kernels recorded in the graph
        self.ws = _ws_cache.get(torch.cuda.current_device())   # the captured workspace must stay allocated

    def __call__(self, theta_rows, varK_rows=None, khp_rows=None):
        src = theta_rows if isinstance(theta_rows, torch.Tensor) else torch.as_tensor(
            np.ascontiguousarray(theta_rows, dtype=np.float64))
        self.theta.copy_(src.reshape(self.theta.shape), non_blocking=True)
        if self.varK is not None:
            self.varK.copy_(torch.as_tensor(np.ascontiguousarray(varK_rows, dtype=np.float64)).reshape(-1))
        if self.khp is not None:
            self.khp.copy_(torch.as_tensor(np.ascontiguousarray(khp_rows, dtype=np.float64)).reshape(-1))
        self.graph.replay()
        replay_stats["replays"] += 1
        replay_stats["kernel_launches"] += self.n_launches
        return self.out


_graph_cache: dict = {}
replay_stats = {"replays": 0, "kernel_launches": 0}   # kernels launched through graph replays (bench.py reports them)


def lml_eval_graphed(X, y, theta_batch, *, n_g=None, slot=None, mode=L.MODE_PRECON, eta=0.0, noise=None,
                     varK_batch=None, pnlt_grad=0.0, want_grad=True, kernel=None, kernel_hp_batch=None):
    """Same result as lml_eval(...)[0], through a cached CUDA graph.  X, y, slot, noise must be device tensors that
    stay alive and unchanged in place between calls (the graph holds their addresses)."""
    n, d = X.shape
    n_g = n if n_g is None else n_g
    B = int(np.prod(theta_batch.shape)) // d
    noisy = noise is not None
    key = (torch.cuda.current_device(), X.data_ptr(), y.data_ptr(), _p(slot), _p(noise), n, n_g, d, B, int(mode),
           float(eta), float(pnlt_grad), bool(want_grad), noisy, _kern(kernel)[0])
    g = _graph_cache.get(key)
    ws_now = _ws_cache.get(torch.cuda.current_device())
    if g is not None and g.ws is not ws_now:   # the workspace was re-allocated since the capture
        g = None
    if g is None:
        if len(_graph_cache) >= 8:
            _graph_cache.clear()
        g = LmlGraph(X, y, B, n_g=n_g, slot=slot, mode=mode, eta=eta, noise=noise, noisy=noisy, pnlt_grad=pnlt_grad,
                     want_grad=want_grad, kernel=kernel)
        _graph_cache[key] = g
    khp = kernel_hp_batch
    if g.khp is not None and khp is None:
        khp = np.full(B, _kern(kernel)[1])
    return g(theta_batch, varK_batch, khp)


def free_graphs():
    _graph_cache.clear()


class PredictState:
    """Factor + solved residual row kept on the device between setup_eval_model and eval_model."""

    def __init__(self, A, dinv, p, info, alpha, n, n_g, d, N, X, slot, theta, mode, beta, kernel=(0, 0.0)):
        self.A, self.dinv, self.p, self.info, self.alpha = A, dinv, p, info, alpha
        self.n, self.n_g, self.d, self.N = n, n_g, d, N
        self.X, self.slot, self.theta, self.mode, self.beta = X, slot, theta, mode, beta
        self.kid, self.khp = kernel


def predict_setup(X, y, theta, beta, *, n_g=None, slot=None, noise=None, mode=L.MODE_PRECON, eta=0.0,
                  want_alpha=True, kernel=None) -> PredictState:
    lib = L.load()
    X, y, theta, noise = to_dev(X), to_dev(y), to_dev(theta), to_dev(noise)
    n, d = X.shape
    n_g = n if n_g is None else n_g
    N = n + n_g * d
    ld = ld_of(N)
    A = torch.empty((N + 1, ld), dtype=F64, device=device())
    dinv = dinv_buffer(N)
    p = torch.empty(2 * N, dtype=F64, device=device())
    info = torch.zeros(1, dtype=torch.int32, device=device())
    alpha = torch.empty(N, dtype=F64, device=device()) if want_alpha else None
    kid, khp = _kern(kernel)
    rc = lib.gegp_predict_setup(n, n_g, d, _p(X), _p(slot), _p(theta), kid, khp, _p(noise), int(mode), float(eta), _p(y),
                                float(beta), _p(A), ld, _p(dinv), _p(p), _p(alpha), _p(info), _stream())
    _check(rc, "gegp_predict_setup")
    return PredictState(A, dinv, p, info, alpha, n, n_g, d, N, X, slot, theta, mode, float(beta), (kid, khp))


def _outputs(*shapes):
    """Uninitialised float64 device tensors of the given shapes, then the zeroed n_negative counter."""
    dev = device()
    return [torch.empty(s, dtype=F64, device=dev) for s in shapes] + [torch.zeros(1, dtype=torch.int32, device=dev)]


def _chunk_workspace(nx: int, per_x: int, chunk_bytes: int, fixed: int = 0):
    """(workspace, its size in bytes) for chunks of as many of the nx points as chunk_bytes hold, at least one."""
    cx = max(1, min(nx, (chunk_bytes - fixed) // per_x))
    nbytes = fixed + cx * per_x
    return workspace(nbytes), nbytes


def predict(st: PredictState, Xs, varK: float, *, chunk_bytes: int = 1 << 30):
    """gegp_predict -> (mu, sig, sig2, n_negative) device tensors."""
    lib = L.load()
    Xs = to_dev(Xs)
    nx = Xs.shape[0]
    mu, sig, sig2, nneg = _outputs(nx, nx, nx)
    ws, nbytes = _chunk_workspace(nx, ld_of(st.N) * 8, chunk_bytes)
    rc = lib.gegp_predict(st.n, st.n_g, st.d, _p(st.X), _p(st.slot), _p(st.theta), st.kid, st.khp, _p(st.A), st.A.stride(0), _p(st.dinv),
                          _p(st.p), int(st.mode), st.beta, float(varK), _p(Xs), nx, _p(mu), _p(sig), _p(sig2), _p(nneg), _p(ws),
                          nbytes, _stream())
    _check(rc, "gegp_predict")
    return mu, sig, sig2, nneg


def predict_grad(st: PredictState, Xs, varK: float, *, chunk_bytes: int = 1 << 30):
    """gegp_predict_grad -> (mu, sig, sig2, dmudx [nx, d], dsigdx [nx, d], n_negative) device tensors."""
    lib = L.load()
    Xs = to_dev(Xs)
    nx, d = Xs.shape[0], st.d
    mu, sig, sig2, dmu, dsg, nneg = _outputs(nx, nx, nx, (nx, d), (nx, d))
    ws, nbytes = _chunk_workspace(nx, (d + 1) * ld_of(st.N) * 8, chunk_bytes)
    rc = lib.gegp_predict_grad(st.n, st.n_g, st.d, _p(st.X), _p(st.slot), _p(st.theta), st.kid, st.khp, _p(st.A), st.A.stride(0),
                               _p(st.dinv), _p(st.p), int(st.mode), st.beta, float(varK), _p(Xs), nx, _p(mu), _p(sig),
                               _p(sig2), _p(dmu), _p(dsg), _p(nneg), _p(ws), nbytes, _stream())
    _check(rc, "gegp_predict_grad")
    return mu, sig, sig2, dmu, dsg, nneg


def predict_hess(st: PredictState, xs, varK: float):
    """gegp_predict_hess at ONE test point -> (mu, sig, sig2, dmudx [d], dsigdx [d], hess3 [3, d, d], n_negative)."""
    lib = L.load()
    xs = to_dev(xs).reshape(-1)
    d = st.d
    assert xs.numel() == d and st.alpha is not None
    mu, sig, sig2, dmu, dsg, h3, nneg = _outputs(1, 1, 1, d, d, (3, d, d))
    nbytes = (d + 2) * ld_of(st.N) * 8
    ws = workspace(nbytes)
    rc = lib.gegp_predict_hess(st.n, st.n_g, st.d, _p(st.X), _p(st.slot), _p(st.theta), st.kid, st.khp, _p(st.A), st.A.stride(0),
                               _p(st.dinv), _p(st.p), _p(st.alpha), int(st.mode), st.beta, float(varK), _p(xs), _p(mu),
                               _p(sig), _p(sig2), _p(dmu), _p(dsg), _p(h3), _p(nneg), _p(ws), nbytes, _stream())
    _check(rc, "gegp_predict_hess")
    return mu, sig, sig2, dmu, dsg, h3, nneg


def predict_hess_batch_bytes(N: int, d: int, nx: int) -> int:
    """Workspace of gegp_predict_hess_batch for chunks of nx points (include/gegp.h)."""
    return L.load().gegp_dinv_doubles(N) * 8 + nx * ((d + 1) * ld_of(N) + 128) * 8


def predict_hess_batch(st: PredictState, Xs, varK: float, *, chunk_bytes: int = 1 << 30):
    """gegp_predict_hess_batch at nx points -> (mu, sig, sig2, dmudx [nx, d], dsigdx [nx, d], hess3 [nx, 3, d, d],
    n_negative) device tensors; chunks of as many points as chunk_bytes of workspace hold (at least one)."""
    lib = L.load()
    Xs = to_dev(Xs)
    nx, d = Xs.shape[0], st.d
    assert Xs.ndim == 2 and Xs.shape[1] == d and st.alpha is not None
    out = _outputs(nx, nx, nx, (nx, d), (nx, d), (nx, 3, d, d))
    if nx == 0:
        return tuple(out)
    mu, sig, sig2, dmu, dsg, h3, nneg = out
    fixed = predict_hess_batch_bytes(st.N, d, 0)
    ws, nbytes = _chunk_workspace(nx, predict_hess_batch_bytes(st.N, d, 1) - fixed, chunk_bytes, fixed)
    rc = lib.gegp_predict_hess_batch(st.n, st.n_g, st.d, _p(st.X), _p(st.slot), _p(st.theta), st.kid, st.khp, _p(st.A),
                                     st.A.stride(0), _p(st.dinv), _p(st.p), _p(st.alpha), int(st.mode), st.beta, float(varK),
                                     _p(Xs), nx, _p(mu), _p(sig), _p(sig2), _p(dmu), _p(dsg), _p(h3), _p(nneg), _p(ws), nbytes,
                                     _stream())
    _check(rc, "gegp_predict_hess_batch")
    return mu, sig, sig2, dmu, dsg, h3, nneg


# ----------------------------------------------------------------------------------------------------------------
# 2-norm condition number and its hyper-parameter gradient (kernel/Kernel.py:240,280; optz/GpHparaCon.py:161-235)
# ----------------------------------------------------------------------------------------------------------------
def symv(M: torch.Tensor, x: torch.Tensor, y: torch.Tensor, N: int):
    """y[:N] = M[:N, :N] @ x[:N] (gegp_symv; M is an [N, ld] row-major device buffer)."""
    rc = L.load().gegp_symv(N, _p(M), M.stride(0), _p(x), _p(y), _stream())
    _check(rc, "gegp_symv")
    return y


def row_abs_sum(M: torch.Tensor, N: int) -> torch.Tensor:
    """Gershgorin row sums sum_c |M[r, c]| of an [N, ld] device buffer (gegp_row_abs_sum)."""
    out = torch.empty(N, dtype=F64, device=M.device)
    rc = L.load().gegp_row_abs_sum(N, _p(M), M.stride(0), _p(out), _stream())
    _check(rc, "gegp_row_abs_sum")
    return out


def fro_norm(M: torch.Tensor, N: int) -> float:
    """Frobenius norm of M[:N, :N] (gegp_row_sq_sum, the N row sums added on the host)."""
    out = torch.empty(N, dtype=F64, device=M.device)
    rc = L.load().gegp_row_sq_sum(N, _p(M), M.stride(0), _p(out), _stream())
    _check(rc, "gegp_row_sq_sum")
    return float(np.sqrt(np.sum(out.cpu().numpy())))


def weighted_grad(X, theta, W: torch.Tensor, *, n_g=None, slot=None, eta=0.0, noisy=False, varK=1.0, kernel=None):
    """gegp_weighted_grad: sum(W .* dKcov/dhp) for every hyper-parameter (base mode) -> device row (GEGP_OUT_* layout)."""
    lib = L.load()
    X, theta = to_dev(X), to_dev(theta)
    n, d = X.shape
    n_g = n if n_g is None else n_g
    N = n + n_g * d
    out = torch.zeros(L.out_len(d), dtype=F64, device=device())
    vk = to_dev(np.array([float(varK)]))
    nbytes = int(lib.gegp_quad_grad_work_bytes(n, n_g, d)) + 8 * (N + 2)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device())
    kid, khp = _kern(kernel)
    rc = lib.gegp_weighted_grad(n, n_g, d, _p(X), _p(slot), _p(theta), kid, khp, _p(W), W.stride(0), L.MODE_BASE, float(eta),
                                int(bool(noisy)), _p(vk), _p(out), _p(ws), nbytes, _stream())
    _check(rc, "gegp_weighted_grad")
    return out


def cond_fro(Kfull: torch.Tensor, Kinv: torch.Tensor, N: int, want_weight: bool):
    """Frobenius condition number |K|_F |K^-1|_F and, if asked, the weight matrix of its gradient
    d cond / dK = frac K - K^-3 / frac, frac = |K^-1|_F / |K|_F  (optz/GpHparaCon.py:237-261); the two matrix
    products run on the DMMA GEMM engine (K^-1 is symmetric, so K^-1 K^-1 = K^-1 (K^-1)^T)."""
    nk, ni = fro_norm(Kfull, N), fro_norm(Kinv, N)
    cond = nk * ni
    if not want_weight:
        return cond, None
    ld = ld_of(N)
    K2 = torch.empty((N, ld), dtype=F64, device=Kinv.device)
    K3 = torch.empty((N, ld), dtype=F64, device=Kinv.device)
    dgemm(Kinv[:, :N], Kinv[:, :N], K2[:, :N], transb=True)
    frac = ni / nk
    K3[:, :N].copy_(Kfull[:, :N])                                            # W = frac K - (K^-2 K^-1) / frac, in one GEMM
    dgemm(K2[:, :N], Kinv[:, :N], K3[:, :N], transb=True, alpha=-1.0 / frac, beta=frac)
    return cond, K3


def extreme_eig(M: torch.Tensor, N: int, *, k: int = 40, tol: float = 1e-12, max_cycles: int = 12, v0=None,
                chunk: int = 8):
    """Largest eigenpair of the symmetric device matrix M[:N, :N]: restarted Lanczos with full re-orthogonalisation.

    The matrix-vector products and the orthogonalisation run on the device (gegp_symv, gegp_lanczos_step,
    gegp_lincomb); every `chunk` steps the small tridiagonal eigenproblem is solved on the host and the iteration
    stops as soon as the residual estimate |beta_j s_j| <= tol |lambda| (or an invariant subspace is hit); after k steps
    it restarts from the Ritz vector.  `v0` (device vector) warm-starts the iteration -- e.g. the eigenvector of the
    previous optimiser iterate; it is mixed with the fixed pseudo-random start vector so that no eigen-direction is
    ever excluded.  Returns (lambda, v [N] device tensor with |v| = 1, relative residual estimate, matvecs).
    This is the one-candidate case of extreme_eig_batch."""
    lam, v, resid, matvecs = extreme_eig_batch(M[None], N, k=k, tol=tol, max_cycles=max_cycles, v0=[v0], chunk=chunk)
    return lam[0], v[0], resid[0], matvecs[0]


def _tridiag_ritz(a, b, j):
    """Largest Ritz pair of the j-step Lanczos tridiagonal (a, b) -> (basis size m, lambda, s, relative residual)."""
    from scipy.linalg import eigh_tridiagonal
    scale = max(float(np.max(np.abs(a[:j]))), 1e-300)
    m = j
    for q in range(j):            # breakdown: an invariant subspace was found after q + 1 steps
        if not (b[q] > 1e-14 * scale):
            m = q + 1
            break
    evals, evecs = eigh_tridiagonal(a[:m], b[:m - 1]) if m > 1 else (a[:1], np.ones((1, 1)))
    lam, s_vec = float(evals[-1]), evecs[:, -1]
    return m, lam, s_vec, abs(float(b[m - 1]) * float(s_vec[-1])) / max(abs(lam), 1e-300)


def extreme_eig_batch(M: torch.Tensor, N: int, *, k: int = 40, tol: float = 1e-12, max_cycles: int = 12, v0=None,
                      chunk: int = 8, rows=None):
    """extreme_eig for B symmetric matrices at once.  M: [B, >= N, ld] device view with unit column stride (e.g. the
    candidates' buffers in a gegp_lml_eval workspace); v0: None or a list of B warm-start vectors (entries may be None).

    Every candidate still iterating is at the same Lanczos step within a cycle, so each step is one gegp_symv_batch and
    one gegp_lanczos_step_batch over those candidates; after each `chunk` steps the alphas and betas of all candidates
    come to the host in one copy, and each candidate takes its own converge / restart / breakdown decision exactly as
    extreme_eig does alone.  Converged candidates leave the launches through the active list.  A candidate's result is
    bit-identical to extreme_eig on its matrix alone.  rows: the candidates to iterate (default all); the others are
    skipped and get None.  -> (lambdas, vectors [N] device tensors, residuals, matvecs), lists of B."""
    lib = L.load()
    B = M.shape[0]
    assert M.stride(-1) == 1 and B >= 1
    k = int(max(2, min(k, N, 200)))
    ld = ld_of(N)
    dev = device()
    st = _stream()
    ldm, sM = M.stride(-2), (M.stride(0) if B > 1 else 0)
    V = torch.zeros((B, k + 1, ld), dtype=F64, device=dev)
    w = torch.zeros((B, ld), dtype=F64, device=dev)
    r = torch.zeros((B, ld), dtype=F64, device=dev)
    ab = torch.zeros((B, 2, k), dtype=F64, device=dev)     # alpha_z, beta_z: one device-to-host copy per chunk
    coef = torch.zeros((B, k), dtype=F64, device=dev)
    ks = torch.ones(B, dtype=torch.int32, device=dev)
    rnd = to_dev(np.random.default_rng(12345).standard_normal(N))   # fixed: deterministic results
    V[:, 0, :N] = rnd
    for c, v in enumerate(v0 if v0 is not None else []):
        if v is not None:
            V[c, 0, :N] = v[:N] + (1e-3 / np.sqrt(N)) * rnd
    sV = (k + 1) * ld

    def lincomb(rows, kmax):
        act = None if len(rows) == B else torch.as_tensor(np.asarray(rows, dtype=np.int32)).to(dev)
        rc = lib.gegp_lincomb_batch(len(rows), N, kmax, _p(ks), _p(V), ld, sV, _p(coef), k, _p(r), ld, _p(act), st)
        _check(rc, "gegp_lincomb_batch")
        idx = torch.as_tensor(rows, dtype=torch.long, device=dev)
        V[idx, 0] = r[idx]

    alive = list(range(B)) if rows is None else sorted(set(int(c) for c in rows))
    todo = set(alive)
    lam, resid, matvecs = [float("nan")] * B, [float("inf")] * B, [0] * B
    if not alive:
        return [None] * B, [None] * B, [None] * B, [None] * B
    coef[:, 0] = 1.0
    lincomb(alive, 1)                                                       # normalise the start vectors
    for _cycle in range(max_cycles):
        if not alive:
            break
        j, active = 0, list(alive)
        while j < k and active:
            act = None if len(active) == B else torch.as_tensor(np.asarray(active, dtype=np.int32)).to(dev)
            jn = min(k, j + chunk)
            for jj in range(j, jn):
                rc = lib.gegp_symv_batch(len(active), N, _p(M), ldm, sM, _p(V[0, jj]), sV, _p(w), ld, _p(act), st)
                _check(rc, "gegp_symv_batch")
                rc = lib.gegp_lanczos_step_batch(len(active), N, jj, _p(V), ld, sV, _p(w), ld, _p(ab[0, 0]), _p(ab[0, 1]),
                                                 2 * k, _p(act), st)
                _check(rc, "gegp_lanczos_step_batch")
            h = ab.cpu().numpy()
            finished, coef_h, ks_h, kmax = [], np.zeros((B, k)), np.ones(B, dtype=np.int32), 1
            for c in active:
                matvecs[c] += jn - j
                m, lam[c], s_vec, resid[c] = _tridiag_ritz(h[c, 0], h[c, 1], jn)
                done = resid[c] <= tol or m < jn
                if done or jn == k:            # restart (or finish) from the Ritz vector
                    finished.append(c)
                    coef_h[c, :m], ks_h[c], kmax = s_vec, m, max(kmax, m)
                    if done:
                        alive.remove(c)
            j = jn
            if finished:
                coef.copy_(torch.from_numpy(coef_h))
                ks.copy_(torch.from_numpy(ks_h))
                lincomb(finished, kmax)
                active = [c for c in active if c not in finished]
    return ([lam[c] if c in todo else None for c in range(B)], [r[c, :N].clone() if c in todo else None for c in range(B)],
            [resid[c] if c in todo else None for c in range(B)], [matvecs[c] if c in todo else None for c in range(B)])


def cond2(Kfull: torch.Tensor, Kinv: torch.Tensor, N: int, *, tol: float = 1e-12, warm=None):
    """kappa_2 = lambda_max(K) * lambda_max(K^-1) with both extreme eigenvectors.  `warm`: a previous result of this
    function for a nearby matrix of the same order (its eigenvectors warm-start the two iterations).
    -> dict(cond, lam_max, lam_min, v_max, v_min, resid_max, resid_min, cycles = matvecs of the two iterations)."""
    return cond2_batch(Kfull[None], Kinv[None], N, tol=tol, warm=[warm])[0]


def cond2_batch(Kfull: torch.Tensor, Kinv: torch.Tensor, N: int, *, tol: float = 1e-12, warm=None, rows=None):
    """cond2 for B candidates: Kfull, Kinv [B, >= N, ld] device views (e.g. the U and Kinv buffers of a gegp_lml_eval
    workspace, lml_views_batch); warm: None or a list of B earlier results (entries may be None); rows: the candidates
    to evaluate (default all; the others get None).  -> list of B dicts, each bit-identical to cond2 on that candidate
    alone."""
    B = Kfull.shape[0]
    warm = warm if warm is not None else [None] * B
    ok = [wm is not None and wm.get("v_max") is not None and wm["v_max"].numel() == N for wm in warm]
    lmax, vmax, r1, c1 = extreme_eig_batch(Kfull, N, tol=tol, v0=[wm["v_max"] if o else None for wm, o in zip(warm, ok)],
                                           rows=rows)
    imax, vmin, r2, c2 = extreme_eig_batch(Kinv, N, tol=tol, v0=[wm["v_min"] if o else None for wm, o in zip(warm, ok)],
                                           rows=rows)
    return [None if lmax[c] is None else
            dict(cond=lmax[c] * imax[c], lam_max=lmax[c], lam_min=1.0 / imax[c], v_max=vmax[c], v_min=vmin[c],
                 resid_max=r1[c], resid_min=r2[c], cycles=(c1[c], c2[c])) for c in range(B)]


def quad_grad(X, theta, v, *, n_g=None, slot=None, eta=0.0, noisy=False, varK=1.0, kernel=None):
    """gegp_quad_grad: v^T (dKcov/dhp) v for every hyper-parameter (base mode) -> device row laid out as GEGP_OUT_*."""
    lib = L.load()
    X, theta, v = to_dev(X), to_dev(theta), to_dev(v)
    n, d = X.shape
    n_g = n if n_g is None else n_g
    out = torch.zeros(L.out_len(d), dtype=F64, device=device())
    vk = to_dev(np.array([float(varK)]))
    nbytes = int(lib.gegp_quad_grad_work_bytes(n, n_g, d))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device())
    kid, khp = _kern(kernel)
    rc = lib.gegp_quad_grad(n, n_g, d, _p(X), _p(slot), _p(theta), kid, khp, _p(v), L.MODE_BASE, float(eta), int(bool(noisy)),
                            _p(vk), _p(out), _p(ws), nbytes, _stream())
    _check(rc, "gegp_quad_grad")
    return out


def lml_direct_terms(X, theta, *, n_g=None, slot=None, mode=L.MODE_PRECON, eta=0.0, noisy=False, varK=1.0, kernel=None):
    """gegp_lml_direct_terms right after a B = 1 lml_eval(want_grad=True) on this device -> dict of per-hyper-parameter
    rows (GEGP_OUT_* layout, NumPy): aDa = a^T D a, hDa = h^T D a, trKinvD = tr(K^-1 D), and the scalars HKH, Ha."""
    lib = L.load()
    X, theta = to_dev(X), to_dev(theta)
    n, d = X.shape
    n_g = n if n_g is None else n_g
    N = n + n_g * d
    ws = _ws_cache.get(torch.cuda.current_device())
    assert ws is not None, "no likelihood evaluation has run on this device yet"
    ol = L.out_len(d)
    out = torch.zeros(4 * ol + 2, dtype=F64, device=device())
    scratch = torch.empty(4 * ld_of(N), dtype=F64, device=device())
    vk = to_dev(np.array([float(varK)]))
    kid, khp = _kern(kernel)
    rc = lib.gegp_lml_direct_terms(n, n_g, d, _p(X), _p(slot), _p(theta), kid, khp, int(mode), float(eta), int(bool(noisy)),
                                   _p(vk), _p(ws), ws.numel(), _p(scratch), _p(out), _stream())
    _check(rc, "gegp_lml_direct_terms")
    o = out.cpu().numpy()
    rows = o[:4 * ol].reshape(4, ol)
    return dict(aDa=rows[0], hDa=0.25 * (rows[1] - rows[2]), trKinvD=rows[3], HKH=float(o[4 * ol]), Ha=float(o[4 * ol + 1]))


def lml_views(n: int, n_g: int, d: int):
    """Views of candidate 0's arrays inside the shared workspace, valid right after a B = 1 lml_eval(want_grad=True)
    (eager or graph replay) on this device: dict(A [N+2, ld] factor, U [N, ld], Kinv [N, ld], ld)."""
    v = lml_views_batch(n, n_g, d, 1)
    return dict(A=v["A"][0], U=v["U"][0], Kinv=v["Kinv"][0], p=v["p"][0], pinv=v["pinv"][0], ld=v["ld"])


def lml_views_batch(n: int, n_g: int, d: int, B: int):
    """Strided views of the arrays of candidates 0 .. B-1 inside the shared workspace, valid right after an
    lml_eval(want_grad=True) of B rows that fitted the workspace in one chunk (lml_chunk_rows): dict(A [B, N+2, ld],
    U [B, N, ld], Kinv [B, N, ld], p [B, N], pinv [B, N], ld, stride = doubles between candidates)."""
    lib = L.load()
    o = (C.c_int64 * 8)()
    rc = lib.gegp_lml_layout(n, n_g, d, 1, B, o)
    _check(rc, "gegp_lml_layout")
    header, ld, per, offA, offP, _offD, offU, offK = (int(x) for x in o)
    ws = _ws_cache.get(torch.cuda.current_device())
    assert ws is not None and ws.numel() >= header + 8 * per * B, "no likelihood evaluation of this size has run on this device"
    dbl = ws[header:header + 8 * per * B].view(F64)
    N = n + n_g * d

    def view(off, rows, cols=None):   # as_strided takes the offset from the start of the storage, not of `dbl`
        if cols is None:
            return dbl.as_strided((B, rows), (per, 1), dbl.storage_offset() + off)
        return dbl.as_strided((B, rows, cols), (per, ld, 1), dbl.storage_offset() + off)
    return dict(A=view(offA, N + 2, ld), U=view(offU, N, ld), Kinv=view(offK, N, ld), p=view(offP, N),
                pinv=view(offP + ld, N), ld=ld, stride=per)


def lml_chunk_rows(n: int, n_g: int, d: int, B: int, *, want_grad=True, max_ws_bytes=None) -> int:
    """How many of B candidate rows to hand to one lml_eval call whose workspace arrays are read afterwards (gegp_lml_eval
    chunks the rows itself and overwrites earlier chunks' arrays with later ones).  At most max_ws_bytes of workspace
    (default: what lml_eval would use); the workspace is grown so that an lml_eval of that many rows runs in one chunk."""
    lib = L.load()
    op = L.OP_LML_GRAD if want_grad else L.OP_LML
    ws = _lml_workspace(lib, op, n, n_g, d, B, max_ws_bytes)
    o = (C.c_int64 * 8)()
    _check(lib.gegp_lml_layout(n, n_g, d, int(bool(want_grad)), B, o), "gegp_lml_layout")
    header, per = int(o[0]), 8 * int(o[2])
    avail = ws.numel() if max_ws_bytes is None else min(ws.numel(), int(max_ws_bytes))
    c = int(max(1, min(B, (avail - header - 4 * B - 256) // per)))
    workspace(int(lib.gegp_workspace_bytes(op, n, n_g, d, c)) + 4 * c + 256)   # lml_eval of c rows: one chunk
    return c


def build_cov_batch(X, theta_rows, *, n_g=None, slot=None, noise=None, varK_rows=None, mode=L.MODE_BASE, eta=0.0,
                    out=None, kernel=None, kernel_hp_rows=None):
    """gegp_build_cov_batch: one covariance matrix per theta row into out [B, >= N, ld] (strided device view, e.g. the
    U buffers of lml_views_batch).  noise: one device vector for every row, divided by varK_rows[z] on the device."""
    lib = L.load()
    X, th = to_dev(X), to_dev(theta_rows)
    n, d = X.shape
    th = th.reshape(-1, d).contiguous()
    B = th.shape[0]
    n_g = n if n_g is None else n_g
    N = n + n_g * d
    vk = to_dev(varK_rows).reshape(-1).contiguous() if varK_rows is not None else None
    kid, khp = _kern(kernel)
    khp_dev = None
    if kid == L.KERNEL_RATQUAD:
        khp_dev = to_dev(kernel_hp_rows).reshape(-1) if kernel_hp_rows is not None else torch.full((B,), khp, dtype=F64,
                                                                                                   device=device())
    ld = ld_of(N)
    p = torch.empty((B, 2 * ld), dtype=F64, device=device()) if mode == L.MODE_PRECON else None
    rc = lib.gegp_build_cov_batch(B, _p(th), _p(vk), kid, _p(khp_dev), n, n_g, d, _p(X), _p(slot), _p(noise), int(mode),
                                  float(eta), _p(out), out.stride(1), out.stride(0) if B > 1 else 0, _p(p), 2 * ld, 0,
                                  _stream())
    _check(rc, "gegp_build_cov_batch")
    return out


def quad_grad_batch(X, theta_rows, V: torch.Tensor, *, n_g=None, slot=None, eta=0.0, noisy=False, varK_rows=None,
                    kernel=None, kernel_hp_rows=None):
    """gegp_quad_grad_batch: v_z^T (dKcov/dhp) v_z for the rows of V [B, >= N] (unit column stride), each with its own
    theta row (base mode) -> device table [B, 9+d] laid out as GEGP_OUT_*; row z is bit-identical to quad_grad."""
    lib = L.load()
    X, th = to_dev(X), to_dev(theta_rows)
    n, d = X.shape
    th = th.reshape(-1, d).contiguous()
    B = th.shape[0]
    n_g = n if n_g is None else n_g
    assert V.shape[0] == B and V.stride(-1) == 1
    out = torch.zeros((B, L.out_len(d)), dtype=F64, device=device())
    vk = to_dev(varK_rows).reshape(-1).contiguous() if noisy else None
    kid, khp = _kern(kernel)
    khp_dev = None
    if kid == L.KERNEL_RATQUAD:
        khp_dev = to_dev(kernel_hp_rows).reshape(-1) if kernel_hp_rows is not None else torch.full((B,), khp, dtype=F64,
                                                                                                   device=device())
    nbytes = int(lib.gegp_quad_grad_batch_work_bytes(B, n, n_g, d))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device())
    rc = lib.gegp_quad_grad_batch(B, _p(th), _p(vk), kid, _p(khp_dev), n, n_g, d, _p(X), _p(slot), _p(V), V.stride(0),
                                  L.MODE_BASE, float(eta), int(bool(noisy)), _p(out), _p(ws), nbytes, _stream())
    _check(rc, "gegp_quad_grad_batch")
    return out


def cond_fro_of_matrix(K: torch.Tensor, N: int) -> float:
    """Frobenius condition number of an explicit SPD device matrix (factor a copy, explicit inverse, two norms)."""
    ld = ld_of(N)
    A = torch.empty((N, ld), dtype=F64, device=K.device)
    A[:, :N] = K[:, :N]
    info, dinv = potrf(A, N, 0)
    if int(info.item()) != 0:
        return 1e18
    _, Kinv = potri(A, dinv, N)
    return cond_fro(K, Kinv, N, False)[0]


def cond2_of_matrix(K: torch.Tensor, N: int, *, tol: float = 1e-12):
    """Condition number of an explicit symmetric positive-definite device matrix K[:N, :N] ([N, ld] buffer):
    factor a copy, explicit inverse, then cond2().  A failed factorisation is retried once on K + delta I and the
    shift is taken out of lambda_min again (K is then numerically singular: kappa ~ 1 / eps)."""
    ld = ld_of(N)
    shift = 0.0
    for attempt in range(2):
        A = torch.empty((N, ld), dtype=F64, device=K.device)
        A[:, :N] = K[:, :N]
        if shift:
            A[:, :N].diagonal().add_(shift)
        info, dinv = potrf(A, N, 0)
        if int(info.item()) == 0:
            break
        if attempt == 1:   # still not positive definite: report "numerically singular"
            return dict(cond=1e18, lam_max=float("nan"), lam_min=0.0, v_max=None, v_min=None, shift=shift)
        shift = 1e-13 * float(torch.sum(torch.abs(K[:, :N]), dim=1).max().item())
    U, Kinv = potri(A, dinv, N)
    res = cond2(K if K.stride(0) % 2 == 0 and K.data_ptr() % 16 == 0 else K.contiguous(), Kinv, N, tol=tol)
    if shift:
        lmin = max(res["lam_min"] - shift, 2.3e-16 * res["lam_max"])
        res["lam_min"], res["cond"] = lmin, res["lam_max"] / lmin
    res["shift"] = shift
    return res
