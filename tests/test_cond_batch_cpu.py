"""CPU: argument codes of the batched condition-number entry points, and the condition-number-constrained lock-step
multi-start fit (base mode) over a gloo world of 2, with the device evaluator and the condition number replaced by the
CPU oracle: the sharded result equals the one-rank lock step and the reference's sequential loop."""
import os

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy.optimize import Bounds

from test_multistart import _free_port


def test_batched_argument_codes_without_touching_the_gpu():
    from gpgradpy_b200 import _lib
    lib = _lib.load()
    # gegp_symv_batch: B, N, M (16-byte aligned), ld (>= N, even), strideM (even), x, strideX, y, strideY
    assert lib.gegp_symv_batch(0, 8, 16, 8, 0, 16, 0, 16, 0, 0, 0) == -1
    assert lib.gegp_symv_batch(70000, 8, 16, 8, 0, 16, 0, 16, 0, 0, 0) == -1
    assert lib.gegp_symv_batch(2, 0, 16, 8, 0, 16, 0, 16, 0, 0, 0) == -2
    assert lib.gegp_symv_batch(2, 8, 8, 8, 0, 16, 0, 16, 0, 0, 0) == -3
    assert lib.gegp_symv_batch(2, 8, 16, 7, 0, 16, 0, 16, 0, 0, 0) == -4
    assert lib.gegp_symv_batch(2, 8, 16, 8, 3, 16, 0, 16, 0, 0, 0) == -5
    assert lib.gegp_symv_batch(2, 8, 16, 8, 0, 8, 0, 16, 0, 0, 0) == -6
    assert lib.gegp_symv_batch(2, 8, 16, 8, 0, 16, 1, 16, 0, 0, 0) == -7
    assert lib.gegp_symv_batch(2, 8, 16, 8, 0, 16, 0, 0, 0, 0, 0) == -8
    # gegp_lanczos_step_batch: B, N, j < 255, V, ldv, strideV, w, strideW, alpha, beta, strideAB
    assert lib.gegp_lanczos_step_batch(0, 8, 0, 16, 8, 0, 16, 0, 16, 16, 0, 0, 0) == -1
    assert lib.gegp_lanczos_step_batch(2, 8, 255, 16, 8, 0, 16, 0, 16, 16, 0, 0, 0) == -3
    assert lib.gegp_lanczos_step_batch(2, 8, 0, 0, 8, 0, 16, 0, 16, 16, 0, 0, 0) == -4
    assert lib.gegp_lanczos_step_batch(2, 8, 0, 16, 8, 0, 16, 0, 16, 0, 0, 0, 0) == -10
    assert lib.gegp_lanczos_step_batch(2, 8, 0, 16, 8, 0, 16, 0, 16, 16, -1, 0, 0) == -11
    # gegp_lincomb_batch: B, N, k in 1..256, ks, V, ldv, strideV, coef, strideCoef, out, strideOut
    assert lib.gegp_lincomb_batch(2, 8, 0, 0, 16, 8, 0, 16, 0, 16, 0, 0, 0) == -3
    assert lib.gegp_lincomb_batch(2, 8, 257, 0, 16, 8, 0, 16, 0, 16, 0, 0, 0) == -3
    assert lib.gegp_lincomb_batch(2, 8, 4, 0, 16, 8, 0, 0, 0, 16, 0, 0, 0) == -8
    assert lib.gegp_lincomb_batch(2, 8, 4, 0, 16, 8, 0, 16, 0, 0, 0, 0, 0) == -10
    # gegp_quad_grad_batch: base mode only, RatQu needs per-row alphas, work size
    n, d = 4, 3
    wb = lib.gegp_quad_grad_batch_work_bytes(5, n, n, d)
    assert wb > lib.gegp_quad_grad_work_bytes(n, n, d) and lib.gegp_quad_grad_batch_work_bytes(0, n, n, d) == 0
    assert 4 * wb < 5 * 5 * lib.gegp_quad_grad_work_bytes(n, n, d)     # one shared p^-1 vector, one partial table each
    args = [5, 16, 0, 0, 0, n, n, d, 16, 0, 16, 16, _lib.MODE_BASE, 0.0, 0, 16, 16, wb, 0]
    bad = lambda i, v: lib.gegp_quad_grad_batch(*(args[:i] + [v] + args[i + 1:]))
    assert bad(0, 0) == -1 and bad(1, 0) == -2 and bad(14, 1) == -3 and bad(3, _lib.KERNEL_RATQUAD) == -50
    assert bad(12, _lib.MODE_PRECON) == -13 and bad(11, 8) == -12 and bad(17, wb - 8) == -18 and bad(16, 8) == -17
    # gegp_build_cov_batch: mode range, p_out for precon, its stride
    bargs = [3, 16, 0, 0, 0, n, n, d, 16, 0, 0, _lib.MODE_BASE, 0.0, 16, 16, 16 * 16, 0, 0, 0, 0]
    bbad = lambda i, v: lib.gegp_build_cov_batch(*(bargs[:i] + [v] + bargs[i + 1:]))
    assert bbad(0, 0) == -1 and bbad(11, 7) == -12 and bbad(11, _lib.MODE_PRECON) == -17 and bbad(14, 15) == -15
    assert bbad(16, 16) == -18 and bbad(13, 0) == -14 and bbad(3, _lib.KERNEL_RATQUAD) == -50


def _make_gp(cond_max=1e10):
    """Base-mode GaussianProcess whose likelihood and condition number come from the CPU oracle."""
    from gpgradpy_b200.gp import GaussianProcess
    from gpgradpy_b200 import _lib as L
    from oracle import gegp_oracle as O
    x, f, g = O.synthetic_problem(10, 2, 0)
    GP = GaussianProcess(2, True, "SqExp", "base")
    GP.cond_max = cond_max
    GP.set_wellcond_mtd("base")          # the SLSQP constraint takes cond_max from here
    GP.set_data(x, f, np.zeros(10), g, np.zeros((10, 2)))
    GP.cond_warm_start = False
    eta = GP._etaK

    def fake_eval_rows(theta_rows, *, want_grad, **kw):
        import torch
        th = np.atleast_2d(np.asarray(theta_rows, dtype=float))
        out = np.zeros((th.shape[0], L.out_len(2)))
        for r in range(th.shape[0]):
            o = O.lkd_wo_noise(x, f, g, th[r], "base", eta, calc_grad=want_grad)
            if not o.chofac_good:
                out[r, L.OUT_INFO] = 1
                continue
            out[r, L.OUT_LML], out[r, L.OUT_SIGMA2], out[r, L.OUT_BETA] = o.ln_lkd, o.hp_varK, o.hp_beta[0]
            if want_grad:
                out[r, L.OUT_GRAD:] = o.ln_lkd_grad
        return torch.as_tensor(out)

    def fake_cond2(hp_list, calc_grad, warm, rows=None):
        rows = range(len(hp_list)) if rows is None else rows
        conds, grads, res = [None] * len(hp_list), [None] * len(hp_list), [None] * len(hp_list)
        for i in rows:
            c, cg = O.cond_wo_noise(x, np.asarray(hp_list[i].theta), "base", eta, calc_grad=calc_grad)
            conds[i], grads[i], res[i] = float(c), cg, dict(cond=float(c))
        return conds, grads, res

    GP._eval_rows = fake_eval_rows
    GP._cond2_from_workspace = fake_cond2
    GP._cond_chunk_rows = lambda B: B
    GP._final_cond = lambda best: np.nan     # the closing condition number is a device computation (GPU tests cover it)
    return GP


X0 = np.log10(10.0 ** np.random.default_rng(3).uniform(-1.5, 0.5, (5, 2)))
BOUND = Bounds(-5 * np.ones(2), 1 * np.ones(2), keep_feasible=True)
COND_MAX = 1e6     # active for part of the starts


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    GP = _make_gp(COND_MAX)
    best, cond, info = GP.optz_hp_max_lkd(X0, BOUND)
    q.put((rank, best, info, GP._lockstep_stats, GP._multistart_table))
    dist.barrier()
    dist.destroy_process_group()


def test_constrained_lockstep_sharded_world2():
    """5 start rows over 2 ranks (3 + 2) with the kappa <= cond_max constraint: both ranks select the same point and
    report the same info and per-start table as the one-rank lock step, which equals the sequential loop bit for bit."""
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=240) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    GP = _make_gp(COND_MAX)
    assert GP._can_batch_fit()
    best1, _, info1 = GP.optz_hp_max_lkd(X0, BOUND)                # one rank, lock step
    table1 = GP._multistart_table
    assert GP._lockstep_stats["batch_sizes"][0] == 5 and table1.shape == (5, 2 + 6)
    assert np.any(table1[:, 2 + 5] > COND_MAX)                     # some starts begin infeasible
    GP.lockstep_multistart = False
    best_seq, _, info_seq = GP.optz_hp_max_lkd(X0, BOUND)          # the reference's sequential loop
    assert np.array_equal(best1, best_seq) and info1 == info_seq
    for rank, best, info, stats, table in res:
        assert np.array_equal(best, best1) and info == info1
        assert np.array_equal(table, table1, equal_nan=True)
        assert stats["batch_sizes"][0] == (3 if rank == 0 else 2)
