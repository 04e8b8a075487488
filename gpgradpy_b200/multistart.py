"""Lock-step multi-start optimisation: batch point B of the reference (optz/OptzLkd.py:249-270).

The reference runs one SciPy SLSQP per start row, one after the other; every iteration of every start needs one
LML + gradient evaluation.  The starts are independent, so here each SLSQP instance runs in its own host thread and
the threads meet at a barrier whenever they need the objective: the requests of all live starts are evaluated as ONE
batched device call (`gegp_lml_eval` with B = number of live starts), which fills the GPU where a single N ~ 5000
evaluation is bound by the latency of its leaf chain.  A batched candidate is evaluated bit-identically to a lone
one (tested), so every start follows exactly the trajectory it would follow in the sequential loop and the selected
optimum is the same.  Start rows can additionally be sharded over the ranks of a process group; the per-start
results are exchanged with one all_gather (parallel.gather_rows).
"""
from __future__ import annotations

import threading

import numpy as np
from scipy.optimize import NonlinearConstraint, minimize


class LockstepEvaluator:
    """Barrier-style batcher: `evaluate(i, x)` blocks until every live worker has asked, then one of them runs
    `batch_fn(list of (i, x))` -> dict i -> result for all requests at once."""

    def __init__(self, batch_fn, n_workers: int):
        self._fn = batch_fn
        self._cv = threading.Condition()
        self._active = n_workers
        self._pending: dict = {}
        self._results: dict = {}
        self._error = None
        self.n_batches = 0
        self.n_evals = 0
        self.batch_sizes: list = []

    def _flush_locked(self):
        req = sorted(self._pending.items())
        self._pending = {}
        try:
            out = self._fn(req)
        except BaseException as exc:   # noqa: BLE001 -- hand the failure to every waiting worker
            self._error = exc
            out = {i: None for i, _ in req}
        self.n_batches += 1
        self.n_evals += len(req)
        self.batch_sizes.append(len(req))
        self._results.update(out)
        self._cv.notify_all()

    def evaluate(self, idx: int, x):
        with self._cv:
            self._pending[idx] = np.array(x, dtype=float, copy=True)
            if len(self._pending) >= self._active:
                self._flush_locked()
            while idx not in self._results:
                self._cv.wait()
            res = self._results.pop(idx)
            if self._error is not None:
                raise RuntimeError("batched evaluation failed") from self._error
            return res

    def retire(self, idx: int):
        """Worker `idx` is done: the barrier no longer waits for it."""
        with self._cv:
            self._active -= 1
            if self._pending and len(self._pending) >= self._active:
                self._flush_locked()


def minimize_lockstep(batch_val_and_grad, x0_rows, bounds, options, constraints=(), thread_init=None, *,
                      with_ids=False, cond_ub=None):
    """SLSQP from every row of x0_rows, objective/gradient requests batched across the rows.

    batch_val_and_grad(X [b, n_hp]) -> (vals [b], grads [b, n_hp]) of the function to MINIMISE; with_ids: it is called
    as batch_val_and_grad(X, ids) with the start row of every request (for per-start state such as warm starts).
    thread_init: called first in every worker thread (the CUDA device is per-thread state: a worker that ends up
    running the batched device call must select the caller's device).
    cond_ub: the condition-number-constrained fit of optz/OptzLkd.py:225-270.  batch_val_and_grad then also returns
    (conds [b], cond_grads [b, n_hp]); every start gets the SLSQP constraint cond <= cond_ub, whose callbacks read the
    start's cache that the same request filled.  As in the sequential loop, every start is evaluated once at its x0
    before its SLSQP runs (with a cleared cache afterwards) and once more at its solution; those two results per start
    are kept in ev.at_x0 and ev.at_solution as (val, grad, cond, cond_grad).
    Returns (list of scipy OptimizeResult in row order, LockstepEvaluator with its statistics)."""
    x0_rows = np.atleast_2d(np.asarray(x0_rows, dtype=float))
    n = x0_rows.shape[0]

    def batch_fn(req):
        X = np.vstack([x for _, x in req])
        outs = batch_val_and_grad(X, [i for i, _ in req]) if with_ids else batch_val_and_grad(X)
        return {i: tuple(float(o[k]) if np.ndim(o[k]) == 0 else np.array(o[k], dtype=float) for o in outs)
                for k, (i, _) in enumerate(req)}

    ev = LockstepEvaluator(batch_fn, n)
    ev.at_x0, ev.at_solution = [None] * n, [None] * n
    results = [None] * n
    errors = [None] * n

    def worker(i):
        last = {"x": None, "r": None}

        def get(x):
            if last["x"] is None or not np.array_equal(x, last["x"]):
                r = ev.evaluate(i, x)
                last.update(x=np.array(x, copy=True), r=r)
            return last["r"]

        try:
            if thread_init is not None:
                thread_init()
            cons = constraints
            if cond_ub is not None:
                ev.at_x0[i] = get(x0_rows[i])
                last["x"] = None
                cons = NonlinearConstraint(lambda x: get(x)[2], -np.inf, cond_ub, jac=lambda x: get(x)[3])
            results[i] = minimize(lambda x: get(x)[0], x0_rows[i], method="SLSQP", jac=lambda x: get(x)[1],
                                  bounds=bounds, constraints=cons, options=options)
            if cond_ub is not None:
                ev.at_solution[i] = get(results[i].x)
        except BaseException as exc:   # noqa: BLE001
            errors[i] = exc
        finally:
            ev.retire(i)

    threads = [threading.Thread(target=worker, args=(i,), daemon=True) for i in range(n)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in errors:
        if e is not None:
            raise e
    return results, ev
