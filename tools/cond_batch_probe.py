"""Batched condition numbers against the one-candidate paths, old build against new build, in one run.

Times, on the host around work that ends in a device synchronise (the results come back to the host), after a warm-up
of the same shapes:
  * grid:   BASELINE config 1 (12 x 12 length-scale grid, n = 20, d = 2) in the base, rescale_origin and precon modes, as
            the loop of calc_lkd_all(calc_cond=True) calls of examples/config1_cond_lkd_grid.py and as ONE
            calc_lkd_batch(calc_cond=True) call per mode;
  * fit:    a 5-start lhs base-mode fit with the kappa <= cond_max constraint (optz_hp_max_lkd) at n = 200, d = 5 and at
            config 2 (n = 500, d = 10; --c2-maxiter SLSQP iterations), the sequential loop against the lock step;
  * single: one calc_lkd_all(calc_cond=True, calc_grad=True) at config 2 (N = 5500), the one-candidate path.
Each case runs in a fresh process per build; the builds alternate (--reps rounds of old, new).  The old build (a tree
with the parent's package and its libgegp.so, --old ROOT) has no batched kappa: there only the loops run.  Prints the
card's name and power limit first, then one JSON line per (round, build, case).
Usage: python tools/cond_batch_probe.py --old ROOT [--reps 2] [--cases grid,fit,single] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


# ------------------------------------------------------------------------------------------------------------ worker
def _sync_time(fn, reps=1):
    import torch
    fn()                                   # warm-up: the same shapes
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps, out


def case_grid(batched):
    import numpy as np
    from gpgradpy_b200.gp import GaussianProcess
    n_eval, dim, n_gamma = 20, 2, 12
    x = np.random.default_rng(2).uniform(0.9, 1.1, (n_eval, dim))
    f = np.sum(10 * (x[:, 1:] - x[:, :-1] ** 2) ** 2 + (1 - x[:, :-1]) ** 2, axis=1)
    g = np.zeros_like(x)
    g[:, :-1] += -2 * (1 - x[:, :-1]) - 40 * x[:, :-1] * (x[:, 1:] - x[:, :-1] ** 2)
    g[:, 1:] += 20 * (x[:, 1:] - x[:, :-1] ** 2)
    nugget = GaussianProcess(dim, True, "SqExp", "precon").calc_nugget(n_eval)[1]
    tv = np.logspace(*np.log10(GaussianProcess.gamma2theta(np.array([1e-4, 1e8]))), n_gamma)
    out = {}
    for mode in ("base", "rescale_origin", "precon"):
        GP = GaussianProcess(dim, True, "SqExp", mode)
        GP.cond_eta_is_const = True
        GP.cond_warm_start = False
        GP.set_data(x, f, np.zeros(n_eval), g, np.zeros(g.shape))
        GP._etaK = GP._eta_Kgrad = nugget
        GP.cond_max = 1e10

        def loop():
            c = np.zeros((n_gamma, n_gamma))
            for i in range(n_gamma):
                for j in range(n_gamma):
                    hp = GP.make_hp_class(theta=np.array([tv[i], tv[j]]))
                    c[i, j] = GP.calc_lkd_all(hp, calc_lkd=True, calc_cond=True, calc_grad=False)[0].cond
            return c

        rows = np.log10(np.array([[tv[i], tv[j]] for i in range(n_gamma) for j in range(n_gamma)]))
        t_loop, c_loop = _sync_time(loop)
        out[mode] = {"loop_s": t_loop}
        if batched:
            from gpgradpy_b200 import _lib as L
            t_b, tab = _sync_time(lambda: GP.calc_lkd_batch(rows, calc_cond=True))
            c_b = tab[:, L.out_len(dim)].reshape(n_gamma, n_gamma)
            ok = np.isfinite(c_loop) & (c_loop < 1e12)
            out[mode].update(batch_s=t_b, max_rel_diff_cond_lt_1e12=float(np.max(np.abs(c_b[ok] / c_loop[ok] - 1))))
    return out


def _fit_gp(n, d, maxiter):
    import numpy as np
    from gpgradpy_b200.gp import GaussianProcess
    from oracle import gegp_oracle as O
    x, f, g = O.synthetic_problem(n, d, 0)
    GP = GaussianProcess(d, True, "SqExp", "base")
    GP.optz_iter_max = maxiter
    GP.init_optz_surr(3)
    GP.set_data(x[:1], f[:1], np.zeros(1), g[:1], np.zeros((1, d)))
    GP.set_hpara("optz", 0)
    GP.set_data(x, f, np.zeros(n), g, np.zeros((n, d)))
    hp_x0, bounds = GP.get_hp_x0_lhs_median(1, GP.hp_info_optz_lkd, 5)
    return GP, hp_x0, bounds


def case_fit(batched, c2_maxiter):
    import numpy as np
    import torch
    out = {}
    for name, n, d, maxiter in (("n200_d5", 200, 5, 250), ("c2", 500, 10, c2_maxiter)):
        GP, hp_x0, bounds = _fit_gp(n, d, maxiter)
        GP.cond_warm_start = False
        res = {}
        for lock in ((False, True) if batched else (False,)):
            GP.lockstep_multistart = lock
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            best, cond, info = GP.optz_hp_max_lkd(hp_x0, bounds)
            torch.cuda.synchronize()
            res["lockstep" if lock else "sequential"] = dict(s=time.perf_counter() - t0, best=np.asarray(best).tolist(),
                                                             cond=float(cond), iter_mean=info["hp_optz_iter_mean"],
                                                             con_good=info["hp_optz_con_good"])
        out[name] = res
    return out


def case_single():
    import numpy as np
    from gpgradpy_b200.gp import GaussianProcess
    from oracle import gegp_oracle as O
    n, d = 500, 10
    x, f, g = O.synthetic_problem(n, d, 0)
    GP = GaussianProcess(d, True, "SqExp", "base")
    GP.cond_warm_start = False
    GP.set_data(x, f, np.zeros(n), g, np.zeros((n, d)))
    hp = GP.make_hp_class(theta=O.bench_theta(d) * 4.0)
    t, r = _sync_time(lambda: GP.calc_lkd_all(hp, calc_cond=True, calc_grad=True)[0], reps=10)
    return {"s": t, "cond": float(r.cond), "cond_grad": np.asarray(r.cond_grad).tolist(), "ln_lkd": float(r.ln_lkd)}


def worker(args):
    sys.path.insert(0, args.root)
    sys.path.insert(1, HERE)           # the oracle (checker side) of this tree
    from gpgradpy_b200.gp import GaussianProcess
    batched = "calc_cond" in GaussianProcess.calc_lkd_batch.__code__.co_varnames
    if args.case == "grid":
        res = case_grid(batched)
    elif args.case == "fit":
        res = case_fit(batched, args.c2_maxiter)
    else:
        res = case_single()
    print("RESULT " + json.dumps(res))


# -------------------------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old", help="root of a tree holding the old build's gpgradpy_b200 package (with libgegp.so)")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--cases", default="grid,fit,single")
    ap.add_argument("--c2-maxiter", type=int, default=250)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--root", default=HERE)
    ap.add_argument("--case", default=None)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    print(f"card: {card()}", flush=True)
    builds = ([("old", os.path.abspath(args.old))] if args.old else []) + [("new", HERE)]
    lines = []
    for rep in range(args.reps):
        for case in args.cases.split(","):
            for build, root in builds:
                cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--root", root, "--case", case,
                       "--c2-maxiter", str(args.c2_maxiter)]
                r = subprocess.run(cmd, capture_output=True, text=True, cwd=HERE)
                res = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
                line = dict(round=rep, build=build, case=case,
                            result=json.loads(res[-1][7:]) if res else None,
                            error=None if res else (r.stderr[-2000:] or f"exit {r.returncode}"))
                print(json.dumps(line), flush=True)
                lines.append(line)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(dict(card=card(), lines=lines), fh, indent=1)


if __name__ == "__main__":
    main()
