"""Batched surrogate Hessians against the one-point loop, on the device.

For configurations 2 (n = 500, d = 10, N = 5500) and 3 (n = 1000, d = 20, N = 21000) and nx in {1, 16, 256, 1024} test
points: Hessians per second of GaussianProcess.eval_model_hess_batch (one chunked pass) and of a loop of one-point
eval_model(x[i:i+1], calc_grad=True, calc_hess=True) calls over the same points, both timed on the host around work that
ends in a device synchronise (the results come back to the host), after a warm-up of the same shapes; the forward solve's
rate, (d + 1) N^2 nx flops over the CUDA-event time of gegp_trsm_rows on the (d + 1) nx rows the batched call solves (and
on the d + 1 rows of one point); and the largest difference between the two paths, relative to each output's largest
entry.  Prints the card's name and power limit first.  Usage: python tools/hess_batch_probe.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return torch.cuda.get_device_name(0), q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def solve_rate(bk, st, rows, reps):
    """(d + 1) N^2 nx flops / event time of the forward solve of `rows` rows against the GP's factor."""
    N = st.N
    B = torch.randn((rows, bk.ld_of(N)), dtype=torch.float64, device="cuda")
    bk.trsm_rows(st.A, st.dinv, N, B)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        bk.trsm_rows(st.A, st.dinv, N, B)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return ms, rows * float(N) ** 2 / (ms * 1e-3) / 1e12


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--nx", default="1,16,256,1024")
    ap.add_argument("--configs", default="c2,c3")
    args = ap.parse_args()
    from gpgradpy_b200 import backend as bk
    from gpgradpy_b200.gp import GaussianProcess
    from oracle import gegp_oracle as O
    name, plim = card()
    print(f"card: {name}  power.limit: {plim}", flush=True)
    sizes = {"c2": (500, 10), "c3": (1000, 20)}
    rows = []
    for cfg in args.configs.split(","):
        n, d = sizes[cfg]
        x, f, g = O.synthetic_problem(n, d, 0)
        GP = GaussianProcess(d, True, "SqExp", "precon")
        GP.set_data(x, f, np.zeros(n), g, np.zeros((n, d)))
        GP.set_hpara("set", 1, GP.make_hp_class(theta=O.bench_theta(d), varK=1.7, beta=np.array([float(np.mean(f))])))
        st = GP._pred
        one_ms, one_tf = solve_rate(bk, st, d + 1, 20)
        for nx in (int(v) for v in args.nx.split(",")):
            xs = np.random.default_rng(nx).uniform(-1.5, 1.5, (nx, d))
            reps_b = max(1, min(20, 2048 // nx))
            t_b, got = timed(lambda: GP.eval_model_hess_batch(xs), reps_b)
            # warm-up of the one-point shapes, then the full loop once
            for i in range(min(nx, 4)):
                GP.eval_model(xs[i:i + 1], calc_grad=True, calc_hess=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            loop = [GP.eval_model(xs[i:i + 1], calc_grad=True, calc_hess=True) for i in range(nx)]
            torch.cuda.synchronize()
            t_l = time.perf_counter() - t0
            diff = 0.0
            far = got[1] > 0.1 * np.max(got[1])
            for k in range(6):
                ref = np.stack([np.asarray(o[k])[0] for o in loop])
                a, b = (got[k][far], ref[far]) if k in (3, 5) else (got[k], ref)
                if a.size:
                    diff = max(diff, float(np.max(np.abs(a - b)) / np.max(np.abs(b))))
            s_ms, s_tf = solve_rate(bk, st, (d + 1) * nx, max(1, min(10, 1024 // nx)))
            r = dict(config=cfg, n=n, d=d, N=st.N, nx=nx, batched_s=t_b, looped_s=t_l, batched_hess_per_s=nx / t_b,
                     looped_hess_per_s=nx / t_l, solve_ms=s_ms, solve_tflops=s_tf, one_point_solve_ms=one_ms,
                     one_point_solve_tflops=one_tf, max_rel_diff=diff)
            rows.append(r)
            print(f"{cfg} N={st.N} nx={nx:5d}: batched {nx / t_b:10.1f} Hess/s ({t_b * 1e3:9.2f} ms)  looped "
                  f"{nx / t_l:8.1f} Hess/s ({t_l * 1e3:9.2f} ms)  forward solve {(d + 1) * nx} rows {s_ms:8.2f} ms "
                  f"{s_tf:6.2f} TFLOP/s (one point: {one_ms:.2f} ms, {one_tf:.3f} TFLOP/s)  max rel diff {diff:.1e}",
                  flush=True)
        del GP, st
        bk.free_workspace()
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(dict(card=name, power_limit=plim, rows=rows), fh, indent=1)


if __name__ == "__main__":
    main()
