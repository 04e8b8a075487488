#!/usr/bin/env python
"""bench.py -- LML + hyper-parameter-gradient evaluations per second of the gradient-enhanced GP hot path.

    python bench.py --gpus 1 --steps 20 --warmup 3              # this repo's CUDA path (one JSON line)
    python bench.py --workload c3 ...                           # the north-star size as the headline workload
    python bench.py --impl reference --steps 2 --warmup 1       # the reference on the host cores (same --workload)
    torchrun --nproc-per-node N ... bench.py --gpus N ...       # N ranks (see "multi-GPU" below)
    python bench.py ... --dump-outputs DIR                      # also save what the last timed step computed

A "step" is one evaluation of LML and its full theta-gradient (build -> Cholesky -> solves -> inverse -> gradient
contraction).  Headline workload: BASELINE.json `configs[1]` (c2: d=10, n=500, N=5500, preconditioned) unless
`--workload c3` (configs[2], the north-star size d=20, n=1000, N=21000).  `value` times the device path with inputs
resident in HBM; `e2e` goes through the public GaussianProcess.calc_lkd_all API with host buffers (H2D of X, y, theta and
D2H of the result every step).  The same line carries, measured in the same run on rank 0 at N=1:
  peaks    fp64 DMMA issue peak (gegp_dmma_peak) and cuBLAS DGEMM / cuSOLVER potrf on this GPU -- the denominators;
  phases   Cholesky alone (graph replay, as the product runs it, and eager) beside cuSOLVER potrf, build GB/s, GEMM share;
  c3       the same phases at N=21000 plus e2e, the posterior at 10^4 test points and parity against the CPU port;
  c4_scan  BASELINE configs[3]: 1024 candidate thetas (d=5, n=200) through GaussianProcess.calc_lkd_batch, LML-only
           (what select_hp_optz_x0 runs) and with gradient -- sharded over ALL ranks at every --gpus N (strong scaling);
  c5       BASELINE configs[4]: N=51000 build + Cholesky in the base / rescale_origin / precon modes.
Multi-GPU: the headline stays the c2 evaluation, one independent candidate per rank and step plus one all_gather of the
result rows ("weak"); the sharded candidate scan rides along as `c4_scan` with its own strong-scaling numbers.
--steps sets the number of timed steps, each on its own theta (step_theta); with the same arguments the inputs (seeded
data and thetas) are the same from run to run.  --dump-outputs DIR writes the result rows of the last timed step, as the
caller of gegp_lml_eval receives them ([ranks, 10 + d] float64 in the OUT_* slots of include/gegp.h: LML, sigma^2, beta,
ln det, info, ..., then the theta-gradient), to DIR/lml_eval_out.npy, so that two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "LML+gradient evals/sec (fp64, preconditioned GE-GP)"
UNIT = "evals/s"
WORKLOADS = {"c2": (500, 10), "c3": (1000, 20)}
C4 = dict(n=200, d=5, B=1024)
C5 = dict(n=1000, d=50)
REF_TIME_BUDGET_S = 60.0        # the reference arm stops after this much timed work (one c2 step is ~5-15 s)


def workload_label(wl):
    n, d = WORKLOADS[wl]
    return f"{wl}: d={d}, n={n}, N={n * (d + 1)}, precon, LML+grad"


# ----------------------------------------------------------------------------------------------- synthetic inputs
def rosenbrock(x, a=10.0):
    return np.sum(a * (x[:, 1:] - x[:, :-1] ** 2) ** 2 + (1.0 - x[:, :-1]) ** 2, axis=1)


def rosenbrock_grad(x, a=10.0):
    g = np.zeros_like(x)
    g[:, :-1] += -2.0 * (1.0 - x[:, :-1]) - 4.0 * a * x[:, :-1] * (x[:, 1:] - x[:, :-1] ** 2)
    g[:, 1:] += 2.0 * a * (x[:, 1:] - x[:, :-1] ** 2)
    return g


def make_problem(n, d, seed=0):
    """SURVEY.md 8(d): X ~ U[-2,2]^d (default_rng(seed)), Rosenbrock a=10, theta_i = 0.05 linspace(.5,1.5,d) 10/d."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-2.0, 2.0, (n, d))
    theta = 0.05 * np.linspace(0.5, 1.5, d) * (10.0 / d)
    return x, rosenbrock(x), rosenbrock_grad(x), theta


def step_theta(theta, step, rank):
    """A different candidate every step and rank (no result can be cached)."""
    return theta * (1.0 + 0.003 * step + 0.0007 * rank)


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: each device tensor as out_dir/<name>.npy in float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy().astype(np.float64))


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- reference arm
def _use_all_host_threads():
    """Give the host BLAS every core (returns the thread count actually in effect)."""
    want = os.cpu_count() or 1
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=want)
        got = [p.get("num_threads", 1) for p in threadpoolctl.threadpool_info() if p.get("user_api") == "blas"]
        return int(max(got)) if got else want
    except Exception:
        return int(os.environ.get("OMP_NUM_THREADS", want))


class CpuArm:
    """The reference's own implementation of the path on the host cores.

    kind "reference": the UNMODIFIED reference (marchildon/gpgradpy v1.3.2) imported from baseline/_ref (installed by
    oracle/install_ref.py; needs the `smt` stand-in next to it) -- GaussianProcess.calc_lkd_all(calc_grad=True).
    kind "port": oracle/gegp_oracle.py, the NumPy/SciPy restatement pinned to the reference's outputs, used when the
    reference is not importable and always at c3, where the reference cannot run (its dK/dtheta tensor alone is
    70.6 GB; the lean form contracts it tile by tile)."""

    def __init__(self, workload):
        from oracle import gegp_oracle as O     # the one place bench.py executes oracle/ as the thing measured
        self.O = O
        self.workload = workload
        self.n, self.d = WORKLOADS[workload]
        self.x, self.f, self.g, self.theta = make_problem(self.n, self.d)
        self.eta = O.nugget(self.n, self.d, "precon")[1]
        self.kind, self.GP, self.why_port = "port", None, None
        if workload == "c3":
            self.why_port = "restatement, reference infeasible at N=21000 (its dK/dtheta tensor alone is 70.6 GB)"
        else:
            try:
                ref_dir = os.path.join(ROOT, "baseline", "_ref")
                if not os.path.isdir(os.path.join(ref_dir, "gpgradpy")):
                    raise ImportError("baseline/_ref/gpgradpy is missing (run oracle/install_ref.py in the build container)")
                if ref_dir not in sys.path:
                    sys.path.insert(0, ref_dir)
                from gpgradpy.src.GaussianProcess import GaussianProcess as RefGP   # the reference itself
                self.GP = RefGP(self.d, True, "SqExp", "precon")
                self.GP.set_data(self.x, self.f, np.zeros(self.n), self.g, np.zeros((self.n, self.d)))
                self.kind = "reference"
            except Exception as exc:   # noqa: BLE001 -- report why the port stands in
                self.why_port = f"reference not importable here ({type(exc).__name__}: {exc})"[:300]
        self.cores = _use_all_host_threads()    # torchrun exports OMP_NUM_THREADS=1: undo that for the CPU arm

    def warm(self):
        """Numba JIT (reference) / BLAS thread pools on a tiny problem of the same dimension."""
        n, d = 24, self.d
        xs, fs, gs, ths = make_problem(n, d)
        if self.kind == "reference":
            from gpgradpy.src.GaussianProcess import GaussianProcess as RefGP
            G = RefGP(d, True, "SqExp", "precon")
            G.set_data(xs, fs, np.zeros(n), gs, np.zeros((n, d)))
            G.calc_lkd_all(G.make_hp_class(theta=ths), calc_grad=True)
        else:
            self.O.lkd_wo_noise_lean(xs, fs, gs, ths, "precon", self.O.nugget(n, d, "precon")[1])

    def eval(self, theta):
        """-> (ln_lkd, grad[d], varK, beta)"""
        if self.kind == "reference":
            info, good = self.GP.calc_lkd_all(self.GP.make_hp_class(theta=theta), calc_grad=True)
            assert good
            return float(info.ln_lkd), np.asarray(info.ln_lkd_grad, float), float(info.hp_varK), float(np.ravel(info.hp_beta)[0])
        fn = self.O.lkd_wo_noise_lean if self.workload == "c3" else self.O.lkd_wo_noise
        r = fn(self.x, self.f, self.g, theta, "precon", self.eta, calc_grad=True)
        return float(r.ln_lkd), np.asarray(r.ln_lkd_grad, float), float(r.hp_varK), float(r.hp_beta[0])

    def describe(self, steps):
        if self.kind == "reference":
            what = ("the unmodified reference (gpgradpy 1.3.2 from baseline/_ref, GaussianProcess.calc_lkd_all(calc_grad=True), "
                    "Numba kernels single-threaded as shipped, BLAS on all cores)")
        elif self.workload == "c3":
            what = "oracle/gegp_oracle.lkd_wo_noise_lean (LAPACK dpotrf/dpotri, dK/dtheta tiles on the fly): " + self.why_port
        else:
            what = "oracle/gegp_oracle.lkd_wo_noise (NumPy/SciPy restatement that materialises dK/dtheta and K^-1 like the " \
                   "reference): " + str(self.why_port)
        return f"{steps} full LML+gradient evaluation(s) of the same workload by {what}"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args.workload)
    arm.warm()
    W = max(args.warmup, 3)                  # the CUDA arm's warm-up count: the timed steps use the same thetas
    t0 = time.perf_counter()
    steps = 0
    for s in range(max(1, args.steps)):
        arm.eval(step_theta(arm.theta, W + s, 0))
        steps += 1
        if time.perf_counter() - t0 > REF_TIME_BUDGET_S:
            break
    dt = time.perf_counter() - t0
    val = steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_label(args.workload), "seed": 0},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.describe(steps)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": f"bounded sample: stops after {REF_TIME_BUDGET_S:.0f} s of timed work; thetas are the CUDA arm's timed steps"}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- CUDA arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from gpgradpy_b200 import backend as bk, _lib as L
    from gpgradpy_b200.gp import GaussianProcess
    from gpgradpy_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = L.load()
    n, d = WORKLOADS[args.workload]
    N = n * (d + 1)
    x, f, g, theta = make_problem(n, d)
    GP = GaussianProcess(d, True, "SqExp", "precon")
    GP.set_data(x, f, np.zeros(n), g, np.zeros((n, d)))
    eta = GP._etaK
    y = GP.make_data_vec(f, g)
    X_dev, y_dev = bk.to_dev(x), bk.to_dev(y)
    K, W = args.steps, max(args.warmup, 3)
    thetas = torch.stack([bk.to_dev(step_theta(theta, s, rank)) for s in range(K + W)])

    def device_step(s):
        # the product path of the optimiser's inner loop: one captured CUDA graph per problem, replayed per candidate
        out = bk.lml_eval_graphed(X_dev, y_dev, thetas[s:s + 1], mode=L.MODE_PRECON, eta=eta, want_grad=True)
        if world > 1:
            out = parallel.gather_rows(out, world)   # scalar results of all ranks, one NCCL all_gather
        return out

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for s in range(W):
        device_step(s)
    sync()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    L.profile_begin(False)
    replayed0 = bk.replay_stats["kernel_launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    last = None
    for s in range(W, W + K):
        last = device_step(s)
    e1.record()
    sync()
    launches = L.profile_end()["launches"] + bk.replay_stats["kernel_launches"] - replayed0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    last = last.clone()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lml_eval_out=last)
    info_ok = bool((last[:, L.OUT_INFO] == 0).all().item())
    value = world * K / (ms_total * 1e-3)

    # ---- end to end through the public API with host buffers (pinned H2D of X, y, theta; D2H of the result)
    def api_e2e(gp, th0, n_, d_, steps, warm=2):
        for s in range(warm):
            gp._dev_ready = False
            gp.calc_lkd_all(gp.make_hp_class(theta=step_theta(th0, s, rank)), calc_grad=True)
        sync()
        t0 = time.perf_counter()
        for s in range(W, W + steps):
            gp._dev_ready = False                    # forces the host -> device copy of X and y again
            gp.calc_lkd_all(gp.make_hp_class(theta=step_theta(th0, s, rank)), calc_grad=True)
        sync()
        dt = max_over_ranks(time.perf_counter() - t0)
        return {"value": world * steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(8 * (n_ * d_ + n_ * (d_ + 1) + d_)),
                "d2h_bytes_per_step": int(8 * L.out_len(d_)), "steps": steps,
                "api": "GaussianProcess.calc_lkd_all(hp_vals, calc_grad=True)"}

    e2e = api_e2e(GP, theta, n, d, K)

    # ---- BASELINE configs[3]: the 1024-candidate scan through the public API, sharded over all ranks (strong scaling)
    def c4_scan():
        n4, d4, B4 = C4["n"], C4["d"], C4["B"]
        x4, f4, g4, _ = make_problem(n4, d4)
        G4 = GaussianProcess(d4, True, "SqExp", "precon")
        G4.set_data(x4, f4, np.zeros(n4), g4, np.zeros((n4, d4)))
        rows = np.random.default_rng(0).uniform(-5.0, 1.0, (B4, d4))     # SURVEY 8(d): log10 theta ~ U[-5, 1]^d
        res = {"workload": f"c4: d={d4}, n={n4}, N={n4 * (d4 + 1)}, {B4} candidate thetas, precon", "scaling": "strong",
               "n_gpus": world, "candidates_per_rank": -(-B4 // world),
               "api": "GaussianProcess.calc_lkd_batch(hp_vec_rows, calc_grad) -- host rows in, host table out "
                      "(H2D of the rows, batched gegp_lml_eval on each rank's shard, one all_gather, D2H of the table)"}
        N4 = n4 * (d4 + 1)
        for grad, key in ((False, "lml_only"), (True, "lml_grad")):
            tab = G4.calc_lkd_batch(rows, calc_grad=grad)
            sync()
            reps, best = 3, 1e30
            for _ in range(reps):
                sync()
                t0 = time.perf_counter()
                tab = G4.calc_lkd_batch(rows, calc_grad=grad)
                best = min(best, max_over_ranks(time.perf_counter() - t0))
            flops = B4 * (N4 ** 3 if grad else N4 ** 3 / 3.0)
            ok = tab[:, L.OUT_INFO] == 0
            lml = np.where(ok, tab[:, L.OUT_LML], -np.inf)
            res[key] = {"ms_per_scan": best * 1e3, "candidates_per_s": B4 / best, "tflops": flops / best * 1e-12,
                        "flops_per_candidate": "N^3 (factor + explicit inverse)" if grad else "N^3/3 (factor only)",
                        "chol_ok": int(ok.sum()), "argmax": int(np.argmax(lml)), "lml_max": float(lml.max())}
        return res

    c4 = None
    if not args.no_c4:
        try:
            c4 = c4_scan()
        except Exception as exc:   # noqa: BLE001 -- report, never hide
            c4 = {"error": repr(exc)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------------------------------------------------------------------------------- rank 0 only from here
    def ev_ms(fn, reps=3):
        best = 1e30
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b))
        return best

    def graph_of(fn):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            fn()
        return gr

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback of /opt/skills/guides/B200_PROFILING.md"
    # fp64 denominators measured on THIS GPU in THIS run (MEASURED_PEAKS.json has no fp64 entry)
    dmma_peak = bk.dmma_peak_tflops(3)
    in_run = {"fp64_dmma_issue_peak_tflops": dmma_peak,
              "how": "gegp_dmma_peak: 148 CTAs x 16 warps of independent mma.sync.m8n8k4.f64 chains, best of 3, CUDA events"}
    if not args.no_phases:
        try:
            a_ = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
            b_ = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
            torch.matmul(a_, b_)
            in_run["cublas_dgemm_8192_tflops"] = 2 * 8192.0 ** 3 / ev_ms(lambda: torch.matmul(a_, b_)) * 1e-9
            del a_, b_
        except Exception as exc:   # noqa: BLE001
            in_run["cublas_dgemm_8192_tflops"] = repr(exc)

    def phase_numbers(n_, d_, reps=2):
        N_ = n_ * (d_ + 1)
        x_, f_, g_, th_ = make_problem(n_, d_)
        Xd, yd, thd = bk.to_dev(x_), bk.to_dev(np.hstack((f_, g_.reshape(g_.size, order="F")))), bk.to_dev(th_[None, :])
        eta_ = GaussianProcess(d_, True).calc_nugget(n_)[1]
        run = lambda grad: bk.lml_eval(Xd, yd, thd, mode=L.MODE_PRECON, eta=eta_, want_grad=grad)  # noqa: E731
        run(True)
        ms_grad, ms_val = ev_ms(lambda: run(True), reps), ev_ms(lambda: run(False), reps)
        ms_grad_graph = ev_ms(lambda: bk.lml_eval_graphed(Xd, yd, thd, mode=L.MODE_PRECON, eta=eta_, want_grad=True), reps + 1)
        # per-launch GEMM timing: with the look-ahead on, GEMMs of different streams overlap and their event-bracketed
        # durations would count the same wall time more than once, so this pass runs the single-stream schedule
        old_la = lib.gegp_set_option(L.OPT_LOOKAHEAD, 0)
        try:
            run(True)
            L.profile_begin(True)
            for _ in range(reps):
                run(True)
            pr = L.profile_end()
        finally:
            lib.gegp_set_option(L.OPT_LOOKAHEAD, old_la)
        gemm_ms = pr["gemm_ms"] / reps
        ld = bk.ld_of(N_)
        buf = torch.empty((N_ + 2, ld), dtype=torch.float64, device="cuda")
        dinv_ = bk.dinv_buffer(N_)
        info_ = torch.zeros(1, dtype=torch.int32, device="cuda")
        # the builder runs for tens of microseconds at c2: time a back-to-back burst so that the host-side launch
        # preparation of one call hides behind the previous kernel (every launch rewrites all 8 N^2 bytes; the
        # matrix is larger than L2)
        burst = 20 if N_ < 10000 else 4

        def build(uplo):
            bk.build_cov(Xd, thd[0], mode=L.MODE_PRECON, eta=eta_, out=buf[:N_], uplo=uplo)

        def build_burst(uplo):
            for _ in range(burst):
                build(uplo)
        ms_full = ev_ms(lambda: build_burst(0), reps) / burst
        ms_low = ev_ms(lambda: build_burst(1), reps) / burst

        def potrf_raw():
            rc = lib.gegp_potrf(N_, 0, buf.data_ptr(), buf.stride(0), dinv_.data_ptr(), info_.data_ptr(),
                                torch.cuda.current_stream().cuda_stream)
            assert rc == 0

        def fac():
            build(1)
            potrf_raw()
        # Cholesky alone = (build + factor) - build, both as the product runs them: replayed from a captured graph
        g_fac, g_build = graph_of(fac), graph_of(lambda: build(1))
        ms_chol = ev_ms(g_fac.replay, reps + 2) - ev_ms(g_build.replay, reps + 2)
        ms_chol_eager = ev_ms(fac, reps) - ev_ms(lambda: build(1), reps)
        del g_fac, g_build
        # the vendor library on the same matrix (checker / comparison point only, never on the product path)
        ms_cusolver = None
        try:
            build(0)
            Kf = buf[:N_, :N_].contiguous()
            torch.linalg.cholesky_ex(Kf)
            ms_cusolver = ev_ms(lambda: torch.linalg.cholesky_ex(Kf), reps)
            del Kf
        except Exception:   # noqa: BLE001
            pass
        del buf
        return {"n": n_, "d": d_, "N": N_, "lml_grad_ms": ms_grad, "lml_grad_graph_ms": ms_grad_graph, "lml_only_ms": ms_val,
                "lml_grad_evals_per_s": 1e3 / ms_grad_graph, "overall_tflops_N3": N_ ** 3 / ms_grad_graph * 1e-9,
                "overall_frac_of_dmma_peak": N_ ** 3 / ms_grad_graph * 1e-9 / dmma_peak,
                "cholesky_ms": ms_chol, "cholesky_eager_ms": ms_chol_eager, "cusolver_potrf_ms": ms_cusolver,
                "cholesky_vs_cusolver": (ms_cusolver / ms_chol) if ms_cusolver else None,
                "cholesky_tflops": N_ ** 3 / 3 / ms_chol * 1e-9,
                "cholesky_frac_of_dmma_peak": N_ ** 3 / 3 / ms_chol * 1e-9 / dmma_peak,
                "gemm_ms_per_eval": gemm_ms, "gemm_launches_per_eval": pr["gemm_launches"] // reps,
                "gemm_tflops_executed": pr["gemm_flops"] / reps / gemm_ms * 1e-9,
                "gemm_share_of_step": gemm_ms / ms_grad,
                "build_full_ms": ms_full, "build_full_gbs": 8.0 * N_ * N_ / ms_full * 1e-6,
                "build_full_frac_of_hbm": 8.0 * N_ * N_ / ms_full * 1e-6 / hbm_peak,
                "build_lower_ms": ms_low, "build_lower_gbs": 4.0 * N_ * (N_ + 1) / ms_low * 1e-6,
                "note": "cholesky_ms: gegp_potrf replayed from a captured CUDA graph (how GaussianProcess runs it: "
                        "backend.LmlGraph), build time subtracted; cholesky_eager_ms: the same call launched eagerly from "
                        "Python (host launch overhead of ~700 kernels / events shows at N=5500)"}

    if args.no_phases:      # launch-list / ncu runs: only the timed loop and the e2e loop
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_total / K, "impl": "b200", "gpu_launches": int(launches), "e2e": e2e,
                "config": {"workload": workload_label(args.workload)}, "c4_scan": c4,
                "note": "--no-phases run (profiling aid), not a bench line"}
        print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    ph = phase_numbers(n, d, reps=3 if N < 10000 else 2)
    traffic, traffic_meta = None, None
    for name in (f"r02/dominant_kernel_ncu_{args.workload}.json", "r02/dominant_kernel_ncu.json",
                 "r01/dominant_kernel_ncu.json"):
        try:   # dram bytes of the dominant launch from the committed ncu --set full capture (per launch)
            tm = json.load(open(os.path.join(ROOT, "profiles", name)))
            traffic, traffic_meta = tm.get("dram_bytes_per_launch"), {k: tm.get(k) for k in
                                                                      ("source", "kernel", "grid_size", "duration_us",
                                                                       "dram_read_bytes", "dram_write_bytes",
                                                                       "algorithmic_bytes_per_launch", "algorithmic_flops_per_launch",
                                                                       "dmma_pipe_active_pct", "l2_hit_pct")}
            break
        except Exception:
            continue
    roofline = {"kernel": "fp64 DMMA.8x8x4 GEMM engine = all O(N^3) work of one evaluation (gemm_tma_nt_kernel<128,128,6 stages>: "
                          "TMA + mbarrier ring, one CTA per SM with the SM to itself, products with >= 400 tiles of 128x128; gemm_f64_kernel<64,64,..> / <32,32,..>: "
                          "cp.async ring, the smaller products and the K=128 updates beside the factorisation's chain)",
                "bound": "tensor", "achieved": N ** 3 / ph["gemm_ms_per_eval"] * 1e-9, "peak": dmma_peak,
                "unit": "TFLOP/s", "frac": N ** 3 / ph["gemm_ms_per_eval"] * 1e-9 / dmma_peak,
                "traffic": traffic, "traffic_capture": traffic_meta,
                "algorithmic_flops_per_eval": float(N) ** 3,
                "whole_step_frac": N ** 3 / (ms_total / K) * 1e-9 / dmma_peak,
                "note": "achieved = N^3 (SURVEY 8d: N^3/3 factor + 2N^3/3 inverse) / summed CUDA-event duration of all GEMM "
                        "launches of one evaluation (timed on the single-stream schedule: with the look-ahead on, launches of "
                        "different streams overlap); whole_step_frac = N^3 / ms_per_step / peak; peak = fp64 DMMA issue peak "
                        "measured in this run on this GPU (gegp_dmma_peak; MEASURED_PEAKS.json has no fp64 entry); traffic = "
                        "dram bytes of ONE captured launch of the kernel named in traffic_capture (committed ncu --set full "
                        "summary), beside that launch's algorithmic bytes",
                "hbm_build": {"bound": "hbm", "achieved": ph["build_full_gbs"], "peak": hbm_peak, "peak_source": hbm_src,
                              "unit": "GB/s", "frac": ph["build_full_gbs"] / hbm_peak, "bytes": 8.0 * N * N,
                              "lower_only_gbs": ph["build_lower_gbs"]}}
    extra = {"peaks_in_run": in_run}
    if world == 1:
        # batch point B (multi-start rows in lock step): several candidates per device call fill the GPU where one
        # N ~ 5000 evaluation is bound by the latency of its leaf chain.  Reported beside the headline, never instead.
        try:
            Bc = 4
            thb = torch.stack([bk.to_dev(step_theta(theta, 1000 + s, rank)) for s in range(Bc)])
            runb = lambda: bk.lml_eval(X_dev, y_dev, thb, mode=L.MODE_PRECON, eta=eta, want_grad=True)  # noqa: E731
            runb()
            msb = ev_ms(runb, 3)
            extra["batched"] = {"candidates_per_call": Bc, "ms_per_call": msb, "evals_per_s": Bc / (msb * 1e-3),
                                "note": "same workload, 4 candidate thetas per gegp_lml_eval call (lock-step multi-start)"}
        except Exception as exc:   # noqa: BLE001
            extra["batched"] = {"error": repr(exc)}

    # ---- the north-star size, first class: phases, e2e through the API, posterior at 10^4 points, parity vs the CPU port
    def c3_block():
        n3, d3 = WORKLOADS["c3"]
        N3 = n3 * (d3 + 1)
        out = phase_numbers(n3, d3, reps=2)
        x3, f3, g3, th3 = make_problem(n3, d3)
        G3 = GaussianProcess(d3, True, "SqExp", "precon")
        G3.set_data(x3, f3, np.zeros(n3), g3, np.zeros((n3, d3)))
        out["e2e"] = api_e2e(G3, th3, n3, d3, 3, warm=1)
        th_eval = step_theta(th3, W + 2, 0)
        info3, ok3 = G3.calc_lkd_all(G3.make_hp_class(theta=th_eval), calc_grad=True)
        # posterior at 10^4 test points through the public API (setup_eval_model + eval_model)
        xs = np.random.default_rng(1).uniform(-2.0, 2.0, (10000, d3))
        G3.set_hpara("set", 1, G3.make_hp_class(theta=th_eval, varK=info3.hp_varK, beta=info3.hp_beta))
        G3.eval_model(xs[:64])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mu, sig = G3.eval_model(xs)[:2]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out["predict_10k"] = {"ms": dt * 1e3, "points_per_s": 10000 / dt, "solve_tflops": N3 * N3 * 10000.0 / dt * 1e-12,
                              "solve_frac_of_dmma_peak": N3 * N3 * 10000.0 / dt * 1e-12 / dmma_peak,
                              "api": "GaussianProcess.eval_model(x2model[10000, 20]) with host buffers"}
        bk.free_workspace()
        torch.cuda.empty_cache()
        if not args.no_cpu_baseline:
            arm3 = CpuArm("c3")
            arm3.warm()
            t0 = time.perf_counter()
            r = arm3.O.lkd_wo_noise_lean(x3, f3, g3, th_eval, "precon", G3._etaK, calc_grad=True, Xs=xs[:256])
            dtc = time.perf_counter() - t0
            mu_r, sig_r, _ = r.post
            out["cpu"] = {"value": 1.0 / dtc, "unit": UNIT, "cores": arm3.cores, "kind": "port",
                          "sample": arm3.describe(1) + " (plus the posterior at 256 test points from the same factor)",
                          "speedup_e2e": out["e2e"]["value"] * dtc}
            out["parity_vs_cpu"] = {
                "lml_rel": abs(info3.ln_lkd - r.ln_lkd) / abs(r.ln_lkd),
                "grad_rel": float(np.max(np.abs(info3.ln_lkd_grad - r.ln_lkd_grad)) / np.max(np.abs(r.ln_lkd_grad))),
                "varK_rel": abs(info3.hp_varK - r.hp_varK) / r.hp_varK,
                "mu_rel": float(np.max(np.abs(mu[:256] - mu_r)) / np.max(np.abs(mu_r))),
                "sig2_abs_over_varK": float(np.max(np.abs(sig[:256] ** 2 - sig_r ** 2)) / r.hp_varK),
                "tolerance": 1e-8}
        return out

    if args.workload != "c3" and not args.no_c3 and world == 1:
        try:
            extra["c3"] = c3_block()
        except Exception as exc:  # noqa: BLE001 -- report, never hide
            extra["c3"] = {"error": repr(exc)}

    # ---- BASELINE configs[4]: N=51000 (20.8 GB) build + Cholesky, three conditioning modes
    def c5_block():
        n5, d5 = C5["n"], C5["d"]
        N5 = n5 * (d5 + 1)
        x5, f5, g5, th5 = make_problem(n5, d5)
        ld = bk.ld_of(N5)
        buf = torch.empty((N5, ld), dtype=torch.float64, device="cuda")
        dinv5 = bk.dinv_buffer(N5)
        res = {"n": n5, "d": d5, "N": N5, "matrix_GB": 8.0 * N5 * N5 * 1e-9}
        for mode in ("base", "rescale_origin", "precon"):
            G5 = GaussianProcess(d5, True, "SqExp", mode)
            G5.set_data(x5, f5, np.zeros(n5), g5, np.zeros((n5, d5)))
            xk, thk = G5.get_scl_x_w_dist()[0], th5
            if mode == "rescale_origin":      # the same GP in the rescaled coordinates: theta_s = theta / c^2
                thk = th5 / G5.DataScl.xvec_scale ** 2
            Xk, Tk = bk.to_dev(xk), bk.to_dev(thk)
            m = L.MODE_PRECON if mode == "precon" else L.MODE_BASE
            build = lambda uplo: bk.build_cov(Xk, Tk, mode=m, eta=G5._etaK, out=buf, uplo=uplo)  # noqa: E731
            ms_b = ev_ms(lambda: build(0), 2)
            ms_l = ev_ms(lambda: build(1), 2)
            info5 = [None]

            def fac():
                build(1)
                info5[0] = bk.potrf(buf, N5, 0, dinv5)[0]
            fac()
            ms_f = ev_ms(fac, 2) - ms_l
            res[mode] = {"eta": float(G5._etaK), "build_full_ms": ms_b, "build_full_gbs": 8.0 * N5 * N5 / ms_b * 1e-6,
                         "build_full_frac_of_hbm": 8.0 * N5 * N5 / ms_b * 1e-6 / hbm_peak,
                         "build_lower_gbs": 4.0 * N5 * (N5 + 1) / ms_l * 1e-6,
                         "cholesky_ms": ms_f, "cholesky_tflops": N5 ** 3 / 3 / ms_f * 1e-9,
                         "cholesky_frac_of_dmma_peak": N5 ** 3 / 3 / ms_f * 1e-9 / dmma_peak,
                         "info": int(info5[0].item())}
        del buf
        torch.cuda.empty_cache()
        return res

    if not args.no_c5 and world == 1:
        try:
            extra["c5"] = c5_block()
        except Exception as exc:  # noqa: BLE001
            extra["c5"] = {"error": repr(exc)}
    bk.free_workspace()
    torch.cuda.empty_cache()

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        arm = CpuArm(args.workload)
        arm.warm()
        th_last = step_theta(theta, W + K - 1, 0)
        t0 = time.perf_counter()
        lml_r, grad_r, _, _ = arm.eval(th_last)
        dt = time.perf_counter() - t0
        got = last.cpu().numpy()[0]
        cpu_baseline = {"value": 1.0 / dt, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.describe(1),
                        "parity_vs_gpu_last_step": {
                            "lml_rel": abs(got[L.OUT_LML] - lml_r) / abs(lml_r),
                            "grad_rel": float(np.max(np.abs(got[L.OUT_GRAD:] - grad_r)) / np.max(np.abs(grad_r)))}}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_label(args.workload),
                       "per_rank": "one evaluation per step; every rank evaluates its own candidate theta",
                       "l2": f"working set {3 * 8 * N * N / 1e6:.0f} MB per evaluation > 126 MB L2 and rewritten "
                             "from scratch every step (no reuse across steps); no explicit flush",
                       "seed": 0},
            "impl": "b200", "info_ok": info_ok, "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e,
            "roofline": roofline, "phases": ph, "cpu_baseline": cpu_baseline, "c4_scan": c4}
    line.update(extra)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-c3", action="store_true", help="skip the north-star (N=21000) block")
    ap.add_argument("--no-c4", action="store_true", help="skip the 1024-candidate scan (BASELINE configs[3])")
    ap.add_argument("--no-c5", action="store_true", help="skip the N=51000 build + Cholesky block (BASELINE configs[4])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-phases", action="store_true", help="profiling aid: skip the roofline / phase measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result rows of the last one to DIR/lml_eval_out.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA path computed; it needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
