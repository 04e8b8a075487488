import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gpgradpy_b200 import backend as bk
def ev(fn, reps=5):
    fn(); torch.cuda.synchronize(); best = 1e9
    for _ in range(reps):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1))
    return best
for (M, Nn, K, tb) in [(2048, 2048, 2048, True), (1536, 1536, 768, True), (2560, 1280, 1408, True), (2048, 2048, 128, True), (1200, 1200, 640, True)]:
    A = torch.randn((M, K), dtype=torch.float64, device="cuda")
    Bm = torch.randn((Nn, K) if tb else (K, Nn), dtype=torch.float64, device="cuda")
    Cm = torch.zeros((M, Nn), dtype=torch.float64, device="cuda")
    ms = ev(lambda: bk.dgemm(A, Bm, Cm, transb=tb))
    print(f"dgemm M={M} N={Nn} K={K} transb={tb}: {ms:.3f} ms  {2*M*Nn*K/ms*1e-9:.2f} TFLOP/s", flush=True)
