"""Timing of pilco_gp_predict (GP predictive at B deterministic test points, diagonal variances) on one GPU.

    python scripts/predict_timing.py --out profiles/r03_predict_timing.json

At the metric (n=300, D=12, E=10) and swimmer (n=500, D=10, E=8) shapes and B in {1, 64, 1024, 1e5}: time per call with
CUDA events after warm-up, points/s and achieved fp64 TFLOP/s from 2 B n^2 E + B n (2D+2) E, against
  - the fp64 DMMA peak measured in the same process (pilco_microbench_fp64, as bench.py measures it),
  - cuBLAS DGEMM through torch.matmul (6144^3, same process),
  - a torch-CUDA composition of the same math (cdist -> exp -> matmul -> row dot; it materialises K*), timed alternately
    with the fused kernel in the same windows, and
  - the numpy factor identity on the host cores (one call per B, B <= 1024; not measured at 1e5).
The card's name, power limit and max SM clock are read with nvidia-smi in the same run.  The working set (iK of all
outputs: E pad(n)^2 doubles, 8.2 MB at the metric shape; test points and outputs: 16 MB at B = 1e5) fits the 126 MB L2:
iK is meant to stay L2-resident across calls, and the figures are for that regime.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from pilco_b200 import engine, _lib                       # noqa: E402
from pilco_b200._lib import lib                           # noqa: E402
from gp_predict_oracle import factor_predict_f            # noqa: E402
from util import make_gp_problem                          # noqa: E402

SHAPES = {"metric": (300, 12, 10), "swimmer": (500, 10, 8)}
BS = (1, 64, 1024, 100000)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + q,
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        name, pl, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as exc:                               # (reported, not fatal: the timings stand on their own)
        return {"name": torch.cuda.get_device_name(), "error": str(exc)}


def dmma_peak_tflops():
    sink = torch.zeros(8, dtype=torch.float64, device="cuda")
    ms = C.c_float()
    iters, blocks = 20000, 148 * 4
    _lib.check(lib.pilco_microbench_fp64(1, iters, blocks, engine.ptr(sink), C.byref(ms), engine.stream_ptr()))
    return blocks * 8 * iters * 8.0 * 512 / (ms.value * 1e-3) / 1e12


def dgemm_tflops(nmm=6144):
    a = torch.randn(nmm, nmm, dtype=torch.float64, device="cuda")
    b = torch.randn(nmm, nmm, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        torch.matmul(a, b)
    e1.record()
    torch.cuda.synchronize()
    return 3 * 2.0 * nmm ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12


def torch_predict(Xs, C_, ell, sf2, beta, iK):
    """The same predictive as a straightforward torch composition: K* [E,B,n] materialised."""
    Xe = Xs[None] / ell[:, None, :]
    Ce = C_[None] / ell[:, None, :]
    K = sf2[:, None, None] * torch.exp(-0.5 * torch.cdist(Xe, Ce) ** 2)
    mean = torch.bmm(K, beta[:, :, None])[..., 0].T
    var = (sf2[:, None] - (torch.bmm(K, iK) * K).sum(-1)).T
    return mean, var


def time_calls(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_predict_timing.json"))
    ap.add_argument("--reps", type=int, default=5, help="alternating fused / torch windows per point")
    args = ap.parse_args()
    engine.device()
    info = gpu_info()
    peak = dmma_peak_tflops()
    dgemm = dgemm_tflops()
    res = {"gpu": info, "dmma_peak_tflops_measured": peak, "cublas_dgemm_tflops_measured": dgemm,
           "host_cores": os.cpu_count(), "l2_note": "iK, test points and outputs fit the 126 MB L2 at every point",
           "flops_formula": "2 B n^2 E + B n (2D+2) E", "rows": []}
    for label, (n, D, E) in SHAPES.items():
        X, Y, ell, sf2, sn2 = make_gp_problem(n, D, E, seed=1)
        sn2 = 1e-3 * np.ones(E)
        gp = engine.gp_factorize(X, Y, ell, sf2, sn2)
        iKt = gp.iK[:, :n, :n].contiguous()
        ellt, sf2t = engine.dev(ell), engine.dev(sf2)
        iK_h, beta_h = iKt.cpu().numpy(), gp.beta.cpu().numpy()
        for B in BS:
            Xs = engine.dev(np.random.RandomState(2).rand(B, D))
            fused = lambda: engine.gp_predict(gp, Xs)
            comp = lambda: torch_predict(Xs, gp.X, ellt, sf2t, gp.beta, iKt)
            mf, vf = fused()
            mt, vt = comp()
            torch.cuda.synchronize()
            diff = {"mean": float((mf - mt).abs().max() / mt.abs().max()), "var": float((vf - vt).abs().max() / sf2t.max())}
            iters = 200 if B <= 1024 else 5
            for _ in range(2):                              # warm-up of both arms (allocator, cuBLAS heuristics)
                time_calls(fused, 3); time_calls(comp, 3)
            tf, tt = [], []
            for _ in range(args.reps):                      # alternate the two arms
                tf.append(time_calls(fused, iters))
                tt.append(time_calls(comp, iters))
            ms_f, ms_t = float(np.median(tf)), float(np.median(tt))
            ms_h = None                                     # (B = 1e5: K* alone is 2.4 GB per pass on the host; not measured)
            if B <= 1024:
                t0 = time.perf_counter()
                factor_predict_f(X, ell, sf2, iK_h, beta_h, np.random.RandomState(2).rand(B, D))
                ms_h = (time.perf_counter() - t0) * 1e3
            flops = 2.0 * B * n * n * E + B * n * (2 * D + 2) * E
            tfl = flops / (ms_f * 1e-3) / 1e12
            row = {"shape": label, "n": n, "D": D, "E": E, "B": B,
                   "fused_ms": ms_f, "fused_ms_windows": tf, "torch_ms": ms_t, "torch_ms_windows": tt, "numpy_host_ms": ms_h,
                   "points_per_s": B / (ms_f * 1e-3), "fused_tflops": tfl, "frac_dmma_peak": tfl / peak,
                   "ratio_vs_cublas_dgemm": tfl / dgemm, "speedup_vs_torch": ms_t / ms_f,
                   "torch_tflops": flops / (ms_t * 1e-3) / 1e12, "max_rel_diff_vs_torch": diff}
            res["rows"].append(row)
            print("%-8s B=%-6d fused %9.4f ms  torch %9.4f ms  numpy %s ms  %6.2f TFLOP/s (%.2f of DMMA peak, %.2f of DGEMM)"
                  % (label, B, ms_f, ms_t, "%.2f" % ms_h if ms_h is not None else "-", tfl, tfl / peak, tfl / dgemm), flush=True)
            del Xs, mf, vf, mt, vt
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "dmma_peak_tflops_measured", "cublas_dgemm_tflops_measured")}))


if __name__ == "__main__":
    main()
