"""Binomial cross-validation on one GPU: oem_xval_logistic_dense (arm a) against the work it replaces (arm b: the full
oem_fit_logistic_dense plus one fit per fold at the full fit's lambdas on device-resident training-row handles, and the
held-out score through predict_matrix).  Each fold's rows are gathered into its own handle before its fit is timed,
which is generous to arm b.  Sizes: BASELINE configs[3] (n = 2e6 x p = 1000, y from seed 104, lasso, 100 lambdas),
n = 2.5e5 x 1000, and the vignette's launch-bound n = 5e4 x 100; 10 folds.  Also the fused pass on its own (all 11 models
active) against the single-model slab pass and an in-run cuBLAS DGEMM rate.  One JSON line per size, the card's name
and power limit read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import oem_b200  # noqa: E402
from oem_b200 import api  # noqa: E402
from bench_configs import gen  # noqa: E402

dev = torch.device("cuda", 0)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def dgemm_tflops(n=8192, reps=5):
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    a @ b
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        a @ b
    e1.record()
    torch.cuda.synchronize()
    return 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) / 1e3) / 1e12


def measure_t(y, prob, tm):
    if tm == "deviance":
        pm = prob.clamp(1e-5, 1 - 1e-5)
        return -2.0 * ((1 - y)[:, None] * torch.log(1 - pm) + y[:, None] * torch.log(pm))
    raise ValueError(tm)


def args_for(X, y, nlambda, lam=None):
    p = X.shape[1]
    return [X, y, "binomial", ["lasso"], [], [], [], [], lam if lam is not None else [], nlambda, 1e-4, 1.0, 3.0, 0.5,
            np.ones(p), True, True, False, dict(maxit=500, tol=1e-7, irls_maxit=100, irls_tol=1e-3)]


def sync_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run_size(n, p, seed, nfolds, nlambda, dg):
    X, y = gen(n, p, seed, coef=[.15, .15, -.15, -.15, .25], binomial=True)
    foldid = (np.random.default_rng(seed).permutation(np.resize(np.arange(1, nfolds + 1), n))).astype(np.int32)
    fold_t = torch.from_numpy(foldid).to(dev)
    dm = oem_b200.DeviceMatrix(X)
    M = nfolds + 1

    # ---- arm a: the new entry on a DeviceMatrix (first call warms up every shape) ----
    xa = args_for(dm, y, nlambda)
    xa = xa[:17] + [nfolds, foldid, False, "deviance", xa[18]]
    oem_b200.oem_xval_logistic_dense(*xa)
    wall_a, ra = sync_time(lambda: oem_b200.oem_xval_logistic_dense(*xa))
    st = ra["stats"]

    # ---- arm b: full fit + nfolds fold fits (training rows gathered into their own handle before each timed fit) ----
    af = args_for(dm, y, nlambda)
    oem_b200.oem_fit_logistic_dense(*af)
    t_full, rf = sync_time(lambda: oem_b200.oem_fit_logistic_dense(*af))
    lam = [np.asarray(rf["lambda_"][0])[:rf["beta"][0].shape[1]]]
    t_folds, t_score, betas = [], 0.0, []
    T = torch.empty((n, lam[0].size), dtype=torch.float64, device=dev)
    for k in range(1, nfolds + 1):
        tr = torch.nonzero(fold_t != k).squeeze(1)
        hk = oem_b200.DeviceMatrix(X.t().index_select(1, tr).contiguous().t())
        yk = y.index_select(0, tr)
        t, rk = sync_time(lambda: oem_b200.oem_fit_logistic_dense(*args_for(hk, yk, nlambda, lam)))
        hk.close()
        t_folds.append(t)
        betas.append(rk["beta"][0])
        del hk, yk, tr
        te = torch.nonzero(fold_t == k).squeeze(1)
        xk = X.t().index_select(1, te).contiguous().t()
        out = torch.empty((te.numel(), lam[0].size), dtype=torch.float64, device=dev).t().contiguous().t()
        t, _ = sync_time(lambda: api.predict_matrix(xk, rk["beta"][0], response=True, out=out))
        t_score += t
        T[te] = measure_t(y.index_select(0, te), out, "deviance")
        del xk, out
    t0 = time.perf_counter()
    cvm_b = T.mean(0)
    torch.cuda.synchronize()
    t_score += time.perf_counter() - t0
    wall_b = t_full + sum(t_folds) + t_score
    del T

    # ---- the fused pass alone: all M models active, against one single-model slab pass ----
    L = api.load()
    B = torch.randn(M, p, dtype=torch.float64, device=dev) * (0.5 / p ** 0.5)
    b0 = torch.zeros(M, dtype=torch.float64, device=dev)
    fold_rows = fold_t.clone()
    _, ms_fused, ms_rl, sweeps = oem_b200.logit_fold_pass(X, B, b0, y, fold_rows, reps=10)
    grad1 = torch.empty(p + 1, dtype=torch.float64, device=dev)
    ms1, msr1 = ctypes.c_double(), ctypes.c_double()
    api._check(L.oemb200_logit_slab_pass(X.data_ptr(), n, p, X.stride(1), B[0].data_ptr(), 0.0, y.data_ptr(), None, None,
                                         grad1.data_ptr(), 10, None, ctypes.byref(ms1), ctypes.byref(msr1)))
    dm.close()
    del X
    torch.cuda.empty_cache()
    bytes_sweep = 8.0 * n * p
    ms_sweep = ms_fused / sweeps
    flop_pass = 4.0 * n * p * M
    return {
        "n": n, "p": p, "nfolds": nfolds, "nlambda": nlambda, "models": M,
        "arm_a_wall_s": wall_a, "arm_b_wall_s": wall_b, "speedup_b_over_a": wall_b / wall_a,
        "arm_b_full_fit_s": t_full, "arm_b_fold_fits_s": t_folds, "arm_b_score_s": t_score,
        "arm_a_phases_ms": {k: round(v, 3) for k, v in st.items() if k.startswith("ms_")},
        "arm_a_sweeps": st["data_passes"], "arm_a_host_syncs": st["host_syncs"],
        "arm_a_kernel_launches": st["kernel_launches"], "arm_a_fused_ms_per_sweep": st["ms_irls_xb"] / max(1, st["data_passes"]),
        "max_abs_dbeta_a_vs_b": float(np.max(np.abs(ra["beta"][0] - rf["beta"][0]))),
        "max_abs_dcvm_a_vs_b": float((torch.from_numpy(ra["cvm"][0]).to(dev) - cvm_b).abs().max()),
        "fused_pass": {"models": M, "sweeps": sweeps, "ms_per_pass": ms_fused, "ms_per_sweep": ms_sweep,
                       "relayout_ms": ms_rl, "gbs_per_sweep": bytes_sweep / (ms_sweep / 1e3) / 1e9,
                       "fp64_tflops": flop_pass / (ms_fused / 1e3) / 1e12, "single_model_slab_pass_ms": ms1.value,
                       "fused_over_single_sweep": ms_fused / ms1.value, "dgemm_tflops_in_run": dg,
                       "fp64_frac_of_dgemm": flop_pass / (ms_fused / 1e3) / 1e12 / dg},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="2000000x1000x104,250000x1000x105,50000x100x107", help="n x p x seed, comma-separated")
    ap.add_argument("--nfolds", type=int, default=10)
    ap.add_argument("--nlambda", type=int, default=100)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    info = card()
    dg = dgemm_tflops()
    lines = []
    for s in a.sizes.split(","):
        n, p, seed = (int(v) for v in s.split("x"))
        d = run_size(n, p, seed, a.nfolds, a.nlambda, dg)
        d["card"] = info
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
