"""Streamed cross-validation (oem_xval_big) from pinned host memory, one GPU.  Writes profiles/r03_bench_xval_big.jsonl
(one JSON line per workload, with the card's name, power limit and max SM clock read in the same run).
  (a) configs[2] shape, n = 1e7 x p = 500 (40 GB), 10 folds, lasso + grp.lasso + mcp, 100 lambdas: the streamed entry
      (default gigs) and the resident oem_xval_dense on the same pinned buffer, alternating; max |d beta| and max |d cvm|
      between the arms;
  (b) n = 1.25e7 x p = 1000 (100 GB), which the resident entry cannot hold next to its fold-sorted copy: streamed only.
Run the two workloads as two processes (--only a, --only b): the host keeps (a)'s pinned buffer cached otherwise.
Per pass: pass 1 (fold Grams) is stats.ms_h2d; "rest" = ms_total - ms_h2d - ms_path - ms_assemble is pass 2 (scoring)
plus the fold-count pre-pass and the coefficient build.  The pinned-copy probe copies the same bytes from the same
buffer to the device in gigs-sized chunks (cudaMemcpyAsync through torch), which is the floor of each pass."""
import argparse
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
from bench_configs import gen  # noqa: E402

dev = torch.device("cuda", 0)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q}


def pinned_problem(n, p, seed):
    """X (n x p column-major, pinned host numpy view), y (host), generated on the device column block by column block."""
    X, y = gen(n, p, seed, coef=[.5, .5, -.5, -.5, 1.0], noise=4.0)
    hx = torch.empty((p, n), dtype=torch.float64, pin_memory=True)
    step = max(1, (1 << 31) // (8 * n))
    for j in range(0, p, step):
        hx[j:j + step].copy_(X.t()[j:j + step, :n])
    yh = y.cpu().numpy()
    del X, y
    torch.cuda.empty_cache()
    return hx, hx.t().numpy(), yh


def copy_probe(hx, gigs, reps=2):
    """seconds to copy all bytes of hx (pinned) to the device in contiguous pieces of gigs GB: a plain pinned copy.  (A
    strided slice would take torch's staging path through pageable memory, several times slower than the DMA.)"""
    flat = hx.view(-1)
    step = int(gigs * 1e9 / 8)
    dst = torch.empty(step, dtype=torch.float64, device=dev)
    best = None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k0 in range(0, flat.numel(), step):
            k1 = min(flat.numel(), k0 + step)
            dst[:k1 - k0].copy_(flat[k0:k1], non_blocking=True)
        torch.cuda.synchronize()
        t = time.perf_counter() - t0
        best = t if best is None else min(best, t)
    del dst
    torch.cuda.empty_cache()
    return best


def args(X, y, p, F, foldid, gigs=None):
    groups = np.concatenate([[0], np.repeat(np.arange(1, p // 10 + 1), 10)])
    opts = dict(maxit=500, tol=1e-7, irls_maxit=100, irls_tol=1e-3)
    if gigs is not None:
        opts["gigs"] = gigs
    return [X, y, "gaussian", ["lasso", "grp.lasso", "mcp"], [], groups, np.unique(groups), [], [], 100, 1e-4, 1.0, 3.0, 0.5,
            np.ones(p), True, True, F, foldid, False, "mse", opts]


def run(fn, a):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn(*a)
    wall = time.perf_counter() - t0
    st = out["stats"]
    rec = {"wall_s": wall, "pass1_ms": st["ms_h2d"], "path_ms": st["ms_path"], "assemble_ms": st["ms_assemble"],
           "cvscore_kernel_ms": st["ms_cvscore"], "gram_kernel_ms": st["ms_gram"], "total_ms": st["ms_total"],
           "rest_ms": st["ms_total"] - st["ms_h2d"] - st["ms_path"] - st["ms_assemble"],
           "gram_launches": st["gram_launches"], "data_passes": st["data_passes"], "h2d_bytes": st["h2d_bytes"],
           "host_syncs": st["host_syncs"], "ingest_wait_ms": st["ms_ingest_wait"]}
    return out, rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--only", default="a", choices=["a", "b"], help="workload to run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bench_xval_big.jsonl"))
    args_ = ap.parse_args()
    L = oem_b200.load()
    gigs = oem_b200.make_opts().gigs
    F = 10

    def emit(rec):
        print(json.dumps(rec), flush=True)
        os.makedirs(os.path.dirname(args_.out), exist_ok=True)
        with open(args_.out, "a") as f:
            f.write(json.dumps(rec) + "\n")
    if args_.only == "a":
        n, p = 10_000_000, 500
        hx, X, y = pinned_problem(n, p, 103)
        foldid = (1 + np.random.default_rng(103).permutation(n) % F).astype(np.int32)
        probe = copy_probe(hx, gigs)
        arms = {"streamed": [], "resident": []}
        outs = {}
        for r in range(args_.reps + 1):          # rep 0 warms both arms
            for name, fn in (("streamed", oem_b200.oem_xval_big), ("resident", oem_b200.oem_xval_dense)):
                out, rec = run(fn, args(X, y, p, F, foldid))
                if r:
                    arms[name].append(rec)
                outs[name] = out
        db = max(float(np.max(np.abs(a - b))) for a, b in zip(outs["streamed"]["beta"], outs["resident"]["beta"]))
        dc = max(float(np.max(np.abs(a - b))) for a, b in zip(outs["streamed"]["cvm"], outs["resident"]["cvm"]))
        best = min(arms["streamed"], key=lambda r: r["total_ms"])
        emit({"workload": f"(a) configs[2] shape xval n={n:.3g} x p={p} ({n * p * 8 / 1e9:.0f} GB) {F} folds "
                                 "lasso+grp.lasso+mcp 100 lambdas, X in pinned host memory", "gigs": gigs, "card": card(),
                     "pinned_copy_probe_s": probe, "pinned_copy_probe_gbs": n * p * 8 / 1e9 / probe,
                     "pass1_frac_of_probe": probe * 1e3 / best["pass1_ms"],
                     "rest_frac_of_probe": probe * 1e3 / best["rest_ms"],
                     "streamed": arms["streamed"], "resident": arms["resident"],
                     "max_abs_dbeta_streamed_vs_resident": db, "max_abs_dcvm_streamed_vs_resident": dc})
    else:
        n, p = 12_500_000, 1000
        hx, X, y = pinned_problem(n, p, 104)
        foldid = (1 + np.random.default_rng(104).permutation(n) % F).astype(np.int32)
        probe = copy_probe(hx, gigs)
        runs = []
        for r in range(args_.reps + 1):
            _, rec = run(oem_b200.oem_xval_big, args(X, y, p, F, foldid))
            if r:
                runs.append(rec)
        try:
            oem_b200.oem_xval_dense(*args(X, y, p, F, foldid))
            resident = "ran"
        except oem_b200.OemB200Error as e:
            resident = f"refused: {e}"
        L.oemb200_release_cache()
        best = min(runs, key=lambda r: r["total_ms"])
        emit({"workload": f"(b) xval n={n:.3g} x p={p} ({n * p * 8 / 1e9:.0f} GB) {F} folds lasso+grp.lasso+mcp "
                                 "100 lambdas, X in pinned host memory", "gigs": gigs, "card": card(),
                     "pinned_copy_probe_s": probe, "pinned_copy_probe_gbs": n * p * 8 / 1e9 / probe,
                     "pass1_frac_of_probe": probe * 1e3 / best["pass1_ms"],
                     "rest_frac_of_probe": probe * 1e3 / best["rest_ms"], "streamed": runs,
                     "resident_oem_xval_dense": resident})


if __name__ == "__main__":
    main()
