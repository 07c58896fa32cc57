"""Secondary measurement: oem_fit_logistic_sparse on an rsparsematrix-like design (n = 1e6 x 1000 at 1 % density by default),
device-resident dgCMatrix slots, three penalties.  X'WX and d are rebuilt on every IRLS data pass there, so the time is
the sparse Gram plus one path launch per IRLS iteration; prints the best and worst wall time of the repetitions, the
library's CUDA-event phase timings and its launch / sync counts."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oem_b200  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=1_000_000)
ap.add_argument("--p", type=int, default=1000)
ap.add_argument("--density", type=float, default=0.01)
ap.add_argument("--nlambda", type=int, default=20)
ap.add_argument("--reps", type=int, default=3)
a = ap.parse_args()
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev)
g.manual_seed(11)
per_col = max(1, int(a.n * a.density))
# every column draws `per_col` distinct rows (sorted), like a uniform-density dgCMatrix
rows = torch.empty((a.p, per_col), dtype=torch.int32, device=dev)
for j in range(a.p):
    rows[j] = torch.randperm(a.n, generator=g, device=dev)[:per_col].sort().values.int()
col_ptr = (torch.arange(a.p + 1, device=dev) * per_col).int()
vals = torch.randn(a.p * per_col, generator=g, dtype=torch.float64, device=dev)
beta = torch.zeros(a.p, dtype=torch.float64, device=dev)
beta[:25] = 2.0 * torch.rand(25, generator=g, dtype=torch.float64, device=dev) - 1.0
eta = torch.zeros(a.n, dtype=torch.float64, device=dev)
cols = torch.arange(a.p, device=dev).repeat_interleave(per_col)
eta.index_add_(0, rows.view(-1).long(), vals * beta[cols])
y = (torch.rand(a.n, generator=g, dtype=torch.float64, device=dev) < torch.sigmoid(eta)).double()
slots = (rows.view(-1), col_ptr, vals, (a.n, a.p))
args = [slots, y, "binomial", ["lasso", "mcp", "scad"], [], [], [], [], [], a.nlambda, 1e-2, 1.0, [3.0, 3.0, 3.7], 0.5,
        np.ones(a.p), True, True, False, dict(maxit=500, tol=1e-7)]
times = []
for _ in range(a.reps + 1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = oem_b200.oem_fit_logistic_sparse(*args)
    torch.cuda.synchronize()
    times.append(time.perf_counter() - t0)
times = times[1:]                      # the first call warms the modules and the allocator
st = out["stats"]
print(json.dumps({"config": f"oem_fit_logistic_sparse n={a.n} p={a.p} density={a.density} nnz={a.p * per_col} "
                            f"lasso+mcp+scad {a.nlambda} lambdas",
                  "wall_s_best": min(times), "wall_s_worst": max(times),
                  "phases_ms": {k: round(v, 3) for k, v in st.items() if k.startswith("ms_")},
                  "irls_iterations": int(sum(int(np.sum(v)) for v in out["niter"])), "data_passes": st["data_passes"],
                  "kernel_launches": st["kernel_launches"], "host_syncs": st["host_syncs"],
                  "oem_iterations": st["total_oem_iters"]}))
