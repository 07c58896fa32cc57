"""Crossover of the two logistic data-pass routes at small p: slab (one sweep, 2 launches) vs two sweeps (5 launches)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = r'''
import sys, time, json, numpy as np, torch
sys.path.insert(0, %r)
import oem_b200
dev = torch.device("cuda", 0)
out = {}
for n, p in ((50000, 8), (50000, 16), (50000, 32), (50000, 64), (1000000, 16), (1000000, 64)):
    g = torch.Generator(device=dev); g.manual_seed(n + p)
    Xt = torch.randn((p, n), generator=g, dtype=torch.float64, device=dev)
    b = torch.zeros(p, dtype=torch.float64, device=dev); b[:3] = torch.tensor([.3, -.3, .2], dtype=torch.float64)
    y = (torch.rand(n, generator=g, dtype=torch.float64, device=dev) < torch.sigmoid(Xt.t() @ b)).double()
    a = [Xt.t(), y, "binomial", ["lasso"], [], [], [], [], [], 40, 1e-3, 1.0, 3.0, 0.5, np.ones(p), True, True, False, dict(maxit=500, tol=1e-7)]
    best = 1e9
    for _ in range(3):
        torch.cuda.synchronize(); t0 = time.perf_counter(); r = oem_b200.oem_fit_logistic_dense(*a); torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    out["n=%%d p=%%d" %% (n, p)] = round(best * 1e3, 2)
print(json.dumps(out))
''' % ROOT
for route in ("slab", "sweeps"):
    env = dict(os.environ, OEMB200_LOGIT_ROUTE=route)
    r = subprocess.run([sys.executable, "-c", CHILD], env=env, capture_output=True, text=True)
    print("route", route, r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-400:])
