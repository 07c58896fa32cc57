"""Where does a logistic fit at an 8-GPU shard size (n = 2.5e5 x 1000 on one GPU) spend its wall time?  A/B of the driver's
knobs: legacy default stream vs an explicit stream, one-ahead speculation on / off."""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oem_b200  # noqa: E402

dev = torch.device("cuda", 0)
n, p = int(sys.argv[1]) if len(sys.argv) > 1 else 250000, 1000
g = torch.Generator(device=dev); g.manual_seed(104)
Xt = torch.randn((p, n), generator=g, dtype=torch.float64, device=dev)
b = torch.zeros(p, dtype=torch.float64, device=dev); b[:5] = torch.tensor([.15, .15, -.15, -.15, .25], dtype=torch.float64)
y = (torch.rand(n, generator=g, dtype=torch.float64, device=dev) < torch.sigmoid(Xt.t() @ b)).double()
X = Xt.t()
stream = torch.cuda.Stream()
for label, env, use_stream in (("legacy stream", {}, False), ("explicit stream", {}, True),
                               ("explicit, no speculation", {"OEMB200_IRLS_NO_SPECULATION": "1"}, True)):
    os.environ.pop("OEMB200_IRLS_NO_SPECULATION", None)
    os.environ.update(env)
    opts = dict(maxit=500, tol=1e-7)
    if use_stream:
        opts["stream"] = stream.cuda_stream
    args = [X, y, "binomial", ["lasso"], [], [], [], [], [], 100, 1e-4, 1.0, 3.0, 0.5, np.ones(p), True, True, False, opts]
    best = None
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = oem_b200.oem_fit_logistic_dense(*args)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    st = out["stats"]
    print(json.dumps({"case": label, "wall_ms": round(best * 1e3, 2), "ms_total": round(st["ms_total"], 2),
                      "ms_irls_xb": round(st["ms_irls_xb"], 2), "ms_path": round(st["ms_path"], 2),
                      "irls": int(np.sum(out["niter"][0])), "launches": st["kernel_launches"], "host_syncs": st["host_syncs"]}))
