#!/usr/bin/env python
"""bench.py -- headline benchmark of the OEM hot path on B200 (contract: see the task statement).

Workload (BASELINE.json configs[4], "big.oem-scale tall data n=1e8 p=1000 FP64 ... at 1/2/4/8 B200"):
one STEP = one full big.oem fit -- the one-pass Gram / X'y / column-sum build over the rank's row
shard (n = 1.25e7 x p = 1000 FP64 = 100 GB per GPU), the all-reduce of the packed sufficient
statistics over NVLink, the on-device Lanczos top eigenvalue and the warm-started 100-lambda path for
lasso + SCAD + MCP batched in one call.  Weak scaling: every rank holds 1.25e7 rows, so --gpus 8 is
exactly configs[4] (n = 1e8).  metric = full lambda-path fit time (s), lower is better.

  value      device-resident inputs (X, y already in HBM when the timed region starts)
  e2e        the same fit through the C ABI with HOST buffers (pinned); the library streams row chunks
             host->device inside the timed region and returns beta on the host.  h2d_peak_gbs is a plain
             pinned cudaMemcpyAsync of the same bytes on all ranks at once (the e2e leg's own roofline)
  roofline   the Gram kernel (FP64 DMMA SYRK): algorithmic n*p*(p+1) flops / CUDA-event kernel time,
             against the FP64 tensor peak measured in-run with cuBLAS DGEMM (MEASURED_PEAKS.json has
             no FP64 entry)
  secondary  the other sharded paths under the same clock, STRONG scaling (fixed total n, rows split over the
             ranks): configs[3] logistic lasso n = 2e6 x 1000 (fused single-sweep IRLS data pass, one
             (p+1)-vector all-reduce per pass) and configs[2] xval.oem 10-fold n = 1e7 x 500, with per-phase
             milliseconds, achieved GB/s / TFLOP/s, all-reduce count and latency, the limiting phase, and a
             parity number: small sharded fits against the same fits on rank 0 alone
  cpu_baseline / --impl reference   the CPU oracle (restated reference algorithm, numpy/OpenBLAS +
             plain C; the reference itself cannot be built here: no R / Rcpp / Eigen) on the box's host
             cores.  --impl reference at N = 1 MEASURES full-size fits (1.25e7 x 1000, 100 GB in host RAM)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P = 1000
ROWS_PER_GPU = 12_500_000
PENALTIES = ["lasso", "scad", "mcp"]
GAMMAS = [3.0, 3.7, 3.0]
NLAMBDA = 100
OPTS = dict(maxit=500, tol=1e-7)
# secondary workloads (SURVEY.md 8d): fixed TOTAL size, defined block by block so that any sharding sees the same data
LOGIT = dict(n=2_000_000, p=1000, blocks=8, seed=104, coef=[.15, .15, -.15, -.15, .25])
XVAL = dict(n=10_000_000, p=500, blocks=8, seed=103, coef=[.5, .5, -.5, -.5, 1.0], folds=10, noise=4.0)


def fit_args(X, y):
    p = P
    return [X, y, "gaussian", PENALTIES, [], [], [], [], [], NLAMBDA, 1e-4, 1.0, GAMMAS, 0.5, np.ones(p), True, True,
            False, dict(OPTS)]


def workload_name(n_gpus, rows):
    return (f"configs[4] big.oem n={rows * n_gpus:.3g} x p={P} FP64 ({rows:.3g} rows = {rows * P * 8 / 1e9:.0f} GB "
            f"per GPU, weak scaling), lasso+scad+mcp, 100 lambdas, standardize, intercept, tol 1e-7")


# ----------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi during the timed region
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, power = [], [], set(), []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, w in zip(sm, power) if w > 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(power)), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle (numpy/OpenBLAS data passes + plain-C OEM iterations) on the box's host cores
# ----------------------------------------------------------------------------------------------
def host_cores():
    return len(os.sched_getaffinity(0))


class BlasThreads:
    """Pin the BLAS / OpenMP pools to `n` threads for the duration (torchrun exports OMP_NUM_THREADS=1 when
    nproc > 1, which silently made the round-1 N >= 2 CPU arm single-threaded) and report what was actually set."""

    def __init__(self, n):
        self.n = int(n)
        self.ctx = None
        self.used = None

    def __enter__(self):
        try:
            from threadpoolctl import threadpool_info, threadpool_limits
            self.ctx = threadpool_limits(limits=self.n)
            self.ctx.__enter__()
            pools = [(d.get("user_api"), d.get("internal_api"), d.get("num_threads")) for d in threadpool_info()]
            blas = [t for api, _, t in pools if api == "blas"]
            self.used = int(max(blas)) if blas else None
            self.pools = pools
        except ImportError:
            self.used, self.pools = None, []
        return self

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def gen_host_matrix(rows, p, seed, threads):
    """X ~ N(0,1) rows x p column-major in host RAM and y = X b + N(0,1), generated column by column on `threads` threads
    (numpy releases the GIL inside standard_normal)."""
    from concurrent.futures import ThreadPoolExecutor
    X = np.empty((rows, p), order="F")
    rng = np.random.default_rng(seed)
    b = np.zeros(p)
    b[:25] = rng.uniform(-0.5, 0.5, 25)

    def fill(j):
        g = np.random.Generator(np.random.Philox(key=seed * 100_003 + j))
        g.standard_normal(out=X[:, j])

    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(fill, range(p)))
    y = np.random.Generator(np.random.Philox(key=seed * 100_003 + p)).standard_normal(rows)
    for j in range(25):
        y += X[:, j] * b[j]
    return X, y


def cpu_data_pass_time(X, y):
    """The passes over X of oem_fit_big on their own (what scales with n)."""
    t0 = time.perf_counter()
    _ = X.T @ y; _ = np.ones(X.shape[0]) @ X
    for j in range(X.shape[1]):
        _ = np.dot(X[:, j], X[:, j])
    _ = X.T @ X
    return time.perf_counter() - t0


def cpu_fit_sample(rows_full, sample_rows, steps, warmup, threads, seed=1234):
    """oracle.oem_fit_big on `sample_rows` rows with `threads` BLAS threads; the O(n) data passes are timed again on
    their own and extrapolated linearly to rows_full; the O(p^2) path phase (total - data passes) is not scaled."""
    from oracle import oracle as orc
    orc.build()
    X, y = gen_host_matrix(sample_rows, P, seed, host_cores())
    est, parts = [], []
    with BlasThreads(threads) as bt:
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            orc.oem_fit_big(*fit_args(X, y))
            total = time.perf_counter() - t0
            t_data = min(cpu_data_pass_time(X, y), total)
            t_path = max(total - t_data, 0.0)
            if it >= warmup:
                est.append(t_data * (rows_full / sample_rows) + t_path)
                parts.append((t_data, t_path))
    return float(np.mean(est)), {"cores": bt.used or threads, "sample_rows": sample_rows, "kind": "port",
                                 "t_data_sample_s": float(np.mean([p[0] for p in parts])),
                                 "t_path_s": float(np.mean([p[1] for p in parts]))}


def cpu_c_rowslice(sample_rows, threads, seed=4321):
    """The plain-C OpenMP row-slice X'X of src/oem_dense.h:328-358 (oracle_xtx: ncores slices of floor(n/ncores) rows,
    private p x p partials, critical-section sum) on a bounded sample: seconds and GFLOP/s, all cores and one thread."""
    from oracle import oracle as orc
    X, _ = gen_host_matrix(sample_rows, P, seed, host_cores())
    out = {"rows": sample_rows, "what": "oracle_xtx (plain C, OpenMP row slices like src/oem_dense.h:328-358)"}
    flops = float(sample_rows) * P * (P + 1)
    for name, nc in (("all_cores", threads), ("one_thread", 1)):
        rows = sample_rows if nc > 1 else max(2000, sample_rows // 8)
        t0 = time.perf_counter()
        orc.xtx_port(X[:rows], ncores=nc)
        dt = time.perf_counter() - t0
        out[name] = {"threads": nc, "rows": rows, "seconds": dt, "gflops": float(rows) * P * (P + 1) / dt / 1e9}
    out["flops_sample"] = flops
    return out


def run_reference(args):
    """--impl reference: the CPU implementation of the path on the host cores (the oracle port: the reference itself
    cannot be built in this image).  Rank 0 only.  N = 1: every timed step is a MEASURED full-size fit (1.25e7 x 1000
    rows generated in host RAM) while the time budget allows; otherwise, and at N > 1 (n = N x 1.25e7 does not fit host
    RAM), steps are bounded samples whose data passes are scaled linearly -- the line says which."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    rows, N = args.rows, args.gpus
    cores = host_cores()
    budget = float(os.environ.get("OEMB200_REF_BUDGET_S", "1500"))
    t_start = time.perf_counter()
    # untimed warm-up steps on a small sample (page in numpy / OpenBLAS, spin up the thread pools)
    sec_small, info_small = cpu_fit_sample(rows * N, args.cpu_sample_rows, 1, max(1, min(args.warmup, 2)), cores)
    avail = int(open("/proc/meminfo").read().split("MemAvailable:")[1].split()[0]) * 1024
    need = rows * P * 8 * 1.12 + (4 << 30)
    full_ok = (N == 1) and avail > need and sec_small * 1.3 < budget
    times, detail = [], {}
    if full_ok:
        X, y = gen_host_matrix(rows, P, 105, cores)
        with BlasThreads(cores) as bt:
            for k in range(args.steps):
                t0 = time.perf_counter()
                orc.oem_fit_big(*fit_args(X, y))
                times.append(time.perf_counter() - t0)
                spent = time.perf_counter() - t_start
                if k + 1 < args.steps and spent + 1.15 * np.mean(times) * (args.steps - k - 1) > budget:
                    break
            used = bt.used or cores
        measured_steps = len(times)
        sec = float(np.mean(times))
        if measured_steps < args.steps:
            # not enough budget for all K full-size steps: the remaining steps are bounded samples (extrapolated)
            rem = args.steps - measured_steps
            sec_s, _ = cpu_fit_sample(rows, args.cpu_sample_rows, rem, 0, cores)
            detail["remaining_steps_sampled_s"] = sec_s
        del X, y
        sample = (f"oracle.oem_fit_big MEASURED at full size {rows} x {P} ({rows * P * 8 / 1e9:.0f} GB in host RAM), "
                  f"{measured_steps} of {args.steps} timed steps at full size")
        detail.update({"measured": True, "measured_full_size_steps": measured_steps, "step_seconds": [round(t, 2) for t in times],
                       "extrapolated_from_sample_s": sec_small})
    else:
        # bounded sample per step; data passes scaled to the N-shard workload
        srows = int(min(rows, max(args.cpu_sample_rows, 2_000_000 if avail > (40 << 30) else args.cpu_sample_rows)))
        sec, info = cpu_fit_sample(rows * N, srows, args.steps, 0, cores)
        used = info["cores"]
        sample = (f"oracle.oem_fit_big on {srows} x {P} rows per step; data passes scaled x{rows * N / srows:.1f} to "
                  f"n={rows * N:.3g}, path phase unscaled")
        detail.update({"measured": False, "t_data_sample_s": info["t_data_sample_s"], "t_path_s": info["t_path_s"]})
    line = {"impl": "reference", "metric": "full lambda-path fit time", "value": sec, "unit": "s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.gpus, rows)},
            "cpu_baseline": dict({"value": sec, "unit": "s", "cores": used, "host_cores": cores, "kind": "port", "sample": sample},
                                 **detail),
            "e2e": {"value": sec, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def gen_shard(torch, rows, seed, device):
    """X ~ N(0,1) rows x P column-major on the device, y = X b + N(0,1) (SURVEY.md 8d, config 5)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    ld = rows + (rows & 1)
    Xt = torch.empty((P, ld), dtype=torch.float64, device=device)        # row j = column j of X
    gb = torch.Generator(device="cpu"); gb.manual_seed(105)
    b = torch.zeros(P, dtype=torch.float64)
    b[:25] = torch.rand(25, generator=gb, dtype=torch.float64) - 0.5
    b = b.to(device)
    y = torch.randn(rows, generator=g, dtype=torch.float64, device=device)
    step = 25
    for j in range(0, P, step):
        blk = Xt[j:j + step]
        blk.normal_(generator=g)
        y += blk[:, :rows].t() @ b[j:j + step]
    if ld != rows:
        Xt[:, rows:] = 0
    return Xt.t()[:rows], y            # view with stride (1, ld)


def gen_blocked_rows(torch, cfg, r0, r1, device, binomial):
    """Rows [r0, r1) of a dataset that is DEFINED block by block (cfg['blocks'] equal row blocks, one generator seed per
    block), so that every sharding of the rows -- 1, 2, 4 or 8 ranks -- sees exactly the same matrix.  Returns the
    column-major shard and its response (gaussian: X b + noise; binomial: Bernoulli(sigmoid(X b)))."""
    n, p, nb = cfg["n"], cfg["p"], cfg["blocks"]
    bl = (n + nb - 1) // nb
    rows = r1 - r0
    ld = rows + (rows & 1)
    Xt = torch.zeros((p, ld), dtype=torch.float64, device=device)
    y = torch.empty(rows, dtype=torch.float64, device=device)
    coef = torch.tensor(cfg["coef"], dtype=torch.float64, device=device)
    for b in range(nb):
        b0, b1 = b * bl, min(n, (b + 1) * bl)
        lo, hi = max(b0, r0), min(b1, r1)
        if lo >= hi:
            continue
        g = torch.Generator(device=device)
        g.manual_seed(cfg["seed"] * 1000 + b)
        eta = torch.zeros(b1 - b0, dtype=torch.float64, device=device)
        cstep = max(1, min(p, (1 << 27) // (b1 - b0)))
        for j in range(0, p, cstep):
            blk = torch.empty((min(cstep, p - j), b1 - b0), dtype=torch.float64, device=device)
            blk.normal_(generator=g)
            for jj in range(j, min(j + blk.shape[0], len(cfg["coef"]))):
                eta += coef[jj] * blk[jj - j]
            Xt[j:j + blk.shape[0], lo - r0:hi - r0] = blk[:, lo - b0:hi - b0]
            del blk
        if binomial:
            u = torch.rand(b1 - b0, generator=g, dtype=torch.float64, device=device)
            yb = (u < torch.sigmoid(eta)).double()
        else:
            yb = eta + cfg.get("noise", 1.0) * torch.randn(b1 - b0, generator=g, dtype=torch.float64, device=device)
        y[lo - r0:hi - r0] = yb[lo - b0:hi - b0]
    return Xt.t()[:rows], y


def measure_fp64_peak(torch, device):
    N = 8192
    a = torch.randn(N, N, dtype=torch.float64, device=device)
    b = torch.randn(N, N, dtype=torch.float64, device=device)
    for _ in range(2):
        torch.matmul(a, b)
    best = 1e9
    for _ in range(4):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); torch.matmul(a, b); e.record(); torch.cuda.synchronize()
        best = min(best, s.elapsed_time(e) / 1e3)
    del a, b
    return 2.0 * N ** 3 / best / 1e12


def hbm_peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6550.0, "fallback (B200_PROFILING.md: ~6.55 TB/s measured copy bandwidth)"


def dump_outputs(out_dir, fit):
    """Write what one oem_fit_big call returned as float64 .npy files, one set per penalty (a few MB at p = 1000), so that
    two builds run with the same arguments, and therefore on the same seeded inputs, can be compared array by array."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"d": np.array([fit["d"]])}
    for k, pen in enumerate(PENALTIES):
        for key in ("beta", "lambda_", "niter", "loss"):
            arrays[f"{key.rstrip('_')}_{pen}"] = fit[key][k]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_ours(args):
    import torch
    import oem_b200
    from oem_b200 import api
    from oem_b200.dist import Comm, LibComm
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    comm = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
        # default: the library's own communicator (ncclAllReduce + one-shot NVLink peer kernel issued by the library on
        # its stream); --comm callback routes the all-reduces through torch.distributed instead
        if args.comm == "callback":
            comm = Comm()
        else:
            # every rank must end up with the same transport: agree on whether the in-library communicator came up
            try:
                comm = LibComm(device=local)
                ok = 1.0
            except Exception as e:                      # e.g. no libnccl.so.2 to dlopen
                print(f"[bench] rank {rank}: in-library communicator unavailable ({e!r})", file=sys.stderr, flush=True)
                comm, ok = None, 0.0
            flag = torch.tensor([ok], dtype=torch.float64, device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() < 0.5:
                if comm is not None:
                    comm.close()
                comm = Comm()
                args.comm = "callback"
    api.load()
    rows = args.rows
    fp64_peak = measure_fp64_peak(torch, device)
    X, y = gen_shard(torch, rows, 105_000 + rank, device)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    opts = api.make_opts(dict(OPTS, stream=stream.cuda_stream), comm)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """barrier + sync on both sides, CUDA events on the launching stream, max over ranks."""
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(stream)
        outs, walls = [], []
        for _ in range(steps):
            t0 = time.perf_counter()
            outs.append(fn())
            walls.append(round((time.perf_counter() - t0) * 1e3, 2))
        e.record(stream)
        timed.last_walls = walls
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], dtype=torch.float64, device=device)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms.item()) / steps, outs

    a_dev = fit_args(X, y)
    a_dev[-1] = opts

    def step_dev():
        return oem_b200.oem_fit_big(*a_dev)

    for _ in range(args.warmup):
        step_dev()
    sampler = ClockSampler(local)
    sampler.start()
    ms_step, outs = timed(step_dev, args.steps)
    walls_dev = timed.last_walls
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs[-1])
    st = outs[-1]["stats"]
    gram_ms = float(np.mean([o["stats"]["ms_gram"] / max(1, o["stats"]["gram_launches"]) for o in outs]))
    gram_flops = st["gram_flops"] / max(1, st["gram_launches"])
    achieved = gram_flops / (gram_ms / 1e3) / 1e12
    launches = int(sum(o["stats"]["kernel_launches"] for o in outs))

    traffic, traffic_note = None, None
    try:       # per-launch DRAM bytes of the Gram kernel from the committed ncu capture of this exact launch shape
        tj = json.load(open(os.path.join(ROOT, "profiles", "gram_traffic.json")))
        if tj["rows"] == rows and tj["p"] == P:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            traffic_note = "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu capture in profiles/gram_traffic.json"
    except Exception:
        pass
    sm_count = torch.cuda.get_device_properties(device).multi_processor_count
    sm_mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 0.0
    dmma_limit = 4 * 512 / 16 * sm_count * sm_mhz * 1e6 / 1e12
    line = {"metric": "full lambda-path fit time", "value": ms_step / 1e3, "unit": "s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": False,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(world, rows), "l2": "inputs (100 GB/GPU) exceed L2; no flush needed",
                       "phases_ms": {k: st[k] for k in ("ms_colstats", "ms_gram", "ms_gram_reduce", "ms_allreduce",
                                                        "ms_assemble", "ms_path", "ms_total")},
                       "oem_iterations": st["total_oem_iters"], "lanczos_steps": st["lanczos_steps"],
                       "allreduce": {"transport": ("single process" if world == 1 else
                                                   ("torch.distributed callback" if args.comm == "callback" else
                                                    f"in-library (NCCL + NVLink peer kernel: {'on' if comm.p2p else 'off'})")),
                                     "calls_per_step": st["allreduce_calls"], "doubles_per_step": st["allreduce_doubles"]},
                       "host_wall_ms_per_step": walls_dev, "lib_ms_total_per_step": [round(o["stats"]["ms_total"], 2) for o in outs]},
            "clocks": clocks, "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "gram_syrk_kernel (FP64 DMMA.8x8x4, TMA-staged)",
                         "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
                         "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_note,
                         "algorithmic_bytes_per_launch": 8.0 * rows * P,
                         "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                         "algorithmic_flops_per_launch": gram_flops, "ms_per_launch": gram_ms,
                         # second yardstick: one DMMA.8x8x4 (512 flop) per 16 cycles per SM sub-partition
                         # (tools/micro/fp64_lat.cu) x 4 sub-partitions x SMs x the sampled SM clock
                         "dmma_issue_limit_tflops": dmma_limit,
                         "frac_of_dmma_issue_limit": achieved / dmma_limit if dmma_limit else None}}

    # ---- e2e: HOST buffers through the same C-ABI call ----
    if not args.no_e2e:
        e2e = run_e2e(torch, api, oem_b200, X, y, rows, opts, timed, args, st)
        line["e2e"] = e2e
    del X, y, a_dev
    torch.cuda.empty_cache()
    oem_b200.api.load().oemb200_release_cache()
    # ---- secondary: configs[3] logistic and configs[2] xval.oem, strong scaling, + cross-rank parity ----
    if not args.no_secondary:
        try:
            line["secondary"] = run_secondary(torch, api, oem_b200, comm, opts, timed, barrier, args, device, stream)
        except Exception as e:                                  # never lose the headline line to a secondary leg
            import traceback
            line["secondary"] = {"error": repr(e), "trace": traceback.format_exc()[-1500:]}
    # ---- CPU baseline (rank 0, N = 1 only) ----
    if rank == 0 and world == 1 and not args.no_cpu:
        torch.cuda.empty_cache()
        cores = host_cores()
        sec, info = cpu_fit_sample(rows, args.cpu_sample_rows, 1, 1, cores)
        cb = {"value": sec, "unit": "s", "cores": info["cores"], "host_cores": cores, "kind": "port",
              "sample": f"oracle.oem_fit_big on {info['sample_rows']} x {P} rows; data passes scaled "
                        f"x{rows / info['sample_rows']:.1f} to n={rows:.3g}, path phase unscaled "
                        "(bench.py --impl reference measures the full-size fit)"}
        try:
            one, info1 = cpu_fit_sample(rows, max(20_000, args.cpu_sample_rows // 4), 1, 1, 1)
            cb["one_thread"] = {"value": one, "unit": "s", "cores": info1["cores"], "sample_rows": info1["sample_rows"]}
            cb["c_openmp_rowslice"] = cpu_c_rowslice(min(100_000, args.cpu_sample_rows), cores)
        except Exception as e:                                   # reported extras, never a reason to lose the line
            cb["extras_error"] = repr(e)
        line["cpu_baseline"] = cb
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        if hasattr(comm, "close"):
            comm.close()
        torch.distributed.destroy_process_group()


def run_e2e(torch, api, oem_b200, X, y, rows, opts, timed, args, st_dev):
    """Same fit, inputs in pinned HOST memory; H2D of the row chunks and D2H of beta inside the timed region.  Then the
    leg's own roofline: a plain pinned cudaMemcpyAsync of the same bytes on all ranks at once."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    avail = int(open("/proc/meminfo").read().split("MemAvailable:")[1].split()[0]) * 1024
    budget = int(avail * 0.8 / world)
    rows_h = min(rows, budget // (P * 8) // 72 * 72)
    if world > 1:       # MemAvailable is read at slightly different moments on every rank: agree on one answer
        t = torch.tensor([float(rows_h)], dtype=torch.float64, device=X.device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MIN)
        rows_h = int(t.item())
    if rows_h < rows and not args.allow_partial_e2e:
        return {"value": None, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": f"host RAM cannot hold the {rows * P * 8 / 1e9:.0f} GB shard per rank ({avail / 1e9:.0f} GB available "
                        f"for {world} ranks); no end-to-end number"}
    Xh = torch.empty((P, rows_h), dtype=torch.float64)
    cudart = torch.cuda.cudart()
    nbytes = Xh.numel() * 8
    rc = cudart.cudaHostRegister(Xh.data_ptr(), nbytes, 0)
    pinned = (int(rc) == 0)
    if not pinned:
        # a box whose pinned-memory limit cannot take every rank's shard (seen: 2 x 100 GB on a 251 GB host).  The failed
        # call leaves its code in the runtime's last-error slot, where torch's next launch check would find it: drain it
        # with a throw-away launch, then run this rank's leg from pageable memory (the library stages it through its
        # pinned bounce ring)
        print(f"[bench] rank {os.environ.get('RANK', '0')}: cudaHostRegister({nbytes / 1e9:.0f} GB) failed with code {int(rc)}; "
              "e2e leg uses pageable host memory on this rank", file=sys.stderr, flush=True)
        try:
            torch.zeros(1, device=X.device).add_(1)
            torch.cuda.synchronize()
        except RuntimeError:
            pass
    all_pinned = pinned
    if world > 1:
        flag = torch.tensor([1.0 if pinned else 0.0], dtype=torch.float64, device=X.device)
        torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN)
        all_pinned = bool(flag.item() > 0.5)
    step = 50
    for j in range(0, P, step):
        Xh[j:j + step].copy_(X.t()[j:j + step, :rows_h], non_blocking=False)
    yh = y[:rows_h].cpu().numpy()
    Xh_np = Xh.numpy().T                       # rows_h x P, column-major view
    a = fit_args(Xh_np, yh)
    a[-1] = opts
    opts.gigs = args.gigs

    def step_host():
        return oem_b200.oem_fit_big(*a)

    for _ in range(max(1, args.warmup - 1)):
        step_host()
    ms, outs = timed(step_host, args.steps)
    s = outs[-1]["stats"]
    out = {"value": ms / 1e3, "unit": "s", "h2d_bytes_per_step": int(s["h2d_bytes"]),
           "d2h_bytes_per_step": int(s["d2h_bytes"]), "host_memory": "pinned (cudaHostRegister)" if all_pinned else "pageable on at least one rank (cudaHostRegister refused)",
           "rows_per_gpu": rows_h, "stream_chunk_gb": args.gigs}
    # the leg's roofline: plain pinned H2D copies of the same number of bytes, all ranks at once (max over ranks).  The
    # source is a separate 2 GB pinned buffer sent repeatedly, so the probe does not depend on whether this host let
    # every rank pin its whole shard.
    try:
        piece = torch.empty(1 << 28, dtype=torch.float64, pin_memory=True)          # 2 GB
        piece.normal_()
        dst = torch.empty(2, 1 << 28, dtype=torch.float64, device=X.device)
        reps = max(1, int(round(nbytes / (piece.numel() * 8))))
        def probe():
            for i in range(reps):
                dst[i & 1].copy_(piece, non_blocking=True)
            return None
        probe()
        pms, _ = timed(probe, 2)
        gbs = reps * piece.numel() * 8 / (pms / 1e3) / 1e9
        out["h2d_peak_gbs"] = gbs
        out["h2d_peak_what"] = (f"plain cudaMemcpyAsync from pinned host memory, {reps} x 2 GB = {reps * piece.numel() * 8 / 1e9:.0f} GB per rank, "
                                f"{world} rank(s) at once, device-timed, max over ranks")
        out["h2d_achieved_gbs"] = s["h2d_bytes"] / (ms / 1e3) / 1e9
        out["frac"] = out["h2d_achieved_gbs"] / gbs
        out["h2d_aggregate_gbs"] = gbs * world
        if not all_pinned:
            out["ingest"] = "pageable source staged through the library's pinned bounce ring + reader threads (csrc/ingest.cu)"
        del piece, dst
    except Exception as e:
        out["h2d_probe_error"] = repr(e)
    if pinned:
        cudart.cudaHostUnregister(Xh.data_ptr())
    if all_pinned and world == 1:      # single-process only: at N > 1 the pinned figure above is the e2e number
        # the same call once more from PAGEABLE memory (what an R matrix or a numpy array is): the library stages it through
        # its pinned bounce ring + reader threads (csrc/ingest.cu).  Reported next to the pinned figure, not instead of it.
        try:
            step_host()
            pms2, outs2 = timed(step_host, 2)
            s2 = outs2[-1]["stats"]
            out["from_pageable"] = {"value": pms2 / 1e3, "unit": "s", "h2d_achieved_gbs": s2["h2d_bytes"] / (pms2 / 1e3) / 1e9,
                                    "host_fill_ms": s2["ms_ingest_wait"],
                                    "what": "identical call, host buffer not pinned: pinned bounce ring + reader threads inside the library"}
        except Exception as e:
            out["from_pageable"] = {"error": repr(e)}
    if rows_h < rows:
        out["note"] = f"host buffer holds {rows_h} of {rows} rows per rank"
    return out


# ----------------------------------------------------------------------------------------------
# secondary workloads
# ----------------------------------------------------------------------------------------------
def _max_over_ranks(torch, v, device, world):
    t = torch.tensor([float(v)], dtype=torch.float64, device=device)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def run_secondary(torch, api, oem_b200, comm, opts, timed, barrier, args, device, stream):
    from oem_b200.dist import shard_rows
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    hbm, hbm_src = hbm_peak_gbs()
    out = {"scaling": "strong (fixed total n, contiguous row shards)", "hbm_peak_gbs": hbm, "hbm_peak_source": hbm_src}
    steps = max(1, args.secondary_steps)

    # ---- all-reduce latency of the (p+1)-vector, on its own ----
    if world > 1 and hasattr(comm, "all_reduce"):
        t = torch.ones(LOGIT["p"] + 1, dtype=torch.float64, device=device)
        for _ in range(5):
            comm.all_reduce(t, stream=stream.cuda_stream)
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(stream)
        for _ in range(100):
            comm.all_reduce(t, stream=stream.cuda_stream)
        e.record(stream)
        torch.cuda.synchronize()
        big = torch.ones(P * P + 3 * P + 3, dtype=torch.float64, device=device)
        comm.all_reduce(big, stream=stream.cuda_stream)
        barrier()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s2.record(stream)
        for _ in range(10):
            comm.all_reduce(big, stream=stream.cuda_stream)
        e2.record(stream)
        torch.cuda.synchronize()
        out["allreduce_probe"] = {"vector_doubles": LOGIT["p"] + 1, "vector_us": s.elapsed_time(e) * 1e3 / 100,
                                  "vector_transport": "one-shot NVLink peer-memory kernel" if comm.p2p else "ncclAllReduce",
                                  "bundle_doubles": int(big.numel()), "bundle_us": s2.elapsed_time(e2) * 1e3 / 10,
                                  "bundle_transport": "ncclAllReduce"}
        del big, t

    # ---- configs[3]: logistic lasso n = 2e6 x 1000, rows sharded over the ranks ----
    cfg = LOGIT
    r0, r1 = shard_rows(cfg["n"], rank, world)
    X, y = gen_blocked_rows(torch, cfg, r0, r1, device, binomial=True)
    a = [X, y, "binomial", ["lasso"], [], [], [], [], [], 100, 1e-4, 1.0, 3.0, 0.5, np.ones(cfg["p"]), True, True, False, opts]
    fn = lambda: oem_b200.oem_fit_logistic_dense(*a)
    fn()
    ms, outs = timed(fn, steps)
    st = outs[-1]["stats"]
    passes = max(1, st["data_passes"])
    ms_pass = (st["ms_irls_xb"] + st["ms_irls_xtr"]) / passes
    rows_local = r1 - r0
    gb_pass = 8.0 * rows_local * cfg["p"] / 1e9
    phases = {k: round(st[k], 3) for k in ("ms_colstats", "ms_relayout", "ms_gram", "ms_irls_xb", "ms_irls_xtr", "ms_allreduce",
                                           "ms_path", "ms_total")}
    other = st["ms_total"] - sum(v for k, v in phases.items() if k != "ms_total")
    phases["ms_launch_and_sync_gaps"] = round(other, 3)
    limiting = max((k for k in phases if k != "ms_total"), key=lambda k: phases[k])
    beta_sum = float(np.sum(np.abs(outs[-1]["beta"][0])))
    out["logistic_configs3"] = {
        "workload": f"configs[3] logistic lasso n={cfg['n']:.3g} x p={cfg['p']} FP64 ({cfg['n'] * cfg['p'] * 8 / 1e9:.0f} GB total), "
                    f"100 lambdas, standardize, intercept, irls.tol 1e-3, {world} row shard(s) of {rows_local}",
        "fit_s": ms / 1e3, "phases_ms_rank0": phases, "limiting_phase": limiting,
        "irls_iterations": int(np.sum(outs[-1]["niter"][0])), "data_passes": int(passes), "oem_iterations": int(st["total_oem_iters"]),
        "ms_per_data_pass": ms_pass, "data_pass_algorithmic_gb": gb_pass, "data_pass_gbs": gb_pass / (ms_pass / 1e3),
        "data_pass_frac_of_hbm": gb_pass / (ms_pass / 1e3) / hbm,
        "data_pass_kernel": "logit_slab_kernel: X read from HBM once per IRLS pass (sigma(X b) and X'r from the same shared-memory slab)"
                            if st["ms_relayout"] > 0 else "xb_kernel + colstats_kernel (two HBM sweeps)",
        "allreduce_calls": int(st["allreduce_calls"]), "allreduce_avg_us": (st["ms_allreduce"] * 1e3 / st["allreduce_calls"]) if st["allreduce_calls"] else None,
        "host_syncs": int(st["host_syncs"]), "kernel_launches": int(st["kernel_launches"]),
        "sum_abs_beta_rank0": beta_sum, "sum_abs_beta_max_minus_min_over_ranks": _max_over_ranks(torch, beta_sum, device, world) +
        _max_over_ranks(torch, -beta_sum, device, world)}
    del X, y, a
    torch.cuda.empty_cache()
    oem_b200.api.load().oemb200_release_cache()

    # ---- configs[2]: xval.oem 10-fold, lasso + grp.lasso + mcp, n = 1e7 x 500 ----
    cfg = XVAL
    r0, r1 = shard_rows(cfg["n"], rank, world)
    X, y = gen_blocked_rows(torch, cfg, r0, r1, device, binomial=False)
    F = cfg["folds"]
    foldid = (1 + np.random.default_rng(cfg["seed"]).permutation(cfg["n"]) % F).astype(np.int32)[r0:r1]
    groups = np.concatenate([[0], np.repeat(np.arange(1, 51), 10)])
    a = [X, y, "gaussian", ["lasso", "grp.lasso", "mcp"], [], groups, np.unique(groups), [], [], 100, 1e-4, 1.0, 3.0, 0.5,
         np.ones(cfg["p"]), True, True, F, foldid, False, "mse", opts]
    fn = lambda: oem_b200.oem_xval_dense(*a)
    fn()
    ms, outs = timed(fn, steps)
    st = outs[-1]["stats"]
    rows_local = r1 - r0
    phases = {k: round(st[k], 3) for k in ("ms_h2d", "ms_colstats", "ms_gram", "ms_gram_reduce", "ms_allreduce", "ms_assemble",
                                           "ms_path", "ms_cvscore", "ms_total")}
    other = st["ms_total"] - sum(v for k, v in phases.items() if k != "ms_total")
    phases["ms_fold_gather_and_gaps"] = round(other, 3)
    limiting = max((k for k in phases if k != "ms_total"), key=lambda k: phases[k])
    cvm_min = float(np.min(outs[-1]["cvm"][0]))
    out["xval_configs2"] = {
        "workload": f"configs[2] xval.oem {F}-fold lasso+grp.lasso+mcp n={cfg['n']:.3g} x p={cfg['p']} FP64 "
                    f"({cfg['n'] * cfg['p'] * 8 / 1e9:.0f} GB total), 100 lambdas, {world} row shard(s) of {rows_local}",
        "fit_s": ms / 1e3, "phases_ms_rank0": phases, "limiting_phase": limiting,
        "gram_tflops": st["gram_flops"] / (st["ms_gram"] / 1e3) / 1e12 if st["ms_gram"] else None,
        "cvscore_tflops": 2.0 * rows_local * cfg["p"] * 300 / (st["ms_cvscore"] / 1e3) / 1e12 if st["ms_cvscore"] else None,
        "allreduce_calls": int(st["allreduce_calls"]), "oem_iterations": int(st["total_oem_iters"]),
        "cvm_min_lasso_rank0": cvm_min,
        "cvm_min_max_minus_min_over_ranks": _max_over_ranks(torch, cvm_min, device, world) + _max_over_ranks(torch, -cvm_min, device, world)}
    del X, y, a
    torch.cuda.empty_cache()
    oem_b200.api.load().oemb200_release_cache()

    # ---- parity: small sharded fits against the same fits on rank 0 alone (outside any timed region) ----
    out["parity"] = parity_vs_single(torch, api, oem_b200, comm, world, rank, device)
    return out


def parity_vs_single(torch, api, oem_b200, comm, world, rank, device):
    """Every rank builds the same small seeded problems on the host, fits its row shard with the communicator, and rank 0
    also fits the whole problem alone (no communicator).  Returns max |beta_sharded - beta_single| over all entries (the
    single-process results themselves are held to the CPU oracle by tests/ -m gpu; at N > 1 this shows the sharded
    sums + all-reduces reproduce them)."""
    from oem_b200.dist import shard_rows
    rng = np.random.default_rng(7)
    res = {"what": "max |beta(sharded over N ranks) - beta(rank 0 alone)| on small seeded problems through the same C-ABI entries",
           "entries": {}}
    o = dict(OPTS)

    def shard(X, y):
        r0, r1 = shard_rows(X.shape[0], rank, world)
        return np.asfortranarray(X[r0:r1]), y[r0:r1], r0, r1

    def diff(got, ref):
        return max(float(np.max(np.abs(g - r))) for g, r in zip(got["beta"], ref["beta"]))

    # big.oem
    n, p = 36_000, 96
    X = np.asfortranarray(rng.normal(0.2, 1.0, size=(n, p))); b = np.zeros(p); b[:10] = rng.uniform(-.5, .5, 10)
    y = X @ b + rng.normal(size=n)
    common = ["gaussian", ["lasso", "scad", "mcp"], [], [], [], [], [], 25, 1e-3, 1.0, [3.0, 3.7, 3.0], 0.5, np.ones(p), True, True, False]
    Xs, ys, _, _ = shard(X, y)
    got = oem_b200.oem_fit_big(Xs, ys, *common, dict(o), comm=comm)
    if rank == 0:
        res["entries"]["oem_fit_big"] = diff(got, oem_b200.oem_fit_big(X, y, *common, dict(o)))
    # oem (centred + scaled)
    got = oem_b200.oem_fit_dense(Xs, ys, *common, dict(o), comm=comm)
    if rank == 0:
        res["entries"]["oem_fit_dense"] = diff(got, oem_b200.oem_fit_dense(X, y, *common, dict(o)))
    # logistic, slab route
    n, p = 24_000, 160
    X = np.asfortranarray(rng.normal(size=(n, p))); b = np.zeros(p); b[:5] = [.3, .3, -.3, -.3, .5]
    y = (rng.uniform(size=n) < 1 / (1 + np.exp(-(X @ b)))).astype(np.float64)
    common = ["binomial", ["lasso"], [], [], [], [], [], 12, 1e-2, 1.0, 3.0, 0.5, np.ones(p), True, True, False]
    Xs, ys, _, _ = shard(X, y)
    got = oem_b200.oem_fit_logistic_dense(Xs, ys, *common, dict(o), comm=comm)
    if rank == 0:
        res["entries"]["oem_fit_logistic_dense"] = diff(got, oem_b200.oem_fit_logistic_dense(X, y, *common, dict(o)))
    # xval
    n, p, F = 30_000, 40, 5
    X = np.asfortranarray(rng.normal(size=(n, p))); b = np.zeros(p); b[:5] = [.5, .5, -.5, -.5, 1.0]
    y = X @ b + 2.0 * rng.normal(size=n)
    foldid = (1 + rng.permutation(n) % F).astype(np.int32)
    Xs, ys, r0, r1 = shard(X, y)
    mk = lambda XX, yy, ff: [XX, yy, "gaussian", ["lasso", "mcp"], [], [], [], [], [], 15, 1e-3, 1.0, 3.0, 0.5, np.ones(p), True,
                             True, F, ff, False, "mse", dict(o)]
    got = oem_b200.oem_xval_dense(*mk(Xs, ys, foldid[r0:r1]), comm=comm)
    if rank == 0:
        ref = oem_b200.oem_xval_dense(*mk(X, y, foldid))
        res["entries"]["oem_xval_dense"] = diff(got, ref)
        res["entries"]["oem_xval_dense_cvm_rel"] = max(float(np.max(np.abs(g - r) / np.abs(r))) for g, r in zip(got["cvm"], ref["cvm"]))
    if world > 1:
        torch.distributed.barrier()
    if rank == 0:
        res["max_dbeta_vs_n1"] = max(v for k, v in res["entries"].items() if not k.endswith("_rel"))
        res["n_ranks"] = world
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=ROWS_PER_GPU, help="rows per GPU (default: the 100 GB shard of configs[4])")
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    ap.add_argument("--gigs", type=float, default=2.0, help="host->device streaming chunk (GB) for the e2e leg")
    ap.add_argument("--comm", default="lib", choices=["lib", "callback"], help="all-reduce transport at N > 1")
    ap.add_argument("--secondary-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--allow-partial-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed fit returned (beta, lambda, niter, loss per "
                         "penalty, and d) as float64 DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
