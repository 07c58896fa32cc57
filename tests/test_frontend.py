"""R front-end mirrors (oem_b200.frontend) and the bigmemory ingest (oem_b200.bigmatrix): host logic on CPU,
end-to-end parity with the oracle on the GPU."""
import numpy as np
import pytest

from cases import gaussian_problem, binomial_problem


def test_getmin_known_answer():
    from oem_b200.frontend import getmin
    lam = [np.array([1.0, 0.5, 0.25, 0.125]), np.array([1.0, 0.5, 0.25, 0.125])]
    cvm = [np.array([4.0, 2.0, 1.0, 1.5]), np.array([3.0, 0.9, 0.95, 2.0])]
    cvsd = [np.array([0.5, 0.5, 0.6, 0.5]), np.array([0.1, 0.2, 0.1, 0.1])]
    r = getmin(lam, cvm, cvsd)
    # model 2 has the smaller minimum (0.9 at lambda 0.5); 1se rule: largest lambda with cvm < 0.9 + 0.2
    assert r["model_min"] == 2 and r["lambda_min"] == 0.5 and r["lambda_1se"] == 0.5
    assert r["lambda_min_models"].tolist() == [0.25, 0.5]
    assert r["lambda_1se_models"].tolist() == [0.25, 0.5]       # model 1: cvm < 1.0 + 0.6 -> {1.0, 1.5} -> lambda 0.25


def test_group_bookkeeping_and_validation():
    from oem_b200 import frontend as fe
    g, ug, gw = fe._groups(["grp.lasso"], [2, 2, 1, 1, 3], None, 5, explicit_intercept=False)
    assert g.tolist() == [2, 2, 1, 1, 3] and ug.tolist() == [1, 2, 3] and gw.size == 0
    g, ug, gw = fe._groups(["grp.lasso"], [2, 2, 1, 1, 3], None, 5, explicit_intercept=True)     # R/oem.R:318-345
    assert g.tolist() == [0, 2, 2, 1, 1, 3] and ug.tolist() == [0, 1, 2, 3]
    g, ug, gw = fe._groups(["grp.lasso"], [0, 2, 1, 1, 3], [9.0, 1.0, 2.0, 3.0], 5, explicit_intercept=True)
    assert ug.tolist() == [0, 1, 2, 3] and gw.tolist() == [0.0, 1.0, 2.0, 3.0]                  # group 0 weight forced to 0
    assert fe._groups(["lasso"], [], None, 5, True)[0].size == 0
    with pytest.raises(ValueError, match="groups must have same length"):
        fe._groups(["grp.lasso"], [1, 2], None, 5, False)
    lam = fe._lambda_list([0.1, 1.0, 0.5], 2)
    assert [l.tolist() for l in lam] == [[1.0, 0.5, 0.1]] * 2                                   # sorted decreasing
    with pytest.raises(ValueError, match="same length as the number of penalties"):
        fe._lambda_list([np.array([1.0])], 2)
    X, y = gaussian_problem(1, 30, 4)
    with pytest.raises(ValueError, match="lengths do not match"):
        fe.oem(X, y[:-1], penalty="lasso")
    with pytest.raises(ValueError, match="lambda.min.ratio"):
        fe.oem(X, y, penalty="lasso", lambda_min_ratio=1.5)
    with pytest.raises(ValueError, match="weights not implemented"):
        fe.oem(X, y, penalty="lasso", weights=np.ones(30))
    with pytest.raises(ValueError, match="nfolds must be bigger than 3"):
        fe.xval_oem(X, y, nfolds=2, penalty="lasso")


def test_bigmatrix_roundtrip(tmp_path):
    from oem_b200 import bigmatrix
    X, _ = gaussian_problem(3, 101, 7)
    bk, desc = str(tmp_path / "bigmat.bk"), str(tmp_path / "bigmatk.desc")
    bigmatrix.write(X, bk, desc)
    d = bigmatrix.read_descriptor(desc)
    assert (d["nrow"], d["ncol"], d["type"], d["filename"]) == (101, 7, "double", "bigmat.bk")
    mm = bigmatrix.attach(desc)
    assert mm.shape == (101, 7) and mm.flags["F_CONTIGUOUS"] and np.array_equal(np.asarray(mm), X)
    assert np.array_equal(np.fromfile(bk, dtype=np.float64), X.ravel(order="F"))     # raw column-major payload


@pytest.mark.gpu
def test_frontends_match_oracle(lib, oracle):
    from oem_b200 import frontend as fe
    X, y = gaussian_problem(41, 3000, 40)
    groups = np.repeat(np.arange(1, 9), 5)
    r = fe.oem(X, y, penalty=["lasso", "grp.lasso"], groups=groups, nlambda=25, tol=1e-9)
    ref = oracle.oem_fit_dense(X, y, "gaussian", ["lasso", "grp.lasso"], [], groups, np.unique(groups), [], [[], []], 25,
                               1e-4, 1.0, 3.0, 0.5, np.ones(40), True, True, False, dict(maxit=500, tol=1e-9))
    for i, pen in enumerate(["lasso", "grp.lasso"]):
        assert np.max(np.abs(r["beta"][pen] - ref["beta"][i])) <= 1e-8
        # lambda_max sits exactly on the threshold of the largest |X'y| entry (strict inequality, src/oem_dense.h:87-90):
        # whether that coefficient is 0 or ~1e-17 depends on the last bit of lmax * scaleY / scaleY, so skip column 0
        assert np.array_equal(r["nzero"][i][1:], np.count_nonzero(ref["beta"][i][1:], axis=0)[1:])
        assert np.array_equal(r["nzero"][i], np.count_nonzero(r["beta"][pen][1:], axis=0))
    assert r["nobs"] == 3000 and r["nvars"] == 40 and r["rownames"][0] == "(Intercept)"
    # binomial: explicit intercept -> group 0 prepended by the front-end like R/oem.R:318-345
    Xb, yb = binomial_problem(42, 3000, 20)
    gb = np.repeat(np.arange(1, 5), 5)
    rb = fe.oem(Xb, yb, family="binomial", penalty="grp.lasso", groups=gb, nlambda=8, lambda_min_ratio=1e-2)
    refb = oracle.oem_fit_logistic_dense(Xb, yb, "binomial", ["grp.lasso"], [], np.concatenate([[0], gb]), np.arange(0, 5), [],
                                         [[]], 8, 1e-2, 1.0, 3.0, 0.5, np.ones(20), True, True, False, dict(maxit=500, tol=1e-7))
    assert np.max(np.abs(rb["beta"]["grp.lasso"] - refb["beta"][0])) <= 1e-8
    # xval.oem: cvm / lambda.min / best model
    rng = np.random.default_rng(7)
    foldid = 1 + rng.permutation(3000) % 5
    rx = fe.xval_oem(X, y, foldid=foldid, penalty=["lasso", "mcp"], nlambda=20)
    refx = oracle.oem_xval_dense(X, y, "gaussian", ["lasso", "mcp"], [], [], [], [], [[], []], 20, 1e-4, 1.0, 3.0, 0.5,
                                 np.ones(40), True, True, 5, foldid, False, "mse", dict(maxit=500, tol=1e-7))
    gm = fe.getmin(refx["lambda_"], refx["cvm"], refx["cvsd"])
    assert rx["model_min"] == gm["model_min"] and abs(rx["lambda_min"] / gm["lambda_min"] - 1) < 1e-12
    assert rx["best_model"] in ("lasso", "mcp") and np.allclose(rx["cvup"][0], refx["cvm"][0] + refx["cvsd"][0], rtol=1e-8)


@pytest.mark.gpu
def test_big_oem_from_file_backed_matrix(lib, oracle, tmp_path):
    from oem_b200 import bigmatrix, frontend as fe
    X, y = gaussian_problem(43, 20000, 30)
    bk, desc = str(tmp_path / "bigmat.bk"), str(tmp_path / "bigmatk.desc")
    bigmatrix.write(X, bk, desc)
    bigmat = bigmatrix.attach(desc)                                   # mmap'd, like attach.big.matrix()
    r = fe.big_oem(bigmat, y, penalty=["lasso", "scad"], gamma=[3.0, 3.7], nlambda=20, gigs=0.001)   # several row chunks
    ref = oracle.oem_fit_big(X, y, "gaussian", ["lasso", "scad"], [], [], [], [], [[], []], 20, 1e-4, 1.0, [3.0, 3.7], 0.5,
                             np.ones(30), True, True, False, dict(maxit=500, tol=1e-7))
    assert np.max(np.abs(r["beta"]["lasso"] - ref["beta"][0])) <= 1e-8
    assert np.max(np.abs(r["beta"]["scad"] - ref["beta"][1])) <= 1e-8
    assert r["stats"]["h2d_bytes"] >= X.nbytes


@pytest.mark.gpu
def test_big_oem_file_backed_ingest_rate(lib, tmp_path):
    """A 2 GB file-backed big.matrix (page cache) streamed through the pinned bounce ring + reader threads (csrc/ingest.cu)
    must give the fit of the same data resident on the device, at a rate well above the driver's pageable-copy path
    (~11 GB/s on the B200 boxes)."""
    import torch
    from oem_b200 import bigmatrix, frontend as fe
    n, p = 500_000, 500
    bk, desc = str(tmp_path / "big.bk"), str(tmp_path / "big.desc")
    rng = np.random.default_rng(99)
    mm = np.memmap(bk, dtype=np.float64, mode="w+", shape=(n, p), order="F")
    for j in range(p):
        mm[:, j] = rng.standard_normal(n)
    b = np.zeros(p); b[:8] = rng.uniform(-0.5, 0.5, 8)
    y = np.asarray(mm @ b) + rng.standard_normal(n)
    mm.flush(); del mm
    bigmatrix.write_descriptor(desc, bk, n, p)
    bigmat = bigmatrix.attach(desc)
    assert isinstance(bigmat, np.memmap)
    r = fe.big_oem(bigmat, y, penalty=["lasso"], nlambda=20, gigs=0.25)
    r = fe.big_oem(bigmat, y, penalty=["lasso"], nlambda=20, gigs=0.25)          # second call: ring and pools warm
    Xd = torch.from_numpy(np.array(np.asarray(bigmat).T, order="C")).cuda().t()
    rd = lib.oem_fit_big(Xd, torch.from_numpy(y).cuda(), "gaussian", ["lasso"], [], [], [], [], [], 20, 1e-4, 1.0, 3.0, 0.5,
                         np.ones(p), True, True, False, dict(maxit=500, tol=1e-7))
    assert np.max(np.abs(r["beta"]["lasso"] - rd["beta"][0])) <= 1e-10
    st = r["stats"]
    rate = st["h2d_bytes"] / (st["ms_h2d"] / 1e3) / 1e9
    print(f"file-backed ingest: {st['h2d_bytes'] / 1e9:.2f} GB in {st['ms_h2d']:.1f} ms = {rate:.1f} GB/s "
          f"(host fill time {st['ms_ingest_wait']:.1f} ms)")
    assert st["h2d_bytes"] >= n * p * 8 and st["ms_ingest_wait"] > 0
    assert rate > 14.0


def test_lambda_interp_and_host_predict_types():
    """R/utils.R:64-87 and the host-only branches of predict.oem (R/methods.R:84-101)."""
    from oem_b200 import frontend as fe
    lam = np.array([1.0, 0.5, 0.25, 0.125])
    left, right, frac = fe.lambda_interp(lam, [0.5, 0.375, 2.0, 0.01])
    assert list(left) == [1, 1, 0, 3] and list(right) == [1, 2, 0, 3]
    assert np.allclose(frac, [1.0, 0.5, 1.0, 1.0])
    B = np.array([[1.0, 2.0, 3.0, 4.0], [0.0, 0.0, 1.0, 2.0], [0.0, -1.0, -1.0, 0.0]])
    fit = dict(beta={"lasso": B}, family="gaussian", nobs=10, loss=[np.array([4.0, 3.0, 2.0, 1.0])])
    fit["lambda"] = [lam]
    co = fe.predict(fit, s=[0.375], type="coefficients")
    assert np.allclose(co[:, 0], 0.5 * B[:, 1] + 0.5 * B[:, 2])
    nz = fe.predict(fit, type="nonzero")
    assert nz[0] is None and list(nz[1]) == [3] and list(nz[2]) == [2, 3] and list(nz[3]) == [2]
    ll = fe.logLik(fit)
    assert np.allclose(ll, -0.5 * 10 * (np.log(2 * np.pi) - np.log(10.0) + np.log(fit["loss"][0])) - 5.0)
    with pytest.raises(ValueError):
        fe.predict(fit, type="link")                      # newx missing
    with pytest.raises(ValueError):
        fe.predict(fit, which_model="mcp", type="coefficients")
    with pytest.raises(ValueError):
        fe.predict(fit, which_model=2, type="coefficients")
    fit["loss"] = [np.full(4, 1e99)]
    with pytest.raises(ValueError):
        fe.logLik(fit)


@pytest.mark.gpu
@pytest.mark.parametrize("n,p,L", [(1000, 30, 25), (4097, 57, 100), (333, 7, 1), (2500, 20, 330)])
def test_predict_on_device(lib, n, p, L):
    """oemb200_predict: newx %*% beta + intercept as one DMMA GEMM (ragged rows / k / more than 320 columns)"""
    rng = np.random.default_rng(n + p)
    X = np.asfortranarray(rng.normal(size=(n, p)))
    B = np.asfortranarray(rng.normal(size=(p + 1, L)) * (rng.uniform(size=(p + 1, L)) < 0.4))
    ref = X @ B[1:] + B[0:1]
    got = lib.predict_matrix(X, B)
    assert got.shape == (n, L) and np.max(np.abs(got - ref)) <= 1e-12 * max(1.0, np.abs(ref).max())
    got = lib.predict_matrix(X, B, response=True)
    assert np.allclose(got, 1.0 / (1.0 + np.exp(-ref)), rtol=1e-13, atol=1e-15)
    got = lib.predict_matrix(X, B[1:])                    # p-row coefficient matrix (oem.xtx): no intercept row
    assert np.max(np.abs(got - X @ B[1:])) <= 1e-12 * max(1.0, np.abs(ref).max())
    import torch
    Xd = torch.from_numpy(np.ascontiguousarray(X.T)).cuda().t()          # column-major device matrix
    out = torch.empty((L, n), dtype=torch.float64, device="cuda").t()
    lib.predict_matrix(Xd, B, out=out)
    assert np.max(np.abs(out.cpu().numpy() - ref)) <= 1e-12 * max(1.0, np.abs(ref).max())
    with pytest.raises(Exception):
        lib.predict_matrix(X, B[:-2])


@pytest.mark.gpu
def test_predict_and_loglik_frontends(lib, oracle):
    from oem_b200 import frontend as fe
    X, y = gaussian_problem(61, 3000, 25)
    fit = fe.oem(X, y, penalty=["lasso", "mcp"], nlambda=20, compute_loss=True)
    Xn, _ = gaussian_problem(62, 500, 25)
    for m, pen in enumerate(["lasso", "mcp"]):
        B = fit["beta"][pen]
        pr = fe.predict(fit, Xn, which_model=pen)
        assert np.max(np.abs(pr - (Xn @ B[1:] + B[0:1]))) <= 1e-12 * np.abs(pr).max()
        lam = fit["lambda"][m]
        s = [0.5 * (lam[3] + lam[4]), lam[7]]
        pr = fe.predict(fit, Xn, s=s, which_model=m + 1, type="response")
        co = fe.predict(fit, s=s, which_model=m + 1, type="coefficients")
        assert np.allclose(co[:, 0], 0.5 * (B[:, 3] + B[:, 4]), atol=1e-12) and np.allclose(co[:, 1], B[:, 7])
        assert np.max(np.abs(pr - (Xn @ co[1:] + co[0:1]))) <= 1e-12 * np.abs(pr).max()
        n = float(X.shape[0])
        assert np.allclose(fe.logLik(fit, pen), -0.5 * n * (np.log(2 * np.pi) - np.log(n) + np.log(fit["loss"][m])) - 0.5 * n)
    # without standardisation the loss member is the raw residual sum of squares (src/oem_dense.h:759-770)
    raw = fe.oem(X, y, penalty=["lasso"], nlambda=10, compute_loss=True, standardize=False, intercept=False)
    rss = ((y[:, None] - fe.predict(raw, X)) ** 2).sum(axis=0)
    assert np.allclose(raw["loss"][0], rss, rtol=1e-10)
    Xb, yb = binomial_problem(63, 2000, 12)
    fb = fe.oem(Xb, yb, family="binomial", penalty=["lasso"], nlambda=8, lambda_min_ratio=1e-2)
    Bb = fb["beta"]["lasso"]
    eta = Xb @ Bb[1:] + Bb[0:1]
    assert np.allclose(fe.predict(fb, Xb, type="response"), 1 / (1 + np.exp(-eta)), rtol=1e-12)
    assert np.array_equal(fe.predict(fb, Xb, type="class"), np.where(eta > 0, 2, 1))


def test_cv_helpers_known_answers():
    """Host helpers of the cv.oem mirror: row selection for every container kind, glmnet's fold-grouped means."""
    import scipy.sparse as sps
    from oem_b200 import frontend as fe
    X = np.asfortranarray(np.arange(12, dtype=np.float64).reshape(4, 3))
    keep = np.array([True, False, True, True])
    d = fe._take_rows(X, keep)
    assert d.flags["F_CONTIGUOUS"] and np.array_equal(d, X[[0, 2, 3]])
    s = fe._take_rows(sps.csc_matrix(X), keep)
    assert sps.issparse(s) and s.format == "csc" and np.array_equal(s.toarray(), X[[0, 2, 3]])
    assert np.array_equal(fe._take_rows(np.array([1.0, 2.0, 3.0, 4.0]), keep), [1.0, 3.0, 4.0])
    # cvcompute (R/utils.R:126-144): per-fold weighted means, NA-aware; N counts the folds that reach each lambda
    mat = np.array([[1.0, 2.0], [3.0, np.nan], [5.0, 6.0], [7.0, np.inf]])
    foldid = np.array([1, 1, 2, 2])
    out, wsum, N = fe._cvcompute(mat, np.array([1.0, 3.0, 1.0, 1.0]), foldid, np.array([2, 1]))
    assert np.allclose(out, [[(1 + 9) / 4.0, 2.0], [6.0, 6.0]]) and wsum.tolist() == [4.0, 2.0] and N.tolist() == [2.0, 1.0]
    # lambda.interp (R/utils.R:64-87): exact at grid points, linear in between, clamped outside
    lam = np.array([1.0, 0.5, 0.25])
    l, r, f = fe.lambda_interp(lam, [0.5, 0.75, 2.0, 0.1])
    assert l.tolist() == [1, 0, 0, 2] and r.tolist() == [1, 1, 0, 2]
    assert np.allclose(f, [1.0, 0.5, 1.0, 1.0])


def test_bench_reference_arm_smoke(tmp_path):
    """bench.py --impl reference (the CPU arm the driver runs next to the GPU arm) on a toy size: one JSON line with the
    contract's keys, a MEASURED full-size fit (the toy 'full size' fits in RAM), and the BLAS thread count it actually used."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, OMP_NUM_THREADS="1")          # what torchrun exports at nproc > 1: the arm must override it
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2",
                          "--warmup", "1", "--rows", "40000", "--cpu-sample-rows", "8000"], capture_output=True, text=True,
                         timeout=600, env=env, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    cb = line["cpu_baseline"]
    assert line["impl"] == "reference" and line["steps"] == 2 and cb["kind"] == "port"
    assert cb["measured"] is True and cb["measured_full_size_steps"] == 2 and len(cb["step_seconds"]) == 2
    assert abs(line["value"] - sum(cb["step_seconds"]) / 2) < 0.02 and line["e2e"]["h2d_bytes_per_step"] == 0
    assert cb["cores"] == len(os.sched_getaffinity(0)) or cb["cores"] >= 1          # the pool size that was set, not the env's 1
    if len(os.sched_getaffinity(0)) > 1:
        assert cb["cores"] > 1


@pytest.mark.gpu
def test_bench_dump_outputs_match_a_fit_of_the_seeded_inputs(lib, tmp_path):
    """bench.py --dump-outputs on a small shard: the timed steps run as many times as --steps says, and the dumped arrays
    (float64, one file per returned array and penalty) equal a fit of the same seeded inputs made here."""
    import json
    import os
    import subprocess
    import sys
    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rows, dump = 20_000, tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3",
                          "--rows", str(rows), "--no-e2e", "--no-cpu", "--no-secondary", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and len(line["config"]["host_wall_ms_per_step"]) == 2
    sys.path.insert(0, root)
    import bench
    X, y = bench.gen_shard(torch, rows, 105_000, torch.device("cuda", 0))
    ref = lib.oem_fit_big(*bench.fit_args(X, y))
    names = {"d.npy"}
    for k, pen in enumerate(bench.PENALTIES):
        for key in ("beta", "lambda_", "niter", "loss"):
            name = f"{key.rstrip('_')}_{pen}.npy"
            names.add(name)
            got = np.load(dump / name)
            assert got.dtype == np.float64 and got.shape == ref[key][k].shape, name
            assert np.allclose(got, ref[key][k], rtol=1e-10, atol=1e-12), name
    assert set(os.listdir(dump)) == names
    assert np.load(dump / "d.npy")[0] == pytest.approx(ref["d"], rel=1e-12)
