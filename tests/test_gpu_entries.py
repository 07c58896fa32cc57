"""-m gpu parity tests: the CUDA path (through the C ABI, via oem_b200.api) against the CPU oracle
on the same seeded inputs.  Bar: max|delta beta| <= 1e-8 (FP64), lambda sequences <= 4 ulp, d to 1e-9."""
import numpy as np
import pytest

from cases import args_xy, assert_same_fit, binomial_problem, gaussian_problem

pytestmark = pytest.mark.gpu

ALL_COORD = ["lasso", "ols", "elastic.net", "scad", "scad.net", "mcp", "mcp.net"]
ALL_GROUP = ["grp.lasso", "grp.lasso.net", "grp.mcp", "grp.scad", "grp.mcp.net", "grp.scad.net", "sparse.grp.lasso"]


@pytest.mark.parametrize("standardize,intercept", [(False, False), (True, False), (False, True), (True, True)])
def test_dense_flags(lib, oracle, standardize, intercept):
    X, y = gaussian_problem(11, 3000, 60, sd_x=2.0, mean_x=0.7)
    a = args_xy(X, y, "gaussian", ["lasso", "mcp"], standardize=standardize, intercept=intercept, nlambda=30,
                opts=dict(tol=1e-10))
    assert_same_fit(lib.oem_fit_dense(*a), oracle.oem_fit_dense(*a))


def test_dense_readme_lasso_config1_small(lib, oracle):
    # BASELINE config 1 shape (README.md:45-65) at n = 2e4: elastic.net alpha=1, intercept, no standardize
    X, y = gaussian_problem(101, 20000, 100, sd_x=3.0)
    a = args_xy(X, y, "gaussian", ["elastic.net"], standardize=False, intercept=True, opts=dict(tol=1e-10))
    assert_same_fit(lib.oem_fit_dense(*a), oracle.oem_fit_dense(*a))


def test_dense_nonconvex_config2(lib, oracle):
    # BASELINE config 2 at full size: MCP gamma=2 + SCAD gamma=4, n=5000 p=200, 200 lambdas, batched
    X, y = gaussian_problem(102, 5000, 200, sd_x=3.0)
    a = args_xy(X, y, "gaussian", ["mcp", "scad"], gamma=[2.0, 4.0], nlambda=200, opts=dict(tol=1e-10))
    got = lib.oem_fit_dense(*a)
    ref = oracle.oem_fit_dense(*a)
    assert_same_fit(got, ref)
    # the per-penalty gamma extension reduces to two scalar-gamma calls of the reference interface
    a1 = args_xy(X, y, "gaussian", ["scad"], gamma=4.0, nlambda=200, opts=dict(tol=1e-10))
    ref1 = oracle.oem_fit_dense(*a1)
    assert np.max(np.abs(got["beta"][1] - ref1["beta"][0])) <= 1e-8


def test_dense_all_penalties(lib, oracle):
    X, y = gaussian_problem(7, 2000, 40)
    groups = np.repeat(np.arange(1, 9), 5)
    groups[:3] = 0
    a = args_xy(X, y, "gaussian", ALL_COORD + ALL_GROUP, groups=groups, unique_groups=np.unique(groups), alpha=0.6,
                gamma=3.0, tau=0.4, nlambda=25, opts=dict(tol=1e-10))
    assert_same_fit(lib.oem_fit_dense(*a), oracle.oem_fit_dense(*a))


def test_dense_odd_rows_user_lambda_accelerate_loss(lib, oracle):
    X, y = gaussian_problem(5, 1501, 33)       # odd n: the non-TMA loader path
    lam = [np.geomspace(1.0, 1e-3, 12), np.geomspace(0.5, 1e-3, 12)]
    pf = np.ones(33); pf[:2] = 0.0; pf[5] = 2.5
    a = args_xy(X, y, "gaussian", ["lasso", "scad"], lambda_=lam, penalty_factor=pf, compute_loss=True,
                opts=dict(tol=1e-9, accelerate=True))
    got, ref = lib.oem_fit_dense(*a), oracle.oem_fit_dense(*a)
    assert_same_fit(got, ref)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg, lr, rtol=1e-10)


def test_xtx_identity_and_scale_factor(lib, oracle):
    X, y = gaussian_problem(3, 4000, 50)
    n = X.shape[0]
    xtx, xty = X.T @ X / n, X.T @ y / n
    pens = ["lasso", "mcp", "grp.lasso"]
    groups = np.repeat(np.arange(1, 11), 5)
    common = ["gaussian", pens, groups, np.unique(groups), [], [], 40, 1e-3, 1.0, 3.0, 0.5]
    o = dict(maxit=500, tol=1e-10)
    got = lib.oem_xtx(xtx, xty, *common, [], np.ones(50), o)
    ref = oracle.oem_xtx(xtx, xty, *common, [], np.ones(50), o)
    assert_same_fit(got, ref, lam_ulps=4)
    # the reference's own printed identity (R/oem_xtx.R:69-103): oem(standardize=F, intercept=F) == oem.xtx
    a = args_xy(X, y, "gaussian", pens, groups=groups, unique_groups=np.unique(groups), standardize=False,
                intercept=False, nlambda=40, lmin_ratio=1e-3, opts=dict(tol=1e-10))
    dense = lib.oem_fit_dense(*a)
    for pp in range(len(pens)):
        assert np.max(np.abs(dense["beta"][pp][1:, :] - got["beta"][pp])) <= 1e-10
    sf = np.sqrt(np.diag(xtx))
    got = lib.oem_xtx(xtx, xty, *common, sf, np.ones(50), o)
    ref = oracle.oem_xtx(xtx, xty, *common, sf, np.ones(50), o)
    assert_same_fit(got, ref)


@pytest.mark.parametrize("standardize,intercept", [(True, True), (False, True), (True, False)])
def test_big_small(lib, oracle, standardize, intercept):
    X, y = gaussian_problem(105, 6000, 130, mean_x=0.3)
    groups = np.concatenate([[0], np.repeat(np.arange(1, 14), 10)]) if intercept else np.repeat(np.arange(1, 14), 10)
    a = args_xy(X, y, "gaussian", ["lasso", "scad", "mcp", "grp.lasso"], gamma=[3.0, 3.7, 3.0, 3.0], groups=groups,
                unique_groups=np.unique(groups), standardize=standardize, intercept=intercept, nlambda=50)
    assert_same_fit(lib.oem_fit_big(*a), oracle.oem_fit_big(*a))


def test_big_streams_host_chunks(lib, oracle):
    # host X larger than one streaming chunk (gigs) -> several accumulate passes, same answer
    X, y = gaussian_problem(106, 20000, 64)
    a = args_xy(X, y, "gaussian", ["lasso"], nlambda=20, opts=dict(gigs=0.002))
    assert_same_fit(lib.oem_fit_big(*a), oracle.oem_fit_big(*a))


def test_big_device_resident(lib, oracle):
    import torch
    X, y = gaussian_problem(107, 9000, 257)
    Xd = torch.from_numpy(np.ascontiguousarray(X.T)).cuda().t()       # column-major on the device
    yd = torch.from_numpy(y).cuda()
    a = args_xy(X, y, "gaussian", ["lasso", "mcp"], nlambda=30)
    ref = oracle.oem_fit_big(*a)
    a[0], a[1] = Xd, yd
    assert_same_fit(lib.oem_fit_big(*a), ref)


@pytest.mark.parametrize("hessian", ["upper.bound", "full"])
def test_logistic(lib, oracle, hessian):
    X, y = binomial_problem(104, 4000, 40)
    groups = np.concatenate([[0], np.repeat(np.arange(1, 9), 5)])
    a = args_xy(X, y, "binomial", ["lasso", "mcp.net", "grp.lasso"], groups=groups, unique_groups=np.unique(groups),
                alpha=0.7, nlambda=15, lmin_ratio=1e-2, compute_loss=True, opts=dict(hessian_type=hessian))
    got, ref = lib.oem_fit_logistic_dense(*a), oracle.oem_fit_logistic_dense(*a)
    assert_same_fit(got, ref, tol=1e-8)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg, lr, rtol=1e-9)


@pytest.mark.parametrize("n,p,intercept,standardize,route", [
    (6002, 130, True, False, None),        # slab route, 16-row slabs, one column per thread
    (5003, 300, True, True, None),         # 16-row slabs, two columns per thread, ragged last slab
    (4001, 530, False, True, None),        # 8-row slabs, three columns per thread
    (3000, 1030, True, True, None),        # 4-row slabs
    (5003, 300, True, True, "sweeps"),     # same problem through the two-sweep route
    (3001, 17, False, True, None),         # small p, small n: launch-bound, the slab route (2 launches per pass) wins
    (3001, 17, False, True, "sweeps"),     # the same through the two sweeps
    (100003, 9, True, True, None),         # small p, n > 1e5: two sweeps by default
    (3001, 5, True, False, None),          # p < 8: two sweeps
])
def test_logistic_data_pass_routes(lib, oracle, monkeypatch, n, p, intercept, standardize, route):
    # the IRLS data pass either reads a row-slab copy of X once (logit_slab.cu: 128 <= p <= 2048, and 8 <= p < 128 when
    # n <= 1e5) or sweeps the column-major X twice (xb_kernel + colstats_kernel); OEMB200_LOGIT_ROUTE=sweeps forces the
    # latter.  Both must reproduce the oracle's path.
    if route:
        monkeypatch.setenv("OEMB200_LOGIT_ROUTE", route)
    X, y = binomial_problem(300 + p, n, p)
    a = args_xy(X, y, "binomial", ["lasso", "mcp"], nlambda=8, lmin_ratio=5e-2, intercept=intercept, standardize=standardize,
                compute_loss=True)
    got, ref = lib.oem_fit_logistic_dense(*a), oracle.oem_fit_logistic_dense(*a)
    assert_same_fit(got, ref, tol=1e-8)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg, lr, rtol=1e-9)
    st = got["stats"]
    expect_slab = route is None and (128 <= p <= 2048 or (8 <= p < 128 and n <= 100000))
    assert st["data_passes"] > 0 and (st["ms_relayout"] > 0) == expect_slab
    assert st["host_syncs"] <= int(sum(np.sum(v) for v in got["niter"])) + 8 * len(got["niter"][0]) + 16


@pytest.mark.parametrize("n,p", [(10007, 128), (4100, 512), (9001, 1000), (2050, 2048)])
def test_logit_slab_pass_matches_fp64_reference(lib, n, p):
    # the fused single-sweep kernel on its own against torch FP64: prob, W and [sum r, X'r]
    import ctypes
    import torch
    from oem_b200 import api
    g = torch.Generator(device="cuda").manual_seed(n + p)
    Xt = torch.randn((p, n + (n & 1)), generator=g, dtype=torch.float64, device="cuda")
    X = Xt.t()[:n]
    b = torch.randn(p, generator=g, dtype=torch.float64, device="cuda") / p ** 0.5
    y = (torch.rand(n, generator=g, dtype=torch.float64, device="cuda") < 0.4).double()
    prob = torch.empty(n, dtype=torch.float64, device="cuda")
    w = torch.empty_like(prob)
    grad = torch.empty(p + 1, dtype=torch.float64, device="cuda")
    ms, msr = ctypes.c_double(), ctypes.c_double()
    api._check(api.load().oemb200_logit_slab_pass(X.data_ptr(), n, p, X.stride(1), b.data_ptr(), 0.3, y.data_ptr(), prob.data_ptr(),
                                                  w.data_ptr(), grad.data_ptr(), 2, None, ctypes.byref(ms), ctypes.byref(msr)))
    pr = torch.sigmoid(X @ b + 0.3)
    r = y - pr
    assert torch.allclose(prob, pr, rtol=0, atol=1e-14)
    assert torch.allclose(w, pr * (1 - pr), rtol=0, atol=1e-14)
    ref = torch.cat([r.sum().view(1), X.t() @ r])
    assert torch.allclose(grad, ref, rtol=1e-12, atol=1e-10 * n ** 0.5)
    # bit-reproducible run to run
    grad2 = torch.empty_like(grad)
    api._check(api.load().oemb200_logit_slab_pass(X.data_ptr(), n, p, X.stride(1), b.data_ptr(), 0.3, y.data_ptr(), None, None,
                                                  grad2.data_ptr(), 1, None, None, None))
    assert torch.equal(grad, grad2)


def test_logistic_speculative_iterations_change_nothing(lib, monkeypatch):
    # the dense logistic driver enqueues IRLS iteration k + 1 before it has read iteration k's stop-rule verdict; every kernel
    # of the chain is predicated on the device-side "converged" flag, so the speculation must be invisible in the results:
    # same beta to the bit, same IRLS counts, same number of executed data passes as with OEMB200_IRLS_NO_SPECULATION=1
    X, y = binomial_problem(404, 6000, 260)
    a = args_xy(X, y, "binomial", ["lasso", "mcp"], nlambda=12, lmin_ratio=2e-2, compute_loss=True)
    spec = lib.oem_fit_logistic_dense(*a)
    monkeypatch.setenv("OEMB200_IRLS_NO_SPECULATION", "1")
    plain = lib.oem_fit_logistic_dense(*a)
    for k in range(2):
        assert np.array_equal(spec["beta"][k], plain["beta"][k])
        assert np.array_equal(spec["niter"][k], plain["niter"][k])
        assert np.array_equal(spec["loss"][k], plain["loss"][k])
    assert spec["stats"]["data_passes"] == plain["stats"]["data_passes"] > 0
    assert spec["stats"]["total_oem_iters"] == plain["stats"]["total_oem_iters"]
    assert spec["stats"]["kernel_launches"] > plain["stats"]["kernel_launches"]       # the predicated extra iterations were enqueued


@pytest.mark.parametrize("irls_maxit", [1, 2, 3])
def test_logistic_irls_maxit_exhausted(lib, oracle, irls_maxit):
    # the IRLS cap cuts the (speculatively pipelined) loop short: niter reports irls_maxit + 1 where the loop did not converge,
    # and the iterate handed to the next lambda is the one the last EXECUTED iteration produced
    X, y = binomial_problem(405, 5000, 140)
    a = args_xy(X, y, "binomial", ["lasso"], nlambda=8, lmin_ratio=2e-2, opts=dict(irls_maxit=irls_maxit, irls_tol=1e-9))
    got, ref = lib.oem_fit_logistic_dense(*a), oracle.oem_fit_logistic_dense(*a)
    assert_same_fit(got, ref, tol=1e-8)
    assert np.array_equal(got["niter"][0], ref["niter"][0]) and got["niter"][0].max() == irls_maxit + 1


def test_logistic_cuda_path_matches_independent_coordinate_descent(lib):
    # the CUDA path itself (slab route, p = 130) against the independent coordinate-descent binomial lasso of
    # tests/independent_cd.py at tight tolerances: agreement at 1e-7, like oem vs glmnet in the reference's README
    from independent_cd import binomial_lasso_cd
    X, y = binomial_problem(78, 2500, 130)
    a = args_xy(X, y, "binomial", ["lasso"], standardize=False, intercept=True, nlambda=5, lmin_ratio=0.2,
                opts=dict(tol=1e-13, maxit=50000, irls_tol=1e-12, irls_maxit=5000))
    r = lib.oem_fit_logistic_dense(*a)
    B, lam = r["beta"][0], r["lambda_"][0]
    assert r["stats"]["ms_relayout"] > 0
    b0, b = 0.0, np.zeros(130)
    for i in range(1, 5):
        b0, b, _ = binomial_lasso_cd(X, y, lam[i], b0=b0, b=b, tol=1e-12)
        assert abs(B[0, i] - b0) <= 1e-7 and np.max(np.abs(B[1:, i] - b)) <= 1e-7
        assert np.array_equal(B[1:, i] != 0, b != 0)


def test_top_eig_step_cap_keeps_the_majorisation_safe(lib):
    # q > 512 (the Lanczos step cap) with a tightly clustered top spectrum: the Ritz value may not reach 1e-10 within the cap.
    # An unconverged Ritz value under-estimates lambda_max, so the kernel adds the residual bound: the returned value must
    # never fall below the true top eigenvalue (d = 1.0005 * it is the only margin the logistic entries have) and stay close.
    import ctypes
    import torch
    from oem_b200 import api
    q = 900
    g = torch.Generator(device="cuda").manual_seed(9)
    Q, _ = torch.linalg.qr(torch.randn(q, q, generator=g, dtype=torch.float64, device="cuda"))
    ev = torch.cat([torch.rand(q - 200, generator=g, dtype=torch.float64, device="cuda") * 0.9,
                    1.0 - 1e-7 * torch.rand(200, generator=g, dtype=torch.float64, device="cuda")])
    XX = (Q * ev) @ Q.t()
    XX = 0.5 * (XX + XX.t())
    true = float(torch.linalg.eigvalsh(XX)[-1])
    out, steps = ctypes.c_double(), ctypes.c_int()
    api._check(api.load().oemb200_top_eig(XX.data_ptr(), q, ctypes.byref(out), ctypes.byref(steps), None))
    assert out.value >= true * (1 - 1e-13), (out.value, true, steps.value)
    assert out.value <= true * (1 + 1e-6), (out.value, true, steps.value)


def test_wide_p_is_refused_up_front(lib):
    # n <= p is served by the p x p Gram route; a p the path kernel cannot hold must fail cleanly BEFORE the Gram is
    # allocated (status 4, a message that says what fits), not with an out-of-memory or a launch error afterwards
    rng = np.random.default_rng(0)
    X = np.asfortranarray(rng.normal(size=(50, 9000)))
    y = rng.normal(size=50)
    a = args_xy(X, y, "gaussian", ["lasso", "mcp", "scad"], nlambda=5)
    with pytest.raises(lib.OemB200Error, match="coefficients") as ei:
        lib.oem_fit_dense(*a)
    assert ei.value.code == 4
    X = np.asfortranarray(rng.normal(size=(60, 2500)))            # wide but within the limit: the n <= p branch works
    got = lib.oem_fit_dense(*args_xy(X, rng.normal(size=60), "gaussian", ["lasso"], nlambda=5, lmin_ratio=0.5))
    assert got["beta"][0].shape == (2501, 5)


def test_device_matrix_handle_fits_without_reupload(lib, oracle, tmp_path):
    # oemb200_matrix_create: x is uploaded once; every *_h entry then runs with zero host -> device traffic for x
    # (device-resident y: h2d_bytes == 0; host y: 8 n bytes), and repeated logistic fits reuse the handle's slab copy
    import torch
    X, y = gaussian_problem(211, 6000, 140, mean_x=0.1)
    Xh = lib.DeviceMatrix(X)
    assert Xh.shape == X.shape and Xh.h2d_bytes == X.nbytes
    a = args_xy(X, y, "gaussian", ["lasso", "mcp"], nlambda=15)
    ref = oracle.oem_fit_dense(*a)
    a[0] = Xh
    g1 = lib.oem_fit_dense(*a)
    assert_same_fit(g1, ref)
    assert g1["stats"]["h2d_bytes"] == 8 * X.shape[0]
    a[1] = torch.from_numpy(y).cuda()
    g2 = lib.oem_fit_dense(*a)
    assert g2["stats"]["h2d_bytes"] == 0
    assert all(np.array_equal(b1, b2) for b1, b2 in zip(g1["beta"], g2["beta"]))
    assert_same_fit(lib.oem_fit_big(*a), oracle.oem_fit_big(*args_xy(X, y, "gaussian", ["lasso", "mcp"], nlambda=15)))
    # xval + predict on the handle
    rng = np.random.default_rng(5)
    foldid = 1 + rng.permutation(X.shape[0]) % 4
    xa = xval_args(X, y, ["lasso"], foldid, 4, nlambda=12)
    refx = oracle.oem_xval_dense(*xa)
    xa[0] = Xh
    gx = lib.oem_xval_dense(*xa)
    assert_same_fit(gx, refx)
    assert np.allclose(gx["cvm"][0], refx["cvm"][0], rtol=1e-9)
    pred = lib.predict_matrix(Xh, g1["beta"][0])
    assert np.allclose(pred, X @ g1["beta"][0][1:] + g1["beta"][0][0], rtol=0, atol=1e-10)
    # logistic: the first fit builds the slab copy, the second one finds it
    Xb, yb = binomial_problem(212, 5000, 200)
    Xbh = lib.DeviceMatrix(Xb)
    ab = args_xy(Xb, yb, "binomial", ["lasso"], nlambda=8, lmin_ratio=5e-2)
    refb = oracle.oem_fit_logistic_dense(*ab)
    ab[0] = Xbh
    l1 = lib.oem_fit_logistic_dense(*ab)
    l2 = lib.oem_fit_logistic_dense(*ab)
    assert_same_fit(l1, refb)
    assert l1["stats"]["ms_relayout"] > 0 and l2["stats"]["ms_relayout"] == 0
    assert np.array_equal(l1["beta"][0], l2["beta"][0])
    # from a bigmemory backing file (.bk = raw column-major doubles)
    from oem_b200 import bigmatrix
    bk, desc = str(tmp_path / "m.bk"), str(tmp_path / "m.desc")
    bigmatrix.write(X, bk, desc)
    Xf = lib.DeviceMatrix(bk, shape=X.shape)
    a[0] = Xf
    g3 = lib.oem_fit_dense(*a)
    assert all(np.array_equal(b1, b3) for b1, b3 in zip(g1["beta"], g3["beta"]))
    Xf.close(); Xh.close(); Xbh.close()
    with pytest.raises(ValueError, match="closed"):
        lib.oem_fit_dense(*a)


def test_errors_mirror_reference(lib):
    X, y = gaussian_problem(1, 100, 5)
    a = args_xy(X, y, "binomial", ["lasso"])
    with pytest.raises(lib.OemB200Error, match="binomial not available"):
        lib.oem_fit_dense(*a)
    a = args_xy(X, y, "gaussian", ["lasso"])
    a[4] = np.ones(100)
    with pytest.raises(lib.OemB200Error, match="weights not implemented"):
        lib.oem_fit_dense(*a)
    a = args_xy(X, y, "gaussian", ["nope"])
    with pytest.raises(lib.OemB200Error, match="unknown penalty"):
        lib.oem_fit_big(*a)


def xval_args(X, y, penalty, foldid, nfolds, **kw):
    tm = kw.pop("type_measure", "mse")
    cl = kw.get("compute_loss", False)
    a = args_xy(X, y, "gaussian", penalty, **kw)
    return a[:17] + [nfolds, foldid, cl, tm, a[18]]


@pytest.mark.parametrize("standardize,intercept,measure", [(True, True, "mse"), (False, True, "mae"), (True, False, "mse")])
def test_xval(lib, oracle, standardize, intercept, measure):
    # BASELINE config 3 shape at n = 6000: lasso + grp.lasso + mcp, 10 folds, fold Grams in one pass
    X, y = gaussian_problem(103, 6000, 50, coef="vignette", noise=4.0)
    rng = np.random.default_rng(103)
    foldid = 1 + rng.permutation(6000) % 10
    g = np.repeat(np.arange(1, 11), 5)
    groups = np.concatenate([[0], g]) if intercept else g
    a = xval_args(X, y, ["lasso", "grp.lasso", "mcp"], foldid, 10, groups=groups, unique_groups=np.unique(groups),
                  nlambda=30, standardize=standardize, intercept=intercept, type_measure=measure, compute_loss=True)
    got, ref = lib.oem_xval_dense(*a), oracle.oem_xval_dense(*a)
    assert_same_fit(got, ref)
    for pp in range(3):
        assert np.allclose(got["cvm"][pp], ref["cvm"][pp], rtol=1e-9, atol=0)
        assert np.allclose(got["cvsd"][pp], ref["cvsd"][pp], rtol=1e-8, atol=0)
        assert np.allclose(got["loss"][pp], ref["loss"][pp], rtol=1e-9)


@pytest.mark.parametrize("standardize,intercept,measure", [(True, True, "mse"), (True, False, "mae"), (False, False, "mse")])
def test_xval_observation_weights(lib, oracle, standardize, intercept, measure):
    # xval.oem(weights=): X'WX fold Grams (XtWX_xval[_int], oem_xval_dense.h:489-627), weighted CV score
    X, y = gaussian_problem(31, 3001, 30, coef="vignette", noise=2.0)
    rng = np.random.default_rng(31)
    foldid = 1 + rng.permutation(3001) % 5
    w = rng.uniform(0.25, 3.0, size=3001)
    a = xval_args(X, y, ["lasso", "mcp", "elastic.net"], foldid, 5, nlambda=25, alpha=0.7, standardize=standardize,
                  intercept=intercept, type_measure=measure, compute_loss=True)
    a[4] = w
    got, ref = lib.oem_xval_dense(*a), oracle.oem_xval_dense(*a)
    assert_same_fit(got, ref)
    for pp in range(3):
        assert np.allclose(got["cvm"][pp], ref["cvm"][pp], rtol=1e-9, atol=0)
        assert np.allclose(got["cvsd"][pp], ref["cvsd"][pp], rtol=1e-8, atol=0)
        assert np.allclose(got["loss"][pp], ref["loss"][pp], rtol=1e-9)
    # unit weights are the unweighted fit (the weighted path takes its column sums from the sweep kernel, the unweighted one
    # from the Gram launch: same numbers up to summation order)
    a[4] = np.ones(3001)
    one = lib.oem_xval_dense(*a)
    a[4] = []
    none = lib.oem_xval_dense(*a)
    for pp in range(3):
        assert np.allclose(one["beta"][pp], none["beta"][pp], rtol=0, atol=1e-11)
        assert np.allclose(one["cvm"][pp], none["cvm"][pp], rtol=1e-11)
    with pytest.raises(Exception):
        a[4] = np.ones(17)
        lib.oem_xval_dense(*a)


def test_xval_many_columns_uneven_folds(lib, oracle):
    # more than 320 (penalty x lambda) columns -> two column blocks in the scoring GEMM; ragged folds; odd n
    X, y = gaussian_problem(9, 2501, 23, noise=2.0)
    rng = np.random.default_rng(9)
    foldid = rng.choice([1, 2, 3], size=2501, p=[0.6, 0.3, 0.1])
    a = xval_args(X, y, ["lasso", "scad", "mcp", "elastic.net"], foldid, 3, nlambda=90, alpha=0.5)
    got, ref = lib.oem_xval_dense(*a), oracle.oem_xval_dense(*a)
    assert_same_fit(got, ref)
    for pp in range(4):
        assert np.allclose(got["cvm"][pp], ref["cvm"][pp], rtol=1e-9)
        assert np.allclose(got["cvsd"][pp], ref["cvsd"][pp], rtol=1e-8)


def test_golden_on_gpu(lib):
    import json, os
    from golden.make_golden import CASES, run_case
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_oracle.json")))
    for name in CASES:
        got, ref = run_case(lib, name), gold[name]
        assert np.allclose(got["d"], ref["d"], rtol=1e-9), name
        for pp in range(len(ref["beta_checksum"])):
            assert np.allclose(got["beta_checksum"][pp], ref["beta_checksum"][pp], rtol=0, atol=2e-7), name
        if "cvm_checksum" in ref:
            assert np.allclose(got["cvm_checksum"], ref["cvm_checksum"], rtol=1e-9), name
            assert np.allclose(got["cvsd_checksum"], ref["cvsd_checksum"], rtol=1e-8), name


@pytest.mark.parametrize("n,p", [(40, 1), (50, 3), (200, 7), (300, 129), (77, 8)])
def test_ragged_shapes(lib, oracle, n, p):
    # columns not a multiple of the 8-wide MMA atom / 128-wide panel, odd and tiny row counts
    X, y = gaussian_problem(n + p, n, p)
    a = args_xy(X, y, "gaussian", ["lasso", "ols"], nlambda=8, opts=dict(tol=1e-9))
    assert_same_fit(lib.oem_fit_dense(*a), oracle.oem_fit_dense(*a))
    assert_same_fit(lib.oem_fit_big(*a), oracle.oem_fit_big(*a))


def test_constant_column_and_single_lambda(lib, oracle):
    X, y = gaussian_problem(31, 500, 6)
    X[:, 2] = 0.0                       # zero column: scale 0 -> 1 in every standardisation convention
    X[:, 4] = 3.0                       # constant column: centred norm 0 -> scale 1 (DataStd), non-zero uncentred norm
    a = args_xy(X, y, "gaussian", ["lasso"], lambda_=[np.array([0.05])], opts=dict(tol=1e-9))
    got, ref = lib.oem_fit_dense(*a), oracle.oem_fit_dense(*a)
    assert got["beta"][0].shape == (7, 1)
    assert_same_fit(got, ref)
    assert_same_fit(lib.oem_fit_big(*a), oracle.oem_fit_big(*a))


def test_maxit_exhausted_reports_maxit_plus_one(lib, oracle):
    X, y = gaussian_problem(32, 400, 30, mean_x=2.0)      # large mean + intercept column: slow convergence
    a = args_xy(X, y, "gaussian", ["lasso"], nlambda=6, standardize=False, opts=dict(maxit=5, tol=1e-12))
    got, ref = lib.oem_fit_big(*a), oracle.oem_fit_big(*a)
    assert np.array_equal(got["niter"][0], ref["niter"][0]) and got["niter"][0].max() == 6     # src/oem_base.h:94-109
    assert_same_fit(got, ref)


def test_unsupported_paths_fail_loudly(lib):
    X, y = gaussian_problem(1, 20, 30)           # n <= p + intercept in big.oem: the reference's own branch is incoherent
    with pytest.raises(lib.OemB200Error) as ei:  # (X' has p rows, beta p + 1: src/oem_big.h:570-581), so there is nothing to match
        lib.oem_fit_big(*args_xy(X, y, "gaussian", ["lasso"]))
    assert ei.value.code == 4
    Xs, ys = gaussian_problem(1, 200, 5)
    a = args_xy(Xs, ys, "gaussian", ["lasso"])
    bad = a[:17] + [3, np.array([0] * 200), False, "mse", a[18]]
    with pytest.raises(lib.OemB200Error, match="foldid"):
        lib.oem_xval_dense(*bad)


@pytest.mark.parametrize("n,p", [(20, 30), (25, 25), (60, 200)])
@pytest.mark.parametrize("standardize,intercept", [(True, True), (False, False), (False, True)])
def test_dense_n_le_p_branch(lib, oracle, n, p, standardize, intercept):
    # src/oem_dense.h:474-483, 515-521 (XX' form): d from XX'/n, u = X'(Y - X beta)/n + d beta
    X, y = gaussian_problem(600 + n + p, n, p)
    groups = np.arange(p) // 5 + 1
    a = args_xy(X, y, "gaussian", ["lasso", "mcp", "grp.lasso"], nlambda=12, lmin_ratio=0.01, standardize=standardize,
                intercept=intercept, groups=groups, unique_groups=np.unique(groups), opts=dict(maxit=500, tol=1e-9))
    got, ref = lib.oem_fit_dense(*a), oracle.oem_fit_dense(*a)
    assert_same_fit(got, ref)


def test_wide_problem_streams_A_from_l2(lib, oracle):
    # q = 2400: a member's column slice of A (24 x 2404 doubles) no longer fits shared memory next to the iterate
    # buffers, so the path kernel streams its slice from L2 (a_in_smem = false) -- same answers
    X, y = gaussian_problem(77, 6000, 2400, nnz=10)
    lam = [np.geomspace(0.3, 0.05, 4)]
    a = args_xy(X, y, "gaussian", ["lasso"], lambda_=lam, opts=dict(maxit=40, tol=1e-7))
    got, ref = lib.oem_fit_big(*a), oracle.oem_fit_big(*a)
    assert_same_fit(got, ref)
