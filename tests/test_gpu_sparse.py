"""oem_fit_sparse (SURVEY.md 8f row 4): dgCMatrix input through the C ABI against the oracle's restatement of
src/oem_sparse.cpp / oem_sparse.h -- all penalties, the four standardize / intercept combinations (the intercept column
is the constant `intval`, get_beta() rescales beta(0) in place), compute.loss, empty rows / columns, device-resident
slots, run-to-run determinism of the atomics-free Gram."""
import re

import numpy as np
import pytest

from cases import args_xy, assert_same_fit, sparse_problem

pytestmark = pytest.mark.gpu

ALL_PENS = ["lasso", "ols", "elastic.net", "scad", "scad.net", "mcp", "mcp.net", "grp.lasso", "grp.lasso.net", "grp.mcp",
            "grp.scad", "grp.mcp.net", "grp.scad.net", "sparse.grp.lasso"]


def _groups(p, size, intercept):
    g = np.arange(p) // size + 1
    if intercept:                     # R/oem.R:300-337: group 0 for the explicit intercept of a sparse x
        g = np.concatenate([[0], g])
    return g, np.unique(g)


@pytest.mark.parametrize("standardize,intercept", [(True, True), (True, False), (False, True), (False, False)])
def test_sparse_all_penalties(lib, oracle, standardize, intercept):
    X, y = sparse_problem(70 + 2 * standardize + intercept, 4000, 45, density=0.08, shift_y=2.0, empty_cols=(7,), empty_rows=5)
    g, ug = _groups(45, 5, intercept)
    a = args_xy(X, y, "gaussian", ALL_PENS, groups=g, unique_groups=ug, alpha=0.6, gamma=3.5, tau=0.4, nlambda=15,
                standardize=standardize, intercept=intercept, compute_loss=True, opts=dict(tol=1e-9))
    got, ref = lib.oem_fit_sparse(*a), oracle.oem_fit_sparse(*a)
    assert_same_fit(got, ref)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg[:len(lr)], lr, rtol=1e-10, atol=0)


@pytest.mark.parametrize("n,p,density", [(300, 7, 0.5), (2500, 130, 0.02), (20000, 300, 0.01), (9000, 1001, 0.004)])
def test_sparse_shapes(lib, oracle, n, p, density):
    # p around / above the 4 * SMs split threshold, ragged sizes, very sparse rows (many empty)
    X, y = sparse_problem(n + p, n, p, density=density)
    a = args_xy(X, y, "gaussian", ["lasso", "mcp"], nlambda=10, lmin_ratio=1e-3, opts=dict(tol=1e-8))
    got, ref = lib.oem_fit_sparse(*a), oracle.oem_fit_sparse(*a)
    assert_same_fit(got, ref)
    assert got["stats"]["gram_launches"] == 1 and got["stats"]["kernel_launches"] >= 8


@pytest.mark.parametrize("route", ["dense", "sparse", None])
def test_sparse_routes_agree(lib, oracle, monkeypatch, route):
    # 40 % density at p = 80: the cost model (sum nnz(row)^2 against n p^2) picks the dense-tile route by itself (None);
    # both forced routes must give the same fit
    if route:
        monkeypatch.setenv("OEMB200_SPARSE_ROUTE", route)
    X, y = sparse_problem(33, 3001, 80, density=0.4, shift_y=0.5, empty_rows=3)
    g, ug = _groups(80, 8, True)
    a = args_xy(X, y, "gaussian", ["lasso", "grp.lasso", "scad"], groups=g, unique_groups=ug, nlambda=12, compute_loss=True,
                opts=dict(tol=1e-9))
    got, ref = lib.oem_fit_sparse(*a), oracle.oem_fit_sparse(*a)
    assert_same_fit(got, ref)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg[:len(lr)], lr, rtol=1e-10, atol=0)
    assert got["stats"]["gram_flops"] == (0.0 if route == "sparse" else 3001.0 * 80 * 81)      # which kernel built X'X


@pytest.mark.parametrize("standardize", [True, False])
@pytest.mark.parametrize("n,p", [(120, 180), (150, 150)])
def test_sparse_wide_no_intercept(lib, oracle, standardize, n, p):
    # n <= p without an intercept (src/oem_sparse.h:609-616, 630-640): raw-X iteration, `standardize` only in lambda_max
    # and get_beta(); with an intercept the reference is dimensionally inconsistent and the call is refused
    X, y = sparse_problem(300 + n + standardize, n, p, density=0.2, nnz=8, noise=0.3)
    g = np.arange(p) // 6 + 1
    a = args_xy(X, y, "gaussian", ["lasso", "mcp", "grp.lasso", "elastic.net"], groups=g, unique_groups=np.unique(g), alpha=0.7,
                nlambda=12, lmin_ratio=0.05, standardize=standardize, intercept=False, compute_loss=True,
                opts=dict(tol=1e-10, maxit=5000))
    got, ref = lib.oem_fit_sparse(*a), oracle.oem_fit_sparse(*a)
    assert_same_fit(got, ref)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg[:len(lr)], lr, rtol=1e-9, atol=0)
    a[16] = True
    with pytest.raises(Exception, match="dimensionally inconsistent"):
        lib.oem_fit_sparse(*a)


def test_sparse_equals_dense_identity(lib):
    # man/oem.Rd:104-125 -> docs/reference/oem.html prints max|dense - sparse| = 1.58e-15 / 1.61e-15 for
    # standardize = FALSE, intercept = FALSE (inputs from rsparsematrix, not reproducible): same order here
    X, y = sparse_problem(5, 6000, 60, density=0.03)
    g, ug = _groups(60, 5, False)
    a = args_xy(X, y, "gaussian", ["lasso", "grp.lasso"], groups=g, unique_groups=ug, standardize=False, intercept=False,
                nlambda=30)
    fs = lib.oem_fit_sparse(*a)
    a[0] = np.asfortranarray(X.toarray())
    a[8] = [np.array(l) for l in fs["lambda_"]]           # lambda = fit$lambda, as in the example
    fd = lib.oem_fit_dense(*a)
    for bs, bd in zip(fs["beta"], fd["beta"]):
        assert np.max(np.abs(bs - bd)) <= 1e-12


def test_sparse_device_slots_and_determinism(lib, oracle):
    import torch
    X, y = sparse_problem(11, 15000, 90, density=0.05)
    a = args_xy(X, y, "gaussian", ["lasso", "scad"], nlambda=12, compute_loss=True)
    ref = oracle.oem_fit_sparse(*a)
    dev = torch.device("cuda", 0)
    slots = (torch.from_numpy(X.indices.astype(np.int32)).to(dev), torch.from_numpy(X.indptr.astype(np.int32)).to(dev),
             torch.from_numpy(X.data).to(dev), X.shape)
    a[0], a[1] = slots, torch.from_numpy(y).to(dev)
    r1, r2 = lib.oem_fit_sparse(*a), lib.oem_fit_sparse(*a)
    assert_same_fit(r1, ref)
    for b1, b2 in zip(r1["beta"], r2["beta"]):
        assert np.array_equal(b1, b2)                      # no floating-point atomics anywhere: bit-identical reruns
    assert r1["d"] == r2["d"] and all(np.array_equal(u, v) for u, v in zip(r1["loss"], r2["loss"]))


def test_sparse_frontend_and_errors(lib, oracle):
    from oem_b200 import frontend as fe
    X, y = sparse_problem(21, 3000, 40, density=0.1, shift_y=-1.0)
    groups = np.repeat(np.arange(1, 9), 5)
    r = fe.oem(X, y, penalty=["lasso", "grp.lasso"], groups=groups, nlambda=20)
    g0 = np.concatenate([[0], groups])
    ref = oracle.oem_fit_sparse(X, y, "gaussian", ["lasso", "grp.lasso"], [], g0, np.unique(g0), [], [[], []], 20, 1e-4, 1.0,
                                3.0, 0.5, np.ones(40), True, True, False, dict(maxit=500, tol=1e-7))
    for i, pen in enumerate(["lasso", "grp.lasso"]):
        assert np.max(np.abs(r["beta"][pen] - ref["beta"][i])) <= 1e-8
    with pytest.raises(NotImplementedError, match="uninitialised"):      # the one combination the reference leaves undefined
        fe.oem(X, (y > 0).astype(float), family="binomial", penalty="lasso", standardize=False)
    Xw, yw = sparse_problem(3, 30, 40, density=0.3)
    with pytest.raises(lib.OemB200Error) as ei:           # n <= p: XX' branch
        lib.oem_fit_sparse(*args_xy(Xw, yw, "gaussian", ["lasso"]))
    assert ei.value.code == 4
    bad = (X.indices.astype(np.int32), X.indptr.astype(np.int32)[::-1].copy(), X.data, X.shape)
    a = args_xy(X, y, "gaussian", ["lasso"])
    a[0] = bad
    with pytest.raises(lib.OemB200Error, match="col_ptr"):
        lib.oem_fit_sparse(*a)
    ri = X.indices.astype(np.int32).copy()
    ri[5] = 3000                                            # row index == n
    a[0] = (ri, X.indptr.astype(np.int32), X.data, X.shape)
    with pytest.raises(lib.OemB200Error, match="outside"):
        lib.oem_fit_sparse(*a)
    ri = X.indices.astype(np.int32).copy()
    ri[1] = ri[0]                                           # duplicate entry inside column 0: not a valid dgCMatrix
    a[0] = (ri, X.indptr.astype(np.int32), X.data, X.shape)
    with pytest.raises(lib.OemB200Error, match="strictly increasing"):
        lib.oem_fit_sparse(*a)


def test_sparse_predict(lib):
    # predict.oem with a sparse newx: as.matrix(newx %*% nbeta) (R/methods.R:113-118) and the binomial response
    from oem_b200 import api, frontend as fe
    X, y = sparse_problem(41, 5003, 33, density=0.07, shift_y=1.0, empty_rows=4)
    rng = np.random.default_rng(5)
    B = rng.normal(size=(34, 9))
    want = B[0][None, :] + X @ B[1:]
    got = api.predict_matrix(X, B)
    assert got.shape == (5003, 9) and np.max(np.abs(got - want)) <= 1e-12
    assert np.max(np.abs(api.predict_matrix(X, B[1:]) - X @ B[1:])) <= 1e-12            # p x L (oem.xtx): no intercept row
    assert np.max(np.abs(api.predict_matrix(X, B, response=True) - 1 / (1 + np.exp(-want)))) <= 1e-14
    assert np.array_equal(got, api.predict_matrix(X, B))                               # fixed summation order
    fit = fe.oem(X, y, penalty=["lasso", "mcp"], nlambda=8)
    pr = fe.predict(fit, newx=X, which_model="mcp", s=[0.03, 0.2])
    nb = fe.predict(fit, which_model="mcp", s=[0.03, 0.2], type="coefficients")
    assert np.max(np.abs(pr - (nb[0][None, :] + X @ nb[1:]))) <= 1e-12
    with pytest.raises(api.OemB200Error, match="columns"):
        api.predict_matrix(X, B[:-2])


# ------------------------------------------------------------------------------------------------------------------
# oem_fit_logistic_sparse (src/oem_logistic_sparse.cpp:30): the three flag combinations the reference defines
# ------------------------------------------------------------------------------------------------------------------
def _sparse_binomial(seed, n, p, density):
    X, _ = sparse_problem(seed, n, p, density=density)
    rng = np.random.default_rng(seed + 1)
    b = np.zeros(p)
    b[:min(6, p)] = [1.0, -1.0, 0.8, -0.8, 0.5, -0.5][:min(6, p)]
    y = (rng.uniform(size=n) < 1.0 / (1.0 + np.exp(-(X @ b) + 0.3))).astype(np.float64)
    return X, y


@pytest.mark.parametrize("standardize,intercept", [(True, True), (True, False), (False, False)])
def test_logistic_sparse_matches_oracle(lib, oracle, standardize, intercept):
    X, y = _sparse_binomial(90 + 2 * standardize + intercept, 5000, 40, 0.08)
    g, ug = _groups(40, 5, intercept)
    a = args_xy(X, y, "binomial", ["lasso", "mcp", "grp.lasso", "scad.net"], groups=g, unique_groups=ug, alpha=0.7, nlambda=10,
                lmin_ratio=2e-2, standardize=standardize, intercept=intercept, compute_loss=True)
    got, ref = lib.oem_fit_logistic_sparse(*a), oracle.oem_fit_logistic_sparse(*a)
    assert_same_fit(got, ref, tol=1e-8)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg[:len(lr)], lr, rtol=1e-9)
    assert got["stats"]["gram_launches"] >= got["stats"]["data_passes"] > 0       # X'WX is rebuilt on every data pass


@pytest.mark.parametrize("route", ["sparse", "dense"])
def test_logistic_sparse_gram_routes_and_device_slots(lib, oracle, monkeypatch, route):
    import torch
    monkeypatch.setenv("OEMB200_SPARSE_ROUTE", route)
    X, y = _sparse_binomial(97, 6000, 130, 0.03)
    a = args_xy(X, y, "binomial", ["lasso"], nlambda=8, lmin_ratio=5e-2)
    ref = oracle.oem_fit_logistic_sparse(*a)
    assert_same_fit(lib.oem_fit_logistic_sparse(*a), ref, tol=1e-8)
    a[0] = (torch.from_numpy(X.indices.astype(np.int32)).cuda(), torch.from_numpy(X.indptr.astype(np.int32)).cuda(),
            torch.from_numpy(X.data).cuda(), X.shape)
    a[1] = torch.from_numpy(y).cuda()
    assert_same_fit(lib.oem_fit_logistic_sparse(*a), ref, tol=1e-8)


@pytest.mark.parametrize("irls_maxit", [1, 2, 3])
def test_logistic_sparse_irls_maxit_exhausted(lib, oracle, irls_maxit):
    # the IRLS cap cuts every loop short: niter reports irls_maxit + 1, and the iterate handed to the next lambda (after
    # get_beta()'s in-place intval scaling) is the one the last executed iteration produced
    X, y = _sparse_binomial(94, 3000, 60, 0.08)
    a = args_xy(X, y, "binomial", ["lasso", "mcp"], nlambda=8, lmin_ratio=2e-2, opts=dict(irls_maxit=irls_maxit, irls_tol=1e-9))
    got, ref = lib.oem_fit_logistic_sparse(*a), oracle.oem_fit_logistic_sparse(*a)
    assert_same_fit(got, ref, tol=1e-8)
    for ng, nr in zip(got["niter"], ref["niter"]):
        assert np.array_equal(ng, nr) and ng.max() == irls_maxit + 1


def test_logistic_sparse_register_resident_global_mode(lib, oracle, monkeypatch, capfd):
    # p = 599 (q = 600 with the intercept): the path launch of an IRLS iteration takes the cooperative global mode with the
    # register-resident mat-vec (rpt > 0), which forms XY = XX beta + grad inside the kernel instead of path_xy_kernel
    monkeypatch.setenv("OEMB200_PATH_PROF", "1")
    X, y = _sparse_binomial(93, 4000, 599, 0.03)
    a = args_xy(X, y, "binomial", ["lasso", "mcp"], nlambda=6, lmin_ratio=5e-2)
    got = lib.oem_fit_logistic_sparse(*a)
    prof = [line for line in capfd.readouterr().err.splitlines() if line.startswith("[path prof] mode=")]
    assert prof and all(re.search(r"mode=2 rpt=[2-5] ", line) for line in prof), prof[:3]
    assert_same_fit(got, oracle.oem_fit_logistic_sparse(*a), tol=1e-8)


def test_logistic_sparse_rejects_the_undefined_combination(lib):
    X, y = _sparse_binomial(98, 500, 10, 0.2)
    a = args_xy(X, y, "binomial", ["lasso"], nlambda=5, standardize=False, intercept=True)
    with pytest.raises(lib.OemB200Error, match="uninitialised"):
        lib.oem_fit_logistic_sparse(*a)
    a = args_xy(X, y, "gaussian", ["lasso"], nlambda=5)
    with pytest.raises(lib.OemB200Error, match="family"):
        lib.oem_fit_logistic_sparse(*a)


def test_frontend_oem_binomial_on_sparse_x(lib, oracle):
    from oem_b200 import frontend as fe
    X, y = _sparse_binomial(99, 4000, 30, 0.1)
    r = fe.oem(X, y, family="binomial", penalty=["lasso"], nlambda=8, lambda_min_ratio=0.05)
    ref = oracle.oem_fit_logistic_sparse(X, y, "binomial", ["lasso"], [], [], [], [], [[]], 8, 0.05, 1.0, 3.0, 0.5, np.ones(30),
                                         True, True, False, dict(maxit=500, tol=1e-7, irls_maxit=100, irls_tol=1e-3))
    assert np.max(np.abs(r["beta"]["lasso"] - ref["beta"][0])) <= 1e-8
