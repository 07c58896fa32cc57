"""Binomial cross-validation (oem_xval_logistic_dense): the fused multi-model data pass against torch FP64, the full-data
model against oem_fit_logistic_dense, cvm / cvsd against the composition it replaces (K + 1 separate logistic fits at the
full model's lambdas plus predict_matrix), and everything against a CPU twin built from oracle.oem_fit_logistic_dense.
The tests without the gpu mark check the interface and the twin's definition on the CPU."""
import math

import numpy as np
import pytest

from cases import DEFAULT_OPTS, args_xy, assert_same_fit, binomial_problem

EUNSUPPORTED, EINVAL, ENODEVICE = 4, 1, 2
MEASURES = ["deviance", "class", "mse", "mae"]


def xargs(a, nfolds, foldid, type_measure="deviance"):
    """args_xy list -> argument list of oem_xval_logistic_dense."""
    return a[:17] + [nfolds, np.asarray(foldid, dtype=np.int32), a[17], type_measure, a[18]]


def measure(y, prob, type_measure):
    """Held-out loss per row and lambda, R/cv_oem.R:288-330 (as in frontend.cv_oem) for y in {0, 1}."""
    y1 = y[:, None]
    y0 = 1.0 - y1
    if type_measure == "deviance":
        pm = np.minimum(np.maximum(prob, 1e-5), 1 - 1e-5)
        return -2.0 * (y0 * np.log(1 - pm) + y1 * np.log(pm))
    if type_measure == "class":
        return y0 * (prob > 0.5) + y1 * (prob <= 0.5)
    if type_measure == "mse":
        return (y0 - (1 - prob)) ** 2 + (y1 - prob) ** 2
    return np.abs(y0 - (1 - prob)) + np.abs(y1 - prob)


def compose(fit, predict_response, a, nfolds, foldid):
    """The definition: the full-data fit, one fit per fold on the other rows at the full fit's lambda sequence, and
    the held-out response of every row under its fold's model.  Returns (full fit, fold fits, score(type_measure))."""
    X, y = np.asarray(a[0]), np.asarray(a[1])
    foldid = np.asarray(foldid)
    full = fit(*a)
    lam = [np.asarray(l)[:np.asarray(b).shape[1]] for l, b in zip(full["lambda_"], full["beta"])]
    folds = []
    for k in range(1, nfolds + 1):
        tr = foldid != k
        ak = list(a)
        ak[0], ak[1], ak[8], ak[17] = np.asfortranarray(X[tr]), y[tr], lam, False
        folds.append(fit(*ak))
    probs = []
    for pp in range(len(full["beta"])):
        P = np.empty((X.shape[0], full["beta"][pp].shape[1]))
        for k in range(1, nfolds + 1):
            idx = np.nonzero(foldid == k)[0]
            P[idx, :] = predict_response(np.asfortranarray(X[idx]), np.asarray(folds[k - 1]["beta"][pp]))
        probs.append(P)

    def score(type_measure):
        cvm, cvsd = [], []
        for P in probs:
            T = measure(y, P, type_measure)
            m = T.mean(axis=0)
            cvm.append(m)
            cvsd.append(np.sqrt(((T - m[None, :]) ** 2).sum(axis=0) / (len(y) - 1.0)) / np.sqrt(len(y)))
        return cvm, cvsd
    return full, folds, score


def twin(oracle, a, nfolds, foldid):
    """CPU twin: the composition on oracle.oem_fit_logistic_dense and a numpy predict."""
    return compose(oracle.oem_fit_logistic_dense,
                   lambda Xh, B: 1.0 / (1.0 + np.exp(-(Xh @ B[1:, :] + B[0:1, :]))), a, nfolds, foldid)


def problem(seed=21, n=600, p=10, nfolds=3, uneven=False):
    X, y = binomial_problem(seed, n, p)
    rng = np.random.default_rng(seed)
    if uneven:
        w = np.arange(1, nfolds + 1, dtype=np.float64)
        foldid = rng.choice(np.arange(1, nfolds + 1), size=n, p=w / w.sum())
    else:
        foldid = rng.permutation(np.resize(np.arange(1, nfolds + 1), n))
    return X, y, foldid.astype(np.int32)


# ---------------------------------------------------------------- CPU ----------------------------------------------------

def test_new_symbols_are_exported(lib):
    L = lib.load()
    for s in ("oemb200_xval_logistic_dense", "oemb200_xval_logistic_dense_h", "oemb200_logit_fold_pass"):
        assert s in lib.EXPORTS and hasattr(L, s)
    assert callable(lib.oem_xval_logistic_dense) and callable(lib.logit_fold_pass)


def test_no_device_no_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the no-device behaviour is checked on the CPU box")
    X, y, foldid = problem(n=200, p=10)
    a = args_xy(X, y, "binomial", ["lasso"], nlambda=5)
    with pytest.raises(lib.OemB200Error) as ei:
        lib.oem_xval_logistic_dense(*xargs(a, 3, foldid))
    assert ei.value.code == ENODEVICE


@pytest.mark.parametrize("kw,match", [
    (dict(type_measure="auc"), "cv_oem"),
    (dict(type_measure="rmse"), "type.measure"),
    (dict(hessian_type="full"), "upper.bound"),
    (dict(nonbinary=True), "binary"),
    (dict(weights=np.ones(300)), "weights"),
])
def test_frontend_rejects_before_any_device_use(kw, match):
    from oem_b200 import frontend as fe
    X, y, foldid = problem(n=300, p=10)
    if kw.pop("nonbinary", False):
        y = y + np.arange(300) % 3
    with pytest.raises(ValueError, match=match):
        fe.xval_oem(X, y, family="binomial", foldid=foldid, penalty="lasso", nlambda=5, **kw)


def _refused(lib, a, nfolds, foldid, tm="deviance", opts=None):
    from oem_b200 import api
    xa = xargs(a, nfolds, foldid, tm)
    if opts is not None:
        xa[-1] = opts
    with pytest.raises(lib.OemB200Error) as ei:
        api.oem_xval_logistic_dense(*xa)
    return ei.value


def test_refused_cases_return_their_codes(lib):
    # every refusal happens before the device is touched, so the codes are the same with and without a GPU
    from oem_b200 import api
    X, y, foldid = problem(n=300, p=10)
    a = args_xy(X, y, "binomial", ["lasso"], nlambda=5)
    assert _refused(lib, a, 3, foldid, opts=dict(DEFAULT_OPTS, hessian_type="full")).code == EUNSUPPORTED
    o = api.make_opts(DEFAULT_OPTS)
    o.world = 2
    assert _refused(lib, a, 3, foldid, opts=o).code == EUNSUPPORTED
    aw = list(a)
    aw[4] = np.ones(300)
    assert _refused(lib, aw, 3, foldid).code == EUNSUPPORTED
    for p in (5, 2049):
        Xp = np.zeros((20, p)) if p > 2048 else X[:, :p]
        yp = y[:Xp.shape[0]]
        ap = args_xy(Xp, yp, "binomial", ["lasso"], nlambda=5)
        assert _refused(lib, ap, 3, foldid[:Xp.shape[0]]).code == EUNSUPPORTED
    e = _refused(lib, a, 3, foldid, tm="auc")
    assert e.code == EINVAL and "cv_oem" in str(e)
    ag = list(a)
    ag[2] = "gaussian"
    assert _refused(lib, ag, 3, foldid).code == EINVAL


def test_twin_full_model_is_the_logistic_fit(oracle):
    X, y, foldid = problem(n=400, p=8)
    a = args_xy(X, y, "binomial", ["lasso", "mcp.net"], nlambda=8, lmin_ratio=1e-2, compute_loss=True)
    full, folds, _ = twin(oracle, a, 3, foldid)
    ref = oracle.oem_fit_logistic_dense(*a)
    for key in ("beta", "lambda_", "niter", "loss"):
        for g, r in zip(full[key], ref[key]):
            assert np.array_equal(g, r)
    assert full["d"] == ref["d"]
    # and a fold model is the plain fit on its training rows at the full model's lambdas
    tr = foldid != 2
    ak = list(a)
    ak[0], ak[1], ak[8], ak[17] = np.asfortranarray(X[tr]), y[tr], [np.asarray(l) for l in ref["lambda_"]], False
    r2 = oracle.oem_fit_logistic_dense(*ak)
    assert all(np.array_equal(g, r) for g, r in zip(folds[1]["beta"], r2["beta"]))


# ---------------------------------------------------------------- GPU ----------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("M,p", [(1, 8), (2, 100), (11, 130), (11, 1000), (21, 1000), (11, 2048), (21, 8)])
def test_fold_pass_matches_torch(lib, M, p):
    import torch
    g = torch.Generator().manual_seed(1000 * M + p)
    n = 3001                                                    # ragged: not a multiple of the 4-row slab
    X = torch.randn(p, n, generator=g, dtype=torch.float64).t()  # column-major on the host ...
    Xd = X.t().contiguous().cuda().t()                           # ... and on the device
    B = torch.randn(M, p, generator=g, dtype=torch.float64) * (0.5 / math.sqrt(p))
    b0 = torch.randn(M, generator=g, dtype=torch.float64) * 0.3
    y = (torch.rand(n, generator=g, dtype=torch.float64) < 0.4).double()
    fold = torch.randint(0, max(M, 2) + 1, (n,), generator=g, dtype=torch.int32)   # 0 = a row of no model
    conv = torch.zeros(M, dtype=torch.int32)
    if M > 2:
        conv[M // 2] = 1                                         # a converged model: no arithmetic, grad row untouched
    grad, ms, ms_rl, sweeps = lib.logit_fold_pass(Xd, B.cuda(), b0.cuda(), y.cuda(), fold.cuda(), conv.cuda(), reps=2)
    grad = grad.cpu()
    assert sweeps >= 1 and ms > 0 and ms_rl > 0
    if (M, p) in ((21, 1000), (11, 2048)):
        assert sweeps >= 2
    for m in range(M):
        if conv[m]:
            assert torch.isnan(grad[m]).all()
            continue
        mask = (fold != 0) & (fold != m)
        r = torch.where(mask, y - torch.sigmoid(X @ B[m] + b0[m]), torch.zeros(()))
        ref = torch.cat([r.sum().view(1), X.t() @ r])
        scale = torch.cat([r.abs().sum().view(1), X.abs().t() @ r.abs()])
        err = (grad[m] - ref).abs()
        assert bool((err <= 1e-12 * scale + 1e-300).all()), (m, float((err / scale).max()))


@pytest.mark.gpu
def test_full_model_is_the_logistic_fit_with_loss(lib):
    X, y, foldid = problem(seed=104, n=4000, p=40, nfolds=5)
    groups = np.concatenate([[0], np.repeat(np.arange(1, 9), 5)])
    a = args_xy(X, y, "binomial", ["lasso", "mcp.net", "grp.lasso"], groups=groups, unique_groups=np.unique(groups),
                alpha=0.7, nlambda=15, lmin_ratio=1e-2, compute_loss=True)
    got = lib.oem_xval_logistic_dense(*xargs(a, 5, foldid))
    ref = lib.oem_fit_logistic_dense(*a)
    assert_same_fit(got, ref, tol=1e-8)
    for lg, lr in zip(got["loss"], ref["loss"]):
        assert np.allclose(lg, lr, rtol=1e-9)
    st = got["stats"]
    assert st["data_passes"] >= 1 and st["gemv_bytes"] > 0


@pytest.mark.gpu
def test_cv_matches_the_composition_it_replaces(lib):
    X, y, foldid = problem(seed=7, n=3000, p=30, nfolds=4, uneven=True)     # uneven folds
    a = args_xy(X, y, "binomial", ["lasso", "mcp"], nlambda=12, lmin_ratio=1e-2)
    full, _, score = compose(lib.oem_fit_logistic_dense, lambda Xh, B: lib.predict_matrix(Xh, B, response=True), a, 4, foldid)
    n = len(y)
    for tm in MEASURES:
        got = lib.oem_xval_logistic_dense(*xargs(a, 4, foldid, tm))
        assert_same_fit(got, full, tol=1e-8)
        cvm, cvsd = score(tm)
        for pp in range(2):
            if tm == "class":
                assert np.array_equal(np.rint(got["cvm"][pp] * n), np.rint(cvm[pp] * n)), tm
                assert np.allclose(got["cvsd"][pp], cvsd[pp], rtol=1e-12, atol=1e-12), tm
            else:
                assert np.allclose(got["cvm"][pp], cvm[pp], rtol=1e-9, atol=0), tm
                assert np.allclose(got["cvsd"][pp], cvsd[pp], rtol=1e-9, atol=1e-12), tm


@pytest.mark.gpu
@pytest.mark.parametrize("standardize,intercept", [(False, False), (True, False), (False, True), (True, True)])
def test_against_the_oracle_twin(lib, oracle, standardize, intercept):
    X, y, foldid = problem(seed=31, n=700, p=12, nfolds=3, uneven=True)
    g = np.repeat(np.arange(1, 5), 3)
    groups = np.concatenate([[0], g]) if intercept else g
    a = args_xy(X, y, "binomial", ["lasso", "mcp.net", "grp.lasso", "sparse.grp.lasso"], groups=groups,
                unique_groups=np.unique(groups), alpha=0.8, nlambda=10, lmin_ratio=1e-2, standardize=standardize,
                intercept=intercept, compute_loss=True)
    full, _, score = twin(oracle, a, 3, foldid)
    for tm in ("deviance", "class"):
        got = lib.oem_xval_logistic_dense(*xargs(a, 3, foldid, tm))
        assert_same_fit(got, full, tol=1e-8)
        for lg, lr in zip(got["loss"], full["loss"]):
            assert np.allclose(lg, lr, rtol=1e-9)
        cvm, cvsd = score(tm)
        for pp in range(4):
            if tm == "class":
                assert np.array_equal(np.rint(got["cvm"][pp] * len(y)), np.rint(cvm[pp] * len(y)))
            else:
                # where every held-out row scores the same (at lambda_max without an intercept every p = 1/2), M2 is
                # rounding noise on both sides
                assert np.allclose(got["cvm"][pp], cvm[pp], rtol=1e-8, atol=0)
                assert np.allclose(got["cvsd"][pp], cvsd[pp], rtol=1e-8, atol=1e-12)


@pytest.mark.gpu
def test_irls_maxit_exhausted_and_bit_reproducible(lib):
    X, y, foldid = problem(seed=5, n=2500, p=20, nfolds=4)
    a = args_xy(X, y, "binomial", ["lasso"], nlambda=10, lmin_ratio=1e-3, opts=dict(irls_maxit=2, irls_tol=1e-12))
    r1 = lib.oem_xval_logistic_dense(*xargs(a, 4, foldid))
    r2 = lib.oem_xval_logistic_dense(*xargs(a, 4, foldid))
    ref = lib.oem_fit_logistic_dense(*a)
    assert np.all(r1["niter"][0] == 3)                          # maxit + 1, as the reference reports an exhausted loop
    assert_same_fit(r1, ref, tol=1e-8)
    for key in ("beta", "niter", "cvm", "cvsd"):
        for u, v in zip(r1[key], r2[key]):
            assert np.array_equal(u, v), key
    assert r1["d"] == r2["d"]


@pytest.mark.gpu
def test_device_matrix_handle(lib):
    X, y, foldid = problem(seed=9, n=3001, p=24, nfolds=5)
    a = args_xy(X, y, "binomial", ["lasso"], nlambda=10, lmin_ratio=1e-2)
    plain = lib.oem_xval_logistic_dense(*xargs(a, 5, foldid))
    dm = lib.DeviceMatrix(X)
    try:
        ah = list(a)
        ah[0] = dm
        got = lib.oem_xval_logistic_dense(*xargs(ah, 5, foldid))
    finally:
        dm.close()
    assert got["stats"]["h2d_bytes"] == 8 * len(y)              # y only: x stays on the device
    for key in ("beta", "cvm", "cvsd"):
        for u, v in zip(got[key], plain[key]):
            assert np.array_equal(u, v), key


@pytest.mark.gpu
def test_frontend_binomial_xval(lib):
    from oem_b200 import frontend as fe
    X, y, foldid = problem(seed=13, n=2000, p=16, nfolds=4)
    fit = fe.xval_oem(X, y, family="binomial", foldid=foldid, penalty=["lasso", "mcp"], nlambda=10, compute_loss=True)
    ref = fe.oem(X, y, family="binomial", penalty=["lasso", "mcp"], nlambda=10, compute_loss=True)
    for pen in ("lasso", "mcp"):
        assert np.max(np.abs(fit["beta"][pen] - ref["beta"][pen])) <= 1e-8
    assert fit["best_model"] in ("lasso", "mcp") and fit["lambda_min"] > 0
    resp = fe.predict(fit, newx=X[:50], type="response")
    assert resp.shape[0] == 50 and np.all((resp > 0) & (resp < 1))
    cls = fe.predict(fit, newx=X[:50], type="class")
    assert set(np.unique(cls)) <= {1, 2}
    assert np.allclose(fe.logLik(fit), -np.asarray(ref["loss"][0]), rtol=1e-9)
