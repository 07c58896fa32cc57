"""R front-end mirrors (SURVEY.md 8f rank 1): oem(), oem_xtx(), xval_oem(), big_oem() with the reference's
argument names, defaults, validation and post-processing, on top of the C-ABI entries of oem_b200.api.

    R/oem.R:162-507        oem()        -> oem_fit_dense / oem_fit_logistic_dense
    R/oem_xtx.R:109-455    oem.xtx()    -> oem_xtx
    R/oem_xval.R:107-460   xval.oem()   -> oem_xval_dense  (+ getmin, cvup / cvlo: R/utils.R:3-26)
    R/big_oem.R:121-543    big.oem()    -> oem_fit_big     (x: ndarray, np.memmap of a big.matrix .bk file, or a
                                                            column-major CUDA tensor)

What the R functions do around .Call and this module reproduces: argument checks and their error messages,
defaults (tol 1e-7, maxit 500, nlambda 100, lambda.min.ratio 1e-4 if n >= p else 0.01, gamma 3, alpha 1, tau 0.5,
irls.tol 1e-3, irls.maxit 100), the group bookkeeping (sorted unique groups, group 0 = unpenalised, the extra
group-0 entry for an explicit intercept column), lambda list normalisation (sorted decreasing, one vector per
penalty), `nzero` per lambda, and for xval.oem lambda.min / lambda.1se / cvup / cvlo / best.model.
Dots in R argument names become underscores.  Results are dicts keyed like the R lists.
"""
import numpy as np

from . import api

PENALTIES = ["elastic.net", "lasso", "ols", "mcp", "scad", "mcp.net", "scad.net", "grp.lasso", "grp.lasso.net",
             "grp.mcp", "grp.scad", "grp.mcp.net", "grp.scad.net", "sparse.grp.lasso"]


def _match_penalty(penalty):
    if penalty is None:
        return ["elastic.net"]          # match.arg(several.ok = FALSE) on the default vector picks the first
    pens = [penalty] if isinstance(penalty, str) else list(penalty)
    for p in pens:
        if p not in PENALTIES:
            raise ValueError(f"'arg' should be one of {PENALTIES}")
    return pens


def _is_sparse(x):
    """A scipy.sparse matrix, or the (i, p, x, dim) slots of a dgCMatrix as a tuple."""
    if isinstance(x, tuple):
        return True
    try:
        import scipy.sparse as sps
    except ImportError:
        return False
    return sps.issparse(x)


def _shape(x):
    if hasattr(x, "shape") and len(x.shape) == 2:
        return int(x.shape[0]), int(x.shape[1])
    raise ValueError("x must have at least two columns")


def _groups(penalty, groups, group_weights, p, explicit_intercept):
    """R/oem.R:282-345 (and the same block in R/big_oem.R:208-264, R/oem_xval.R)."""
    if not any("grp" in pen for pen in penalty):
        return np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0)
    groups = np.asarray(groups).ravel()
    if groups.size != p:
        raise ValueError("If any group penalty is used groups must have same length as number of columns in x")
    unique_groups = np.sort(np.unique(groups))
    has_zero = bool(np.any(unique_groups == 0))
    if group_weights is not None:
        gw = np.asarray(group_weights, dtype=np.float64).ravel().copy()
        if has_zero:
            gw[np.nonzero(unique_groups == 0)[0]] = 0.0
        elif explicit_intercept:
            unique_groups = np.concatenate([[0], unique_groups])
            gw = np.concatenate([[0.0], gw])
        if gw.size != unique_groups.size:
            raise ValueError("group.weights must have same length as the number of groups")
    else:
        gw = np.zeros(0)
        if not has_zero and explicit_intercept:
            unique_groups = np.sort(np.concatenate([[0], unique_groups]))
    if explicit_intercept:
        groups = np.concatenate([[0], groups])
    return groups.astype(np.int32), unique_groups.astype(np.int32), gw


def _lambda_list(lambda_, npen):
    """R/oem.R:366-404."""
    if isinstance(lambda_, (list, tuple)) and len(lambda_) and np.ndim(lambda_[0]) >= 1:
        if len(lambda_) != npen:
            raise ValueError("If list of lambda vectors is provided, it must be the same length as the number of penalties fit")
        n0 = np.asarray(lambda_[0]).size
        out = []
        for lv in lambda_:
            lv = np.asarray(lv, dtype=np.float64).ravel()
            if lv.size < 1:
                raise ValueError("Provided lambda vector must have at least one value")
            if lv.size != n0:
                raise ValueError("All provided lambda vectors must have same length")
            out.append(np.sort(lv)[::-1].copy())
        return out
    lv = np.sort(np.asarray(lambda_ if lambda_ is not None else [], dtype=np.float64).ravel())[::-1].copy()
    return [lv.copy() for _ in range(npen)]


def _common_checks(n, p, y_len, penalty_factor, lambda_min_ratio, nlambda, maxit, irls_maxit, tol, irls_tol):
    if p < 2:
        raise ValueError("x must have at least two columns")
    if y_len != n:
        raise ValueError("x and y lengths do not match")
    pf = np.ones(p) if penalty_factor is None else np.asarray(penalty_factor, dtype=np.float64).ravel()
    if pf.size != p:
        raise ValueError("penalty.factor must have same length as number of columns in x")
    if lambda_min_ratio is None:
        lambda_min_ratio = 0.01 if n < p else 0.0001
    lambda_min_ratio = float(lambda_min_ratio)
    if lambda_min_ratio >= 1 or lambda_min_ratio <= 0:
        raise ValueError("lambda.min.ratio must be between 0 and 1")
    if int(nlambda) <= 0:
        raise ValueError("nlambda must be a positive integer")
    if maxit <= 0 or irls_maxit <= 0:
        raise ValueError("maxit and irls.maxit should be positive")
    if tol < 0 or irls_tol < 0:
        raise ValueError("tol and irls.tol should be nonnegative")
    return pf, lambda_min_ratio


def nonzero_counts(beta):
    """`nzero`: number of non-zero non-intercept coefficients per lambda (predict.oem(type = "nonzero"),
    R/methods.R:48-119 as used at R/oem.R:495-497)."""
    b = np.asarray(beta)
    return np.count_nonzero(b[1:, :] if b.ndim == 2 else b[1:, None], axis=0)


def getmin(lambda_, cvm, cvsd):
    """R/utils.R:3-26 (modified from glmnet)."""
    M = len(cvm)
    lam_min, lam_1se, cv_models = np.zeros(M), np.zeros(M), np.zeros(M)
    for m in range(M):
        lam, c, s = np.asarray(lambda_[m])[:len(cvm[m])], np.asarray(cvm[m]), np.asarray(cvsd[m])
        cvmin = c.min()
        idmin = c <= cvmin
        lam_min[m] = lam[idmin].max()
        cv_models[m] = c[idmin].min()
        first = int(np.nonzero(lam == lam_min[m])[0][0])
        semin = (c + s)[first]
        lam_1se[m] = lam[c < semin].max() if np.any(c < semin) else -np.inf     # max(numeric(0)) = -Inf in R (cvsd == 0)
    mmin = int(np.argmin(cv_models))
    return dict(lambda_min=float(lam_min[mmin]), model_min=mmin + 1, lambda_1se=float(lam_1se[mmin]),
                lambda_min_models=lam_min, lambda_1se_models=lam_1se)


def _decorate(res, penalty, n, p, family, varnames):
    out = dict(res)
    out["lambda"] = out.pop("lambda_")
    out["beta"] = {pen: b for pen, b in zip(penalty, res["beta"])}
    out["nzero"] = [nonzero_counts(b) for b in res["beta"]]
    out.update(nobs=n, nvars=p, penalty=list(penalty), family=family,
               varnames=varnames or [f"V{i + 1}" for i in range(p)], rownames=["(Intercept)"] + (varnames or [f"V{i + 1}" for i in range(p)]))
    return out


def oem(x, y, family="gaussian", penalty=None, weights=(), lambda_=(), nlambda=100, lambda_min_ratio=None, alpha=1.0,
        gamma=3.0, tau=0.5, groups=(), penalty_factor=None, group_weights=None, standardize=True, intercept=True,
        maxit=500, tol=1e-7, irls_maxit=100, irls_tol=1e-3, accelerate=False, ncores=-1, compute_loss=False,
        hessian_type="upper.bound", varnames=None, comm=None):
    """R/oem.R:162-507.  `gamma` may also be one value per penalty (extension)."""
    if family not in ("gaussian", "binomial"):
        raise ValueError("'arg' should be one of 'gaussian', 'binomial'")
    if hessian_type not in ("upper.bound", "full"):
        raise ValueError("'arg' should be one of 'upper.bound', 'full'")
    penalty = _match_penalty(penalty)
    is_sparse = _is_sparse(x)                                  # inherits(x, "sparseMatrix"), R/oem.R:235-241
    n, p = (int(x[3][0]), int(x[3][1])) if isinstance(x, tuple) else _shape(x)
    if len(weights) > 0:
        raise ValueError("weights not implemented yet.")
    ylen = int(y.shape[0]) if hasattr(y, "shape") else len(y)
    pf, lmr = _common_checks(n, p, ylen, penalty_factor, lambda_min_ratio, nlambda, maxit, irls_maxit, tol, irls_tol)
    if family == "binomial" and not hasattr(y, "is_cuda"):
        if np.unique(np.asarray(y)).size > 2:
            raise ValueError("y must be a binary outcome")
    if is_sparse and family != "gaussian" and intercept and not standardize:
        raise NotImplementedError("oem(family = 'binomial') on a sparse x with intercept = TRUE, standardize = FALSE: the reference "
                                  "reads an uninitialised vector there (src/oem_logistic_sparse.h:880); no behaviour to reproduce")
    g, ug, gw = _groups(penalty, groups, group_weights, p,
                        explicit_intercept=(intercept and (family != "gaussian" or is_sparse)))      # R/oem.R:300-337
    lam = _lambda_list(lambda_, len(penalty))
    opts = dict(maxit=int(maxit), tol=float(tol), irls_maxit=int(irls_maxit), irls_tol=float(irls_tol), ncores=int(ncores),
                hessian_type=hessian_type, accelerate=bool(accelerate))
    if is_sparse:                                              # R/oem.R:532-553 (gaussian), 605-625 (binomial)
        fn = api.oem_fit_sparse if family == "gaussian" else api.oem_fit_logistic_sparse
    else:
        fn = api.oem_fit_dense if family == "gaussian" else api.oem_fit_logistic_dense
    res = fn(x, y, family, penalty, [], g, ug, gw, lam, int(nlambda), lmr, float(alpha), gamma, float(tau), pf,
             bool(standardize), bool(intercept), bool(compute_loss), opts, comm=comm)
    return _decorate(res, penalty, n, p, family, varnames)


def big_oem(x, y, family="gaussian", penalty=None, weights=(), lambda_=(), nlambda=100, lambda_min_ratio=None,
            alpha=1.0, gamma=3.0, tau=0.5, groups=(), penalty_factor=None, group_weights=None, standardize=True,
            intercept=True, maxit=500, tol=1e-7, irls_maxit=100, irls_tol=1e-3, compute_loss=False, gigs=4.0,
            hessian_type="full", varnames=None, comm=None):
    """R/big_oem.R:121-543.  `x` plays the role of the big.matrix: an ndarray / np.memmap (see
    oem_b200.bigmatrix.attach for .bk/.desc files) or a column-major CUDA tensor.  Only the gaussian family is
    exists: the reference's own big.oem stops on binomial (R/big_oem.R:159)."""
    if family != "gaussian":
        raise NotImplementedError("binomial case not implemented yet")          # R/big_oem.R:159, same words
    penalty = _match_penalty(penalty)
    n, p = _shape(x)
    if len(weights) > 0:
        raise ValueError("weights not implemented yet.")
    if getattr(x, "dtype", np.dtype("float64")) not in (np.dtype("float64"),) and not hasattr(x, "is_cuda"):
        raise ValueError("big.matrix type must be double")                 # src/oem_big.cpp:57-62
    ylen = int(y.shape[0]) if hasattr(y, "shape") else len(y)
    pf, lmr = _common_checks(n, p, ylen, penalty_factor, lambda_min_ratio, nlambda, maxit, irls_maxit, tol, irls_tol)
    g, ug, gw = _groups(penalty, groups, group_weights, p, explicit_intercept=bool(intercept))
    lam = _lambda_list(lambda_, len(penalty))
    opts = dict(maxit=int(maxit), tol=float(tol), irls_maxit=int(irls_maxit), irls_tol=float(irls_tol), gigs=float(gigs))
    res = api.oem_fit_big(x, y, family, penalty, [], g, ug, gw, lam, int(nlambda), lmr, float(alpha), gamma, float(tau),
                          pf, bool(standardize), bool(intercept), bool(compute_loss), opts, comm=comm)
    return _decorate(res, penalty, n, p, family, varnames)


def oem_xtx(xtx, xty, family="gaussian", penalty=None, lambda_=(), nlambda=100, lambda_min_ratio=None, alpha=1.0,
            gamma=3.0, tau=0.5, groups=(), scale_factor=(), penalty_factor=None, group_weights=None, maxit=500,
            tol=1e-7, irls_maxit=100, irls_tol=1e-3):
    """R/oem_xtx.R:109-455.  xtx, xty must already be divided by n; beta has no intercept row."""
    if family != "gaussian":
        raise ValueError("only the gaussian family is available for oem.xtx")
    penalty = _match_penalty(penalty)
    n, p = _shape(xtx)
    if n != p:
        raise ValueError("xtx must be a square matrix")
    xty = np.asarray(xty, dtype=np.float64).ravel() if not hasattr(xty, "is_cuda") else xty
    # R/oem_xtx.R:225-233: lambda.min.ratio defaults to 1e-4 (n is unknown here)
    pf, lmr = _common_checks(p + 1, p, p + 1, penalty_factor, 1e-4 if lambda_min_ratio is None else lambda_min_ratio,
                             nlambda, maxit, irls_maxit, tol, irls_tol)
    sf = np.asarray(scale_factor, dtype=np.float64).ravel()
    if sf.size and sf.size != p:
        raise ValueError("scale.factor must be same length as xty (nvars)")
    g, ug, gw = _groups(penalty, groups, group_weights, p, explicit_intercept=False)
    lam = _lambda_list(lambda_, len(penalty))
    res = api.oem_xtx(xtx, xty, family, penalty, g, ug, gw, lam, int(nlambda), lmr, float(alpha), gamma, float(tau), sf, pf,
                      dict(maxit=int(maxit), tol=float(tol), irls_maxit=int(irls_maxit), irls_tol=float(irls_tol)))
    out = dict(res)
    out["lambda"] = out.pop("lambda_")
    out["beta"] = {pen: b for pen, b in zip(penalty, res["beta"])}
    out["nzero"] = [np.count_nonzero(b, axis=0) for b in res["beta"]]
    out.update(nvars=p, penalty=list(penalty), family=family)
    return out


def xval_oem(x, y, nfolds=10, foldid=None, type_measure=None, ncores=-1, family="gaussian", penalty=None, weights=(),
             lambda_=(), nlambda=100, lambda_min_ratio=None, alpha=1.0, gamma=3.0, tau=0.5, groups=(),
             penalty_factor=None, group_weights=None, standardize=True, intercept=True, maxit=500, tol=1e-7,
             irls_maxit=100, irls_tol=1e-3, compute_loss=False, varnames=None, seed=None, comm=None,
             hessian_type="upper.bound"):
    """R/oem_xval.R:107-460: fit + fast cross-validation in one call; adds lambda.min / lambda.1se / cvup / cvlo.
    type.measure: gaussian mse (default) | deviance | mae; binomial deviance (default) | class | mse | mae.
    family = "binomial" (which the reference's xval.oem refuses, R/oem_xval.R:160-163) runs oem_xval_logistic_dense:
    the full-data logistic fit of oem() plus one fit per fold at its lambdas, scored with cv.oem's binomial measures
    over all rows; `auc` needs per-fold ranks and stays with cv_oem()."""
    if family not in ("gaussian", "binomial"):
        raise ValueError("'arg' should be one of 'gaussian', 'binomial'")
    binomial = family == "binomial"
    if type_measure is None:
        type_measure = "deviance" if binomial else "mse"
    if binomial:
        if type_measure == "auc":
            raise ValueError("type.measure = 'auc' needs per-fold ranks: use cv_oem(family='binomial', type_measure='auc')")
        if type_measure not in ("deviance", "class", "mse", "mae"):
            raise ValueError("type.measure must be 'deviance', 'class', 'mse' or 'mae' for the binomial family")
        if hessian_type != "upper.bound":
            raise ValueError("xval_oem(family='binomial') supports hessian_type='upper.bound' only; use cv_oem for 'full'")
        if len(weights) > 0:
            raise ValueError("weights not implemented yet.")                       # oem() itself rejects them (R/oem.R:244)
        if not hasattr(y, "is_cuda") and np.unique(np.asarray(y)).size > 2:
            raise ValueError("y must be a binary outcome")
    elif type_measure not in ("mse", "deviance", "mae"):
        raise ValueError("type.measure must be 'mse', 'deviance' or 'mae' for the gaussian family")
    penalty = _match_penalty(penalty)
    n, p = _shape(x)
    weights = np.asarray(weights, dtype=np.float64).ravel() if len(weights) > 0 else np.zeros(0)
    if weights.size and weights.size != n:
        raise ValueError("length of weights not same as number of observations in x")      # R/oem_xval.R:216-221
    if foldid is None:
        rng = np.random.default_rng(seed)
        foldid = rng.permutation(np.resize(np.arange(1, int(nfolds) + 1), n))     # sample(rep(seq(nfolds), length = n))
    else:
        foldid = np.asarray(foldid).ravel()
        nfolds = int(foldid.max())
    if nfolds < 3:
        raise ValueError("nfolds must be bigger than 3; nfolds=10 recommended")
    ylen = int(y.shape[0]) if hasattr(y, "shape") else len(y)
    pf, lmr = _common_checks(n, p, ylen, penalty_factor, lambda_min_ratio, nlambda, maxit, irls_maxit, tol, irls_tol)
    g, ug, gw = _groups(penalty, groups, group_weights, p, explicit_intercept=bool(intercept))
    lam = _lambda_list(lambda_, len(penalty))
    opts = dict(maxit=int(maxit), tol=float(tol), irls_maxit=int(irls_maxit), irls_tol=float(irls_tol), ncores=int(ncores))
    if binomial:
        res = api.oem_xval_logistic_dense(x, y, family, penalty, [], g, ug, gw, lam, int(nlambda), lmr, float(alpha), gamma,
                                          float(tau), pf, bool(standardize), bool(intercept), int(nfolds),
                                          foldid.astype(np.int32), bool(compute_loss), type_measure, opts, comm=comm)
    else:
        res = api.oem_xval_dense(x, y, family, penalty, weights, g, ug, gw, lam, int(nlambda), lmr, float(alpha), gamma,
                                 float(tau), pf, bool(standardize), bool(intercept), int(nfolds), foldid.astype(np.int32),
                                 bool(compute_loss), "mse" if type_measure == "deviance" else type_measure, opts, comm=comm)
    out = _decorate(res, penalty, n, p, family, varnames)
    out.update(getmin(out["lambda"], out["cvm"], out["cvsd"]))
    out["cvup"] = [m + s for m, s in zip(out["cvm"], out["cvsd"])]
    out["cvlo"] = [m - s for m, s in zip(out["cvm"], out["cvsd"])]
    out["best_model"] = penalty[out["model_min"] - 1]
    out["foldid"] = foldid
    return out


def _take_rows(x, keep):
    """x[keep, , drop = FALSE] for a numpy / scipy.sparse matrix or a (column-major) CUDA tensor."""
    if hasattr(x, "is_cuda"):
        import torch
        idx = torch.from_numpy(np.nonzero(keep)[0]).to(x.device)
        if x.dim() == 1:
            return x.index_select(0, idx)
        return x.t().index_select(1, idx).contiguous().t()          # stays column-major
    if _is_sparse(x):
        return x.tocsr()[np.nonzero(keep)[0]].tocsc()
    x = np.asarray(x)
    return np.asfortranarray(x[keep]) if x.ndim == 2 else x[keep]


def _cvcompute(mat, weights, foldid, nlams):
    """R/utils.R:126-144 (after glmnet): weighted mean of the raw losses inside every fold."""
    nfolds = int(foldid.max())
    outmat = np.full((nfolds, mat.shape[1]), np.nan)
    good = np.zeros((nfolds, mat.shape[1]))
    mat = np.where(np.isinf(mat), np.nan, mat)
    wisum = np.zeros(nfolds)
    for i in range(nfolds):
        w = foldid == i + 1
        wi = weights[w]
        wisum[i] = wi.sum()
        mi = mat[w]
        ok = ~np.isnan(mi)
        with np.errstate(invalid="ignore", divide="ignore"):
            outmat[i] = np.where(ok, mi * wi[:, None], 0.0).sum(0) / np.where(ok, wi[:, None], 0.0).sum(0)
        good[i, :int(nlams[i])] = 1
    return outmat, wisum, good.sum(0)


def cv_oem(x, y, penalty=None, weights=(), lambda_=(), type_measure="default", nfolds=10, foldid=None, grouped=True,
           keep=False, seed=None, **oem_args):
    """cv.oem (R/cv_oem.R:58-253): K refits of oem() on the training folds (each with its own lambda sequence), held-out
    predictions interpolated onto the full fit's lambdas (never extrapolated below a fold's smallest lambda), glmnet-style
    fold-grouped cvm / cvsd, then getmin().  Every fit and every prediction runs on the device through oem() / predict();
    xval.oem() computes the same thing from one pass over X and is the fast route (R/oem_xval.R).
    type.measure: gaussian mse | deviance | mae; binomial deviance | class | auc | mse | mae."""
    family = oem_args.get("family", "gaussian")
    if len(lambda_) and all(np.ndim(l) == 0 for l in lambda_) and len(lambda_) < 2:
        raise ValueError("Need more than one value of lambda for cv.oem")
    n, _ = (int(x[3][0]), int(x[3][1])) if isinstance(x, tuple) else _shape(x)
    if len(weights) > 0:
        raise ValueError("weights not implemented yet.")             # oem() itself rejects them (R/oem.R:244)
    fit = oem(x, y, penalty=penalty, lambda_=lambda_, **oem_args)
    pens = fit["penalty"]
    nz = fit["nzero"]
    if foldid is None:
        rng = np.random.default_rng(seed)
        foldid = rng.permutation(np.resize(np.arange(1, int(nfolds) + 1), n))      # sample(rep(seq(nfolds), length = N))
    else:
        foldid = np.asarray(foldid).ravel()
        nfolds = int(foldid.max())
    if nfolds < 3:
        raise ValueError("nfolds must be bigger than 3; nfolds=10 recommended")
    yh = y.cpu().numpy() if hasattr(y, "is_cuda") else np.asarray(y, dtype=np.float64).ravel()
    outlist = []
    for i in range(1, nfolds + 1):
        tr = foldid != i
        outlist.append(oem(_take_rows(x, tr), _take_rows(y, tr), penalty=penalty, lambda_=lambda_, **oem_args))
    lam = fit["lambda"]
    nmodels = len(pens)
    which_lam = []
    for m in range(nmodels):
        mlami = max(float(np.min(o["lambda"][m])) for o in outlist)                 # do not extrapolate smaller lambdas
        which_lam.append(np.asarray(lam[m]) >= mlami)
    nlam0 = len(lam[0])
    predlist = [np.full((n, nlam0), np.nan) for _ in range(nmodels)]
    nlams = np.zeros(nfolds)
    for i in range(1, nfolds + 1):
        w = foldid == i
        xt = _take_rows(x, w)
        for m in range(nmodels):
            s_use = np.asarray(lam[m])[which_lam[m]]
            pr = predict(outlist[i - 1], newx=xt, s=s_use, which_model=m + 1,
                         type="response" if family == "binomial" else "link")
            predlist[m][w, :s_use.size] = pr
            nlams[i - 1] = s_use.size
    if family == "gaussian":
        tm = "mse" if type_measure in ("default", "deviance") else type_measure
        if tm not in ("mse", "mae"):
            raise ValueError("Only 'mse', 'deviance' or 'mae' available for Gaussian models")
        name = "Mean-Squared Error" if tm == "mse" else "Mean Absolute Error"
        cvraw = [(yh[:, None] - p_) ** 2 if tm == "mse" else np.abs(yh[:, None] - p_) for p_ in predlist]
    else:
        tm = "deviance" if type_measure == "default" else type_measure
        if tm not in ("mse", "mae", "deviance", "class", "auc"):
            raise ValueError("Only 'deviance', 'class', 'auc', 'mse' or 'mae' available for binomial models")
        if tm == "auc" and n / nfolds < 10:
            tm = "deviance"                 # "Too few (< 10) observations per fold for type.measure='auc'" (R/cv_oem.R:276-281)
        name = {"mse": "Mean-Squared Error", "mae": "Mean Absolute Error", "deviance": "Binomial Deviance",
                "class": "Misclassification Error", "auc": "AUC"}[tm]
        y1 = (yh == np.max(yh)).astype(np.float64)                                   # second factor level
        y0 = 1.0 - y1
        cvraw = []
        for p_ in predlist:                                                          # R/cv_oem.R:288-330
            if tm == "auc":
                # one AUC per (fold, lambda), R/utils.R:89-124 with unit weights = the rank-sum statistic; tied scores get
                # half credit here (the reference breaks ties with runif(), R/utils.R:103-104)
                from scipy.stats import rankdata
                raw = np.full((nfolds, nlam0), np.nan)
                for i in range(nfolds):
                    w = foldid == i + 1
                    pos = y1[w] == 1
                    n1, n0 = int(pos.sum()), int((~pos).sum())
                    for j in range(int(nlams[i])):
                        r = rankdata(p_[w, j])
                        raw[i, j] = (r[pos].sum() - n1 * (n1 + 1) / 2.0) / (n1 * n0) if n1 and n0 else np.nan
                cvraw.append(raw)
            elif tm == "mse":
                cvraw.append((y0[:, None] - (1 - p_)) ** 2 + (y1[:, None] - p_) ** 2)
            elif tm == "mae":
                cvraw.append(np.abs(y0[:, None] - (1 - p_)) + np.abs(y1[:, None] - p_))
            elif tm == "deviance":
                pm = np.minimum(np.maximum(p_, 1e-5), 1 - 1e-5)
                cvraw.append(-2.0 * (y0[:, None] * np.log(1 - pm) + y1[:, None] * np.log(pm)))
            else:
                cvraw.append(y0[:, None] * (p_ > 0.5) + y1[:, None] * (p_ <= 0.5))
    wts = np.ones(n)
    N = [n - np.isnan(p_).sum(0) for p_ in predlist]
    if n / nfolds < 3 and grouped:
        grouped = False
    cvm, cvsd = [], []
    auc = family != "gaussian" and tm == "auc"
    for m in range(nmodels):
        raw, w_m, N_m = cvraw[m], wts, N[m]
        if auc:                                               # already one row per fold; weights = fold sizes
            w_m = np.array([float((foldid == i + 1).sum()) for i in range(nfolds)])
            good = np.zeros((nfolds, nlam0))
            for i in range(nfolds):
                good[i, :int(nlams[i])] = 1
            N_m = good.sum(0)
        elif grouped:
            raw, w_m, N_m = _cvcompute(raw, wts, foldid, nlams)
        ok = ~np.isnan(raw)
        with np.errstate(invalid="ignore", divide="ignore"):
            wsum = np.where(ok, w_m[:, None], 0.0).sum(0)
            mean = np.where(ok, raw * w_m[:, None], 0.0).sum(0) / wsum
            var = np.where(ok, (raw - mean[None, :]) ** 2 * w_m[:, None], 0.0).sum(0) / wsum
            cvm.append(mean)
            cvsd.append(np.sqrt(var / (N_m - 1)))
    nas = np.zeros(nlam0, dtype=bool)
    for m in range(nmodels):
        nas |= np.isnan(cvsd[m])
    lam_out = [np.asarray(l)[~nas] for l in lam]
    cvm = [c[~nas] for c in cvm]
    cvsd = [c[~nas] for c in cvsd]
    out = dict(lambda_=lam_out, cvm=cvm, cvsd=cvsd, cvup=[a + b for a, b in zip(cvm, cvsd)],
               cvlo=[a - b for a, b in zip(cvm, cvsd)], nzero=[z[~nas] for z in nz], name=name, oem_fit=fit,
               penalty=pens, foldid=foldid)
    out["lambda"] = out.pop("lambda_")
    if keep:
        out["fit_preval"] = predlist
    out.update(getmin(lam_out, [-c for c in cvm], cvsd) if auc else getmin(lam_out, cvm, cvsd))      # R/cv_oem.R:246-247
    out["best_model"] = pens[out["model_min"] - 1]
    return out


# ------------------------------------------------------------------------------------------
# S3 methods the front-ends' users call next (R/methods.R): predict / logLik on the fitted object
# ------------------------------------------------------------------------------------------
def lambda_interp(lambda_, s):
    """R/utils.R:64-87 (copied there from glmnet): linear interpolation weights of `s` on the fitted lambda grid.
    Returns 0-based left / right column indices and the weight of the left column."""
    lam = np.asarray(lambda_, dtype=np.float64)
    s = np.atleast_1d(np.asarray(s, dtype=np.float64)).copy()
    if lam.size == 1:
        z = np.zeros(s.size, dtype=np.int64)
        return z, z.copy(), np.ones(s.size)
    s = np.clip(s, lam.min(), lam.max())
    k = lam.size
    sfrac = (lam[0] - s) / (lam[0] - lam[k - 1])
    t = (lam[0] - lam) / (lam[0] - lam[k - 1])
    coord = np.interp(sfrac, t, np.arange(1, k + 1, dtype=np.float64))       # approx(lambda, seq(lambda), sfrac)$y
    left, right = np.floor(coord).astype(np.int64), np.ceil(coord).astype(np.int64)
    with np.errstate(divide="ignore", invalid="ignore"):
        frac = (sfrac - t[right - 1]) / (t[left - 1] - t[right - 1])
    frac[left == right] = 1.0
    return left - 1, right - 1, frac


def _which_model(fit, which_model):
    names = list(fit["beta"].keys())
    if isinstance(which_model, str):
        if which_model not in names:
            raise ValueError(f"Model {which_model} specified, but {which_model} not computed.")
        return names.index(which_model)
    if which_model > len(names):
        raise ValueError(f"Model {which_model} specified, but only {len(names)} were computed.")
    return int(which_model) - 1


def predict(fit, newx=None, s=None, which_model=1, type="link", opts=None):
    """predict.oem / predict.oemfit_binomial (R/methods.R:48-119, 346-366).  `type` in link / response / coefficients /
    nonzero / class; `s` interpolates the coefficient path at new lambda values (lambda.interp).  The matrix product
    newx %*% beta runs on the device (api.predict_matrix -> oemb200_predict)."""
    if type not in ("link", "response", "coefficients", "nonzero", "class"):
        raise ValueError("'arg' should be one of 'link', 'response', 'coefficients', 'nonzero', 'class'")
    if "oem_fit" in fit or "cvm" in fit:
        # predict.cv.oem / predict.xval.oem (R/methods.R:674-714, 765-806): s defaults to lambda.min, "best.model" allowed
        if s is None or (isinstance(s, str) and s == "lambda.min"):
            s = fit["lambda_min"]
        elif isinstance(s, str):
            if s != "lambda.1se":
                raise ValueError("Invalid form for s")
            s = fit["lambda_1se"]
        if isinstance(which_model, str) and which_model == "best.model":
            which_model = fit["model_min"]
        if "oem_fit" in fit:
            return predict(fit["oem_fit"], newx=newx, s=s, which_model=which_model, type=type, opts=opts)
    m = _which_model(fit, which_model)
    if newx is None and type not in ("coefficients", "nonzero"):
        raise ValueError("A value for 'newx' must be supplied")
    nbeta = np.asarray(list(fit["beta"].values())[m], dtype=np.float64)
    if nbeta.ndim == 1:
        nbeta = nbeta[:, None]
    if s is not None:
        left, right, frac = lambda_interp(fit["lambda"][m][:nbeta.shape[1]], s)
        nbeta = nbeta[:, left] * frac[None, :] + nbeta[:, right] * (1.0 - frac)[None, :]
    if type == "coefficients":
        return nbeta
    if type == "nonzero":
        nz = np.abs(nbeta) > 0
        nz[0, :] = False                                      # "rem intercept" (R/methods.R:95)
        return [np.nonzero(nz[:, j])[0] + 1 if nz[:, j].any() else None for j in range(nz.shape[1])]   # 1-based rows
    binomial = fit.get("family") == "binomial"
    pred = api.predict_matrix(newx, nbeta, response=(binomial and type == "response"), opts=opts)
    if type == "class":
        if not binomial:
            raise ValueError("type = 'class' is only available for the binomial family")
        return np.where(pred > 0, 2, 1)                        # index into object$classnames (R/methods.R:359-364)
    return pred


def logLik(fit, which_model=1):
    """logLik.oem (R/methods.R:431-478, after ncvreg): needs compute_loss=True."""
    if "oem_fit" in fit:                                       # logLik.cv.oem works on the full-data fit
        return logLik(fit["oem_fit"], which_model)
    m = _which_model(fit, which_model)
    loss = np.asarray(fit["loss"][m], dtype=np.float64)
    if np.all(loss == 1e99):
        raise ValueError("oem object needed compute.loss set to TRUE. logLik not returned")
    n = float(fit["nobs"])
    if fit["family"] == "gaussian":
        return -0.5 * n * (np.log(2 * np.pi) - np.log(n) + np.log(loss)) - 0.5 * n
    if fit["family"] == "binomial":
        return -1.0 * loss
    raise ValueError(f"family {fit['family']} not available")
