"""oem_xval_big: oem_xval_dense on an X read in row chunks of opts["gigs"] GB, twice (the fold Grams, then the scores).
One chunk is the resident entry bit for bit; many chunks (ragged last chunk, a chunk without rows of some fold) agree
with the oracle and with the resident entry up to summation order; every source of X gives the same bits; device memory
does not grow with n.  The tests without the gpu mark check the interface on the CPU."""
import numpy as np
import pytest

from cases import DEFAULT_OPTS, args_xy, assert_same_fit, gaussian_problem

EINVAL, ENODEVICE, EUNSUPPORTED = 1, 2, 4
ALIGN = 72          # rows: the fold-segment alignment, and the unit big_chunk_rows rounds a chunk to


def xval_args(X, y, penalty, foldid, nfolds, weights=None, type_measure="mse", compute_loss=False, gigs=None, **kw):
    opts = dict(DEFAULT_OPTS)
    opts.update(kw.pop("opts", {}))
    if gigs is not None:
        opts["gigs"] = gigs
    a = args_xy(X, y, "gaussian", penalty, compute_loss=compute_loss, opts=opts, **kw)
    if weights is not None:
        a[4] = weights
    return a[:17] + [nfolds, np.asarray(foldid, dtype=np.int32), compute_loss, type_measure, a[18]]


def gigs_for(rows, p):
    """opts["gigs"] that makes chunks of exactly `rows` rows (a multiple of ALIGN) for p columns."""
    assert rows % ALIGN == 0
    return (rows + 0.5) * 8.0 * p / 1e9


def fold_ids(seed, n, nfolds, rows=None, hole=None):
    """Balanced random fold ids; with hole = (chunk, fold) no row of that chunk (chunks of `rows` rows) is in that fold."""
    rng = np.random.default_rng(seed)
    f = 1 + rng.permutation(n) % nfolds
    if hole is not None:
        c, k = hole
        seg = f[c * rows:(c + 1) * rows]
        seg[seg == k] = 1 + (k % nfolds)
    return f


OUTPUTS = ("beta", "lambda_", "niter", "loss", "cvm", "cvsd")


def assert_bit_identical(a, b):
    for key in OUTPUTS:
        for u, v in zip(a[key], b[key]):
            assert np.array_equal(np.asarray(u), np.asarray(v)), key
    assert a["d"] == b["d"]


# ---------------------------------------------------------------- CPU: the interface
def test_symbol_is_exported(lib):
    assert "oemb200_xval_big" in lib.EXPORTS
    assert hasattr(lib.load(), "oemb200_xval_big")


def small_case():
    X, y = gaussian_problem(3, 300, 6)
    return X, y, xval_args(X, y, ["lasso"], fold_ids(3, 300, 3), 3)


def test_no_device(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the no-device behaviour is checked on the CPU box")
    _, _, a = small_case()
    with pytest.raises(lib.OemB200Error) as ei:
        lib.oem_xval_big(*a)
    assert ei.value.code == ENODEVICE


def test_refusals_precede_device_use(lib):
    from oem_b200 import api
    X, y, a = small_case()
    b = list(a)
    b[1] = (y > np.median(y)).astype(float)
    b[2] = "binomial"
    with pytest.raises(lib.OemB200Error) as ei:
        lib.oem_xval_big(*b)
    assert ei.value.code == EUNSUPPORTED and "IRLS" in str(ei.value)
    o = api.make_opts(a[-1])
    o.world, o.rank = 2, 0
    b = list(a)
    b[-1] = o
    with pytest.raises(lib.OemB200Error) as ei:
        lib.oem_xval_big(*b)
    assert ei.value.code == EUNSUPPORTED and "one GPU" in str(ei.value)


def test_frontend_refuses_binomial_with_gigs():
    from oem_b200 import frontend
    X, y = gaussian_problem(3, 300, 6)
    with pytest.raises(ValueError, match="gaussian family only"):
        frontend.xval_oem(X, (y > 0).astype(float), family="binomial", gigs=1.0)


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("standardize,intercept", [(False, False), (True, False), (False, True), (True, True)])
def test_one_chunk_is_the_resident_entry(lib, standardize, intercept):
    X, y = gaussian_problem(41, 3001, 30, coef="vignette", noise=2.0)
    foldid = fold_ids(41, 3001, 5)
    w = np.random.default_rng(41).uniform(0.25, 3.0, size=3001)
    for weights in (None, w):
        for measure in ("mse", "mae"):
            kw = dict(nlambda=20, standardize=standardize, intercept=intercept, type_measure=measure, compute_loss=True)
            ref = lib.oem_xval_dense(*xval_args(X, y, ["lasso", "mcp"], foldid, 5, weights=weights, **kw))
            got = lib.oem_xval_big(*xval_args(X, y, ["lasso", "mcp"], foldid, 5, weights=weights, gigs=4.0, **kw))
            assert_bit_identical(got, ref)
            assert got["stats"]["gram_launches"] == 1 and got["stats"]["data_passes"] == 2


MANY = dict(n=6000, p=50, rows=720)      # 9 chunks, the last one 240 rows; chunk 2 has no row of fold 3


@pytest.mark.gpu
@pytest.mark.parametrize("weighted,measure,nfolds", [(False, "mse", 5), (True, "mae", 5), (False, "mse", 70)])
def test_many_chunks(lib, oracle, weighted, measure, nfolds):
    n, p, rows = MANY["n"], MANY["p"], MANY["rows"]
    X, y = gaussian_problem(43, n, p, coef="vignette", noise=3.0)
    foldid = fold_ids(43, n, nfolds, rows=rows, hole=(2, 3))
    assert not np.any(foldid[2 * rows:3 * rows] == 3)
    w = np.random.default_rng(43).uniform(0.25, 3.0, size=n) if weighted else None
    g = np.repeat(np.arange(1, 11), 5)
    kw = dict(nlambda=25, type_measure=measure, compute_loss=True, groups=np.concatenate([[0], g]),
              unique_groups=np.arange(0, 11), opts=dict(tol=1e-10))
    pen = ["lasso", "grp.lasso", "mcp"]
    got = lib.oem_xval_big(*xval_args(X, y, pen, foldid, nfolds, weights=w, gigs=gigs_for(rows, p), **kw))
    assert got["stats"]["gram_launches"] == 9
    ref = oracle.oem_xval_dense(*xval_args(X, y, pen, foldid, nfolds, weights=w, **kw))
    assert_same_fit(got, ref, tol=1e-8)
    for pp in range(len(pen)):
        assert np.allclose(got["cvm"][pp], ref["cvm"][pp], rtol=1e-9, atol=0)
        assert np.allclose(got["cvsd"][pp], ref["cvsd"][pp], rtol=1e-9, atol=0)
        assert np.allclose(got["loss"][pp], ref["loss"][pp], rtol=1e-9)
    res = lib.oem_xval_dense(*xval_args(X, y, pen, foldid, nfolds, weights=w, **kw))
    for pp in range(len(pen)):
        assert np.max(np.abs(got["beta"][pp] - res["beta"][pp])) <= 1e-10


@pytest.mark.gpu
def test_sources_agree_bit_for_bit(lib, tmp_path):
    import torch
    from oem_b200 import bigmatrix
    n, p, rows = MANY["n"], MANY["p"], MANY["rows"]
    X, y = gaussian_problem(47, n, p, coef="vignette", noise=3.0)
    foldid = fold_ids(47, n, 5, rows=rows, hole=(2, 3))
    kw = dict(nlambda=20, compute_loss=True, gigs=gigs_for(rows, p))
    pinned = torch.empty((p, n), dtype=torch.float64).pin_memory()
    pinned.copy_(torch.from_numpy(np.ascontiguousarray(X.T)))
    xp = pinned.t().numpy()
    assert xp.flags.f_contiguous and np.array_equal(xp, X)
    bigmatrix.write(X, str(tmp_path / "x.bk"), str(tmp_path / "x.desc"))
    xm = bigmatrix.attach(str(tmp_path / "x.desc"))
    xd = torch.from_numpy(np.ascontiguousarray(X.T)).cuda().t()
    dm = lib.DeviceMatrix(X)
    base = lib.oem_xval_big(*xval_args(X, y, ["lasso", "mcp"], foldid, 5, **kw))
    assert base["stats"]["gram_launches"] == 9
    for src in (X, xp, xm, xd, dm):
        assert_bit_identical(lib.oem_xval_big(*xval_args(src, y, ["lasso", "mcp"], foldid, 5, **kw)), base)
    # y and foldid on the device too
    a = xval_args(xd, torch.from_numpy(y).cuda(), ["lasso", "mcp"], foldid, 5, **kw)
    a[18] = torch.from_numpy(foldid.astype(np.int32)).cuda()
    assert_bit_identical(lib.oem_xval_big(*a), base)
    dm.close()


@pytest.mark.gpu
def test_counters(lib):
    n, p = 120 * ALIGN, 40
    X, y = gaussian_problem(53, n, p)
    foldid = fold_ids(53, n, 4)
    w = np.random.default_rng(53).uniform(0.5, 2.0, size=n)
    syncs = {}
    for chunks in (4, 12):
        for weights in (None, w):
            st = lib.oem_xval_big(*xval_args(X, y, ["lasso"], foldid, 4, weights=weights, nlambda=10,
                                             gigs=gigs_for(n // chunks, p)))["stats"]
            assert st["gram_launches"] == chunks and st["data_passes"] == 2
            vec = 2 * 8 * n * (2 if weights is not None else 1)            # y (and weights) once per pass
            assert st["h2d_bytes"] == 2 * 8 * n * p + vec + 3 * 4 * n      # foldid: counted once, then once per pass
            syncs[chunks, weights is None] = st["host_syncs"]
    assert syncs[4, True] == syncs[12, True] and syncs[4, False] == syncs[12, False]


FOOTPRINT = r"""
import json, sys
import numpy as np
import torch
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import oem_b200
from test_gpu_xval_big import ALIGN, fold_ids, gigs_for, xval_args
from cases import gaussian_problem
L = oem_b200.load()
p, rows = 200, 40 * ALIGN
out = []
for n in (24 * rows, 96 * rows):
    X, y = gaussian_problem(59, n, p)
    a = xval_args(X, y, ["lasso"], fold_ids(59, n, 5), 5, nlambda=10, gigs=gigs_for(rows, p))
    oem_b200.oem_xval_big(*a)                  # loads the kernels
    L.oemb200_release_cache()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    oem_b200.oem_xval_big(*a)
    free1 = torch.cuda.mem_get_info()[0]
    oem_b200.oem_xval_big(*a)
    free2 = torch.cuda.mem_get_info()[0]
    L.oemb200_release_cache()
    out.append(dict(n=n, held=free0 - free1, again=free1 - free2))
print(json.dumps(out))
"""


@pytest.mark.gpu
def test_device_memory_does_not_grow_with_n(lib):
    """The device memory the library holds after a call (its cache keeps every block the call allocated, so this is
    the call's high-water mark) is the same at n and 4n for one chunk size.  Measured as the drop of the driver's free
    memory in a fresh process: in a process that has freed device memory before, the driver can serve new blocks from
    memory it still holds, which the free count does not show."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", FOOTPRINT, root], capture_output=True, text=True, cwd=root)
    assert r.returncode == 0, r.stderr[-3000:]
    m1, m4 = json.loads(r.stdout.strip().splitlines()[-1])
    # the same call again allocates nothing: every block of the first call was kept and reused
    assert m1["again"] == 0 and m4["again"] == 0, (m1, m4)
    # p = 200, chunks of 2880 rows: two 4.6 MB staging buffers and a 5.2 MB fold-sorted block at least
    assert m1["held"] >= 14 << 20, m1
    # X is 111 MB at n and 442 MB at 4n: a footprint that grew with n would show; 4 MiB = two driver pages
    assert abs(m4["held"] - m1["held"]) <= 4 << 20, (m1, m4)


@pytest.mark.gpu
def test_frontend_streams_a_bigmatrix(lib, tmp_path):
    from oem_b200 import bigmatrix, frontend
    n, p = 5000, 40
    X, y = gaussian_problem(61, n, p, coef="vignette", noise=2.0)
    bigmatrix.write(X, str(tmp_path / "x.bk"), str(tmp_path / "x.desc"))
    big = bigmatrix.attach(str(tmp_path / "x.desc"))
    pen = ["lasso", "mcp"]
    ref = frontend.xval_oem(X, y, nfolds=5, penalty=pen, nlambda=30, seed=7, tol=1e-10)
    got = frontend.xval_oem(big, y, nfolds=5, penalty=pen, nlambda=30, seed=7, tol=1e-10, gigs=gigs_for(8 * ALIGN, p))
    assert got["stats"]["gram_launches"] == 9
    # the lambda grid starts at max|X'y| / n, a sum over the rows in another order: equal to the last bits
    assert np.isclose(got["lambda_min"], ref["lambda_min"], rtol=1e-12, atol=0)
    assert np.isclose(got["lambda_1se"], ref["lambda_1se"], rtol=1e-12, atol=0)
    assert got["best_model"] == ref["best_model"]
    for a, b in zip(got["cvm"], ref["cvm"]):
        assert np.allclose(a, b, rtol=1e-9, atol=0)
