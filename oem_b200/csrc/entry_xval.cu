// entry_xval.cu -- host driver of oem_xval_dense (src/oem_xval_dense.cpp:31-477, solver
// src/oem_xval_dense.h) on the sm_100a kernels.
//
//   1. rows are bucketed by fold (stable counting sort on the host, one gather kernel on the device) so that
//      every fold is a contiguous, 72-row aligned, zero-padded segment of a fold-sorted copy of X;
//   2. ONE Gram launch forms all per-fold Grams G_k as row segments (XtX_xval / XtX_xval_int,
//      oem_xval_dense.h:358-484); column sums / X'y / sum x^2 per fold come from the column-sweep kernel;
//      a row-sharded run all-reduces the whole bundle once;
//   3. assemble_aug builds the full-data and the nfolds leave-one-fold-out systems
//      (compute_/update_XtX_d_update_A, oem_xval_dense.h:667-853);
//   4. ONE path-kernel launch runs all (nfolds+1) x P chains, one CTA team per Gram, each with its own
//      Lanczos eigenvalue (the fold x penalty x lambda loop of oem_xval_dense.cpp:214-340);
//   5. the CV-scoring pass (oem_xval_dense.cpp:345-464) is a fold-segmented FP64 DMMA GEMM with a fused
//      (y - pred)^2 moment epilogue (cvscore.cu).
// Steps 2 and 5 work on one fold-sorted block of rows at a time (xval_bundle_chunk, xval_score_chunk) and accumulate;
// a resident X is one block, and fit_xval_big streams an X that never fits on the device through the same steps.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include "host_common.h"

namespace oemb200 {

// per-fold bundle scaled for the logistic upper-bound Hessian: G_k, the column sums of stats row 0 and the corner
__global__ void xval_hess_scale_kernel(double *G, size_t ng, double *stats, int F, int p, double *corner, double f) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ng) G[i] *= f;
    if (i < (size_t)F * p) stats[(i / p) * 3 * p + i % p] *= f;
    if (i < (size_t)F) corner[i] *= f;
}

namespace {

// The per-fold sums of step 2: bundle = [G F*p*p | stats F*3p | ysum F*2 | nobs F | corner F], one all-reduce.
// unweighted: G_k = X_k'X_k, stats = (colsums, X_k'y, sum x^2), ysum = sum y, corner = n_k.
// weighted:   G_k = X_k'W X_k, stats = (sum w x, X_k'(y*w), UNWEIGHTED sum x^2), ysum = sum y*w, corner = sum w;
//             nobs stays the row count (oem_xval_dense.h:528-545, 596-624).
struct XvalBundle {
    const int F, p;
    const bool weighted;
    const size_t nb;
    DBuf<double> buf, wsum2;             // wsum2 (weighted): [sum w, sum w^2] per fold
    double *G, *stats, *ysum, *nobs, *corner;
    std::vector<char> seen;              // the fold had rows in an earlier chunk: its sweeps accumulate
    XvalBundle(Ctx &cx, int F_, int p_, bool w)
        : F(F_), p(p_), weighted(w), nb((size_t)F_ * p_ * p_ + (size_t)F_ * 3 * p_ + (size_t)F_ * 2 + 2 * (size_t)F_), buf(nb),
          seen(F_, 0) {
        G = buf.p;
        stats = G + (size_t)F * p * p;
        ysum = stats + (size_t)F * 3 * p;
        nobs = ysum + (size_t)F * 2;
        corner = nobs + F;
        if (weighted) {
            wsum2.alloc(2 * (size_t)F);
            wsum2.zero(cx.stream);
        }
    }
};

// Rows [0, nr) of X (column-major, ld ldx), y and w (may be NULL) into fold-sorted order through dest / order: fold k
// becomes sorted rows [off[k], off[k] + cnt[k]) of Xs (ld lds), zero-padded to off[k + 1], and rows off[F]..npad are
// zero.  ys / ws / yws (= y * w) are zeroed first: only the (< 72) padding rows of each segment need zeros, the gather
// writes every other row.
void xval_gather(Ctx &cx, const double *X, int64_t nr, int p, int64_t ldx, const double *y, const double *w, const int *dest,
                 const int *order, const std::vector<int64_t> &cnt, const std::vector<int64_t> &off, int64_t npad, double *Xs,
                 int64_t lds, DBuf<double> &ys, DBuf<double> &ws, DBuf<double> &yws) {
    const int F = (int)cnt.size();
    ys.zero(cx.stream);
    ws.zero(cx.stream);
    yws.zero(cx.stream);
    for (int k = 0; k < F; ++k) {
        const int64_t pad0 = off[k] + cnt[k], npadrows = off[k + 1] - pad0;
        if (npadrows > 0)
            OEM_CUDA(cudaMemset2DAsync(Xs + pad0, (size_t)lds * 8, 0, (size_t)npadrows * 8, p, cx.stream));
    }
    if (off[F] < npad)
        OEM_CUDA(cudaMemset2DAsync(Xs + off[F], (size_t)lds * 8, 0, (size_t)(npad - off[F]) * 8, p, cx.stream));
    fold_gather_launch(cx, X, nr, p, ldx, dest, order, Xs, lds, y, ys.p, w, ws.p, yws.p);
}

// Step 2 for the rows of one fold-sorted block (fold k = rows [off[k], off[k + 1]) of Xs, ld lds, npad rows): ONE
// segmented Gram launch for all F fold Grams, added to the bundle when `accumulate`.  Unweighted: the per-fold column
// sums / X'y / sum x^2 ride in the Gram launch (diagonal-tile CTAs); weighted: a separate sweep per fold (the Gram
// launch's statistics are unweighted).  A fold without rows here launches nothing and keeps its sums.
void xval_bundle_chunk(Ctx &cx, const double *Xs, int64_t npad, int64_t lds, const double *ys, const double *ws,
                       const double *yws, const std::vector<int64_t> &off, bool accumulate, XvalBundle &b) {
    const int F = b.F, p = b.p;
    std::vector<RowSegment> segs;
    for (int k = 0; k < F; ++k) segs.push_back(RowSegment{off[k], off[k + 1], k});
    if (!b.weighted) gram_launch(cx, Xs, npad, p, lds, segs, F, nullptr, nullptr, b.G, accumulate, ys, b.stats);
    else gram_launch(cx, Xs, npad, p, lds, segs, F, nullptr, ws, b.G, accumulate);
    const size_t t_c = cx.tm->start(&cx.st.ms_colstats);
    for (int k = 0; k < F; ++k) {
        const int64_t len = off[k + 1] - off[k];
        if (len == 0) continue;
        const bool acc = b.seen[k] != 0;
        if (b.weighted)
            colstats_launch(cx, Xs + off[k], len, p, lds, ws + off[k], yws + off[k], nullptr, b.stats + (size_t)k * 3 * p, acc);
        vecsum_launch(cx, (b.weighted ? yws : ys) + off[k], len, 0.0, b.ysum + (size_t)k * 2, acc);
        if (b.weighted) vecsum_launch(cx, ws + off[k], len, 0.0, b.wsum2.p + 2 * (size_t)k, acc);   // corner_k = sum w
        b.seen[k] = 1;
    }
    cx.tm->stop(t_c);
}

// The end of step 2 and step 3 once every row is in the bundle: the sums of folds without rows, nobs and corner from
// the row counts cnt, the Hessian scaling, the all-reduce, then the full-data and leave-one-fold-out systems.
void xval_finish_systems(Ctx &cx, const std::vector<int64_t> &cnt, int icpt, bool stdz, double hess_scale, XvalBundle &b,
                         XvalSystems &xs) {
    PhaseTimers &tm = *cx.tm;
    const int F = b.F, p = b.p, q = p + icpt;
    for (int k = 0; k < F; ++k)
        if (!b.seen[k]) {
            if (b.weighted) OEM_CUDA(cudaMemsetAsync(b.stats + (size_t)k * 3 * p, 0, 3 * (size_t)p * 8, cx.stream));
            OEM_CUDA(cudaMemsetAsync(b.ysum + (size_t)k * 2, 0, 16, cx.stream));
        }
    {
        std::vector<double> hc(F);
        for (int k = 0; k < F; ++k) hc[k] = (double)cnt[k];
        OEM_CUDA(cudaMemcpyAsync(b.nobs, hc.data(), F * sizeof(double), cudaMemcpyHostToDevice, cx.stream));
        if (!b.weighted)
            OEM_CUDA(cudaMemcpyAsync(b.corner, hc.data(), F * sizeof(double), cudaMemcpyHostToDevice, cx.stream));
    }
    if (b.weighted) OEM_CUDA(cudaMemcpy2DAsync(b.corner, 8, b.wsum2.p, 16, 8, F, cudaMemcpyDeviceToDevice, cx.stream));
    if (hess_scale != 1.0) {
        const size_t ng = (size_t)F * p * p;
        xval_hess_scale_kernel<<<(unsigned)((ng + 255) / 256), 256, 0, cx.stream>>>(b.G, ng, b.stats, F, p, b.corner, hess_scale);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 1;
    }
    const size_t t_ar = tm.start(&cx.st.ms_allreduce);
    cx.all_reduce(b.buf.p, (int64_t)b.nb);
    tm.stop(t_ar);

    // ---- 3. assemble full-data + leave-one-fold-out systems ----
    xs.F = F;
    xs.NG = F + 1;
    const int NG = xs.NG;
    const size_t t_as = tm.start(&cx.st.ms_assemble);
    xs.XX.alloc((size_t)NG * q * q);
    xs.XY.alloc((size_t)NG * q);
    xs.cinv.alloc((size_t)NG * p);
    xs.nout.alloc(NG);
    assemble_aug_launch(cx, p, icpt, stdz ? 1 : 0, F, NG, b.G, b.stats, b.ysum, 2, b.corner, b.nobs, xs.XX.p, xs.XY.p,
                        xs.cinv.p, xs.nout.p);
    xs.hXY.resize(q);
    xs.hcinv.resize((size_t)NG * p);
    xs.hn.resize(NG);
    xs.XY.download(xs.hXY.data(), q, cx.stream);
    xs.cinv.download(xs.hcinv.data(), xs.hcinv.size(), cx.stream);
    xs.nout.download(xs.hn.data(), NG, cx.stream);
    tm.stop(t_as);
    cx.sync();
}

}  // namespace

// steps 1-3 (see the top of the file) on a resident X, shared by fit_xval and fit_xval_logistic
void xval_build_systems(Ctx &cx, const double *x, int64_t n, int p, int64_t ldx, const double *y, const double *weights,
                        int F, const int *foldid, int icpt, bool stdz, double hess_scale, XvalSystems &xs) {
    PhaseTimers &tm = *cx.tm;
    const bool weighted = weights != nullptr;

    // ---- 1. fold buckets: stable counting sort of the rows by fold (device kernels; host loops only for > 64 folds) ----
    const int64_t align = 2 * gram_kt();
    std::vector<int64_t> &cnt = xs.cnt, &off = xs.off;
    cnt.assign(F, 0);
    off.assign(F + 1, 0);
    const size_t t_h = tm.start(&cx.st.ms_h2d);
    DevMatrix X;
    to_device_matrix(cx, x, n, p, ldx, X);
    DevVector yv, wv;
    to_device_vector(cx, y, n, yv);
    if (weighted) to_device_vector(cx, weights, n, wv);
    DBuf<int> d_dest(n), d_order(n), d_fold;
    const int *fold_dev = foldid;
    if (!is_device_ptr(foldid)) {
        d_fold.alloc(n);
        d_fold.upload(foldid, n, cx.stream);
        fold_dev = d_fold.p;
    }
    tm.stop(t_h);
    collective_guard(cx, [&] {          // fold ids are validated per rank: agree before the first data all-reduce
    if (!fold_bucket_device(cx, fold_dev, n, F, align, d_dest.p, d_order.p, cnt, off)) {
        if (is_device_ptr(foldid)) fail(OEMB200_EUNSUPPORTED, "xval: more than 64 folds needs foldid on the host");
        std::vector<int> dest(n), order(n);
        xval_bucket_host(foldid, n, F, align, cnt, off, dest.data(), order.data());
        d_dest.upload(dest.data(), n, cx.stream);
        d_order.upload(order.data(), n, cx.stream);
        cx.sync();
    }
    });
    const int64_t npad = std::max<int64_t>(off[F], align);
    xs.npad = npad;
    if (npad >= (1ll << 31)) fail(OEMB200_EUNSUPPORTED, "xval: more than 2^31 rows per rank; shard the rows");
    xs.Xs.alloc((size_t)npad * p);
    xs.ys.alloc(npad);
    DBuf<double> yws;
    if (weighted) {
        xs.ws.alloc(npad);
        yws.alloc(npad);
    }
    xval_gather(cx, X.p, n, p, X.ld, yv.p, weighted ? wv.p : nullptr, d_dest.p, d_order.p, cnt, off, npad, xs.Xs.p, npad,
                xs.ys, xs.ws, yws);
    X.own.release();          // the fold-sorted copy replaces the uploaded one

    // ---- 2. per-fold sums, 3. systems ----
    XvalBundle b(cx, F, p, weighted);
    xval_bundle_chunk(cx, xs.Xs.p, npad, npad, xs.ys.p, xs.ws.p, yws.p, off, false, b);
    xval_finish_systems(cx, cnt, icpt, stdz, hess_scale, b, xs);
}

// Stable counting sort of foldid[0, n) by fold on the host (more than fold_bucket_max_folds() folds): cnt / off as in
// XvalSystems, and dest / order for fold_gather_launch.  Refuses ids outside 1..F.
void xval_bucket_host(const int *foldid, int64_t n, int F, int64_t align, std::vector<int64_t> &cnt, std::vector<int64_t> &off,
                      int *dest, int *order) {
    cnt.assign(F, 0);
    off.assign(F + 1, 0);
    for (int64_t i = 0; i < n; ++i) {
        const int f = foldid[i];
        if (f < 1 || f > F) fail(OEMB200_EINVAL, "foldid[%lld] = %d outside 1..%d", (long long)i, f, F);
        cnt[f - 1]++;
    }
    for (int k = 0; k < F; ++k) off[k + 1] = off[k] + (cnt[k] + align - 1) / align * align;
    std::vector<int64_t> cur(off.begin(), off.end() - 1);
    for (int64_t i = 0; i < n; ++i) dest[i] = (int)cur[foldid[i] - 1]++;
    const int64_t TR = fold_gather_tile_rows();
    std::vector<int> c2(F + 1);
    for (int64_t t0 = 0; t0 < n; t0 += TR) {
        const int64_t t1 = std::min(n, t0 + TR);
        std::fill(c2.begin(), c2.end(), 0);
        for (int64_t i = t0; i < t1; ++i) c2[foldid[i]]++;
        int run = 0;
        for (int f = 1; f <= F; ++f) { const int c = c2[f]; c2[f] = run; run += c; }
        for (int64_t i = t0; i < t1; ++i) order[t0 + c2[foldid[i]]++] = (int)(i - t0);
    }
}

namespace {

// the argument checks of oemb200_xval_dense / oemb200_xval_big; returns true for type_measure "mae"
bool xval_check(int64_t n, int p, int64_t ldx, const oemb200_spec *s, int nfolds, const int *foldid, const char *type_measure,
                const oemb200_opts *o, const oemb200_result *res) {
    check_common(s, o, res, "gaussian", /*allow_weights=*/true);
    if (n < 1 || p < 1 || ldx < n) fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d ldx=%lld", (long long)n, p, (long long)ldx);
    // observation weights (xval.oem(weights=), R/oem_xval.R:215-222): XtWX_xval[_int], oem_xval_dense.h:489-627
    if (s->n_weights > 0 && s->n_weights != n)
        fail(OEMB200_EINVAL, "length of weights not same as number of observations in x");      // R/oem_xval.R:218-221
    if (nfolds < 2 || !foldid) fail(OEMB200_EINVAL, "xval needs nfolds >= 2 and foldid");
    if (!res->cvm || !res->cvsd) fail(OEMB200_EINVAL, "xval needs cvm / cvsd result buffers");
    if (type_measure && strcmp(type_measure, "mae") == 0) return true;
    if (type_measure && strcmp(type_measure, "mse") != 0 && strcmp(type_measure, "deviance") != 0)
        fail(OEMB200_EINVAL, "type_measure must be \"mse\" or \"mae\" for the gaussian family");
    return false;
}

const char *const kTooFewRows = "dimension of x larger than number of observations";      // oem_xval_dense.h:690

// step 4: the lambda grid from the full-data system, all chains in one persistent launch, the full-data fit into res
void xval_solve(Ctx &cx, Setup &su, const oemb200_spec *s, const oemb200_opts *o, const XvalSystems &xs, int p, int icpt,
                oemb200_result *res, PathBuffers &pb) {
    PhaseTimers &tm = *cx.tm;
    for (int g = 0; g < xs.NG; ++g)
        if (!(xs.hn[g] > p)) fail(OEMB200_EINVAL, "%s", kTooFewRows);
    double lmax = 0.0;      // X entries only (oem_xval_dense.h:1063-1069)
    for (int j = 0; j < p; ++j) lmax = std::max(lmax, std::fabs(xs.hXY[icpt + j]));
    su.build_lambdas(s, lmax, false);

    PenaltyTables tb(cx, su, s, p, icpt);
    const size_t t_p = tm.start(&cx.st.ms_path);
    run_paths(cx, su, tb, o, xs.NG, xs.XX.p, xs.XY.p, 1.005, false, nullptr, pb);
    tm.stop(t_p);

    const int L = su.Lmax;
    fill_common_outputs(su, res);
    write_beta(su, pb.h_beta.data(), p, icpt, s->standardize ? xs.hcinv.data() : nullptr, res);   // the full-data chains
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) res->niter[(size_t)pp * L + i] = pb.h_niter[(size_t)pp * L + i];
    *res->d = pb.h_d[0];
}

// Step 5, the CV scoring: coefficient matrices [fold][p][ncld] and intercepts [fold][ncld] of the fold models, and with
// compute_loss the full model's (the same for every fold), and the running (count, mean, M2) of both scores.
struct XvalScore {
    int F = 0, nc = 0;
    bool mae = false, loss = false;
    DBuf<double> B, b0, out3;               // fold models: the CV score
    DBuf<double> lB, lb0, lout3;            // full model: the loss
    DBuf<int> nlam;
    std::vector<double> hlB, hlb0;          // host sources of the lB / lb0 uploads
};

void xval_score_setup(Ctx &cx, const Setup &su, const PathBuffers &pb, const XvalSystems &xs, const oemb200_spec *s,
                      const oemb200_result *res, int p, int icpt, bool mae, XvalScore &sc) {
    const int F = xs.F, P = su.P, L = su.Lmax, q = p + icpt;
    sc.F = F;
    sc.nc = P * L;
    sc.mae = mae;
    sc.loss = s->compute_loss && res->loss;
    const int ncld = cv_ncld(sc.nc);
    sc.B.alloc((size_t)F * p * ncld);
    sc.b0.alloc((size_t)F * ncld);
    sc.out3.alloc(3 * (size_t)sc.nc);
    sc.nlam.alloc(P);
    sc.nlam.upload(su.nlam_run.data(), P, cx.stream);
    cv_build_coef_launch(cx, pb.beta_out.p, xs.cinv.p, F, P, L, p, q, icpt, s->standardize != 0, sc.nlam.p, sc.B.p, sc.b0.p);
    if (!sc.loss) return;
    // loss of the full-data fit = sum (y - b0 - x b)^2: the same pass with one coefficient set for every fold
    sc.hlB.assign((size_t)F * p * ncld, 0.0);
    sc.hlb0.assign((size_t)F * ncld, 0.0);
    for (int k = 0; k < F; ++k)
        for (int pp = 0; pp < P; ++pp)
            for (int i = 0; i < su.nlam_run[pp]; ++i) {
                const double *bo = res->beta + ((size_t)pp * L + i) * (p + 1);
                const int c = pp * L + i;
                sc.hlb0[(size_t)k * ncld + c] = bo[0];
                for (int j = 0; j < p; ++j) sc.hlB[((size_t)k * p + j) * ncld + c] = bo[1 + j];
            }
    sc.lB.alloc(sc.hlB.size());
    sc.lb0.alloc(sc.hlb0.size());
    sc.lout3.alloc(3 * (size_t)sc.nc);
    sc.lB.upload(sc.hlB.data(), sc.hlB.size(), cx.stream);
    sc.lb0.upload(sc.hlb0.data(), sc.hlb0.size(), cx.stream);
}

// the rows of one fold-sorted block (as in xval_bundle_chunk; ws may be NULL) merged into the running scores
void xval_score_chunk(Ctx &cx, XvalScore &sc, const double *Xs, int64_t npad, int p, int64_t lds, const double *ys,
                      const double *ws, const std::vector<int64_t> &cnt, const std::vector<int64_t> &off, bool accumulate) {
    std::vector<std::array<int64_t, 3>> cs;
    for (int k = 0; k < sc.F; ++k) cs.push_back({off[k], off[k + 1], off[k] + cnt[k]});
    cvscore_launch(cx, Xs, npad, p, lds, ys, ws, sc.F, cs, sc.B.p, sc.b0.p, sc.nc, sc.mae, sc.out3.p, accumulate);
    if (sc.loss)       // the loss is unweighted (.h:1122-1145)
        cvscore_launch(cx, Xs, npad, p, lds, ys, nullptr, sc.F, cs, sc.lB.p, sc.lb0.p, sc.nc, false, sc.lout3.p, accumulate);
}

// cvm / cvsd (and the loss) from the merged moments; a row-sharded run merges across ranks with sum all-reduces only
void xval_score_finish(Ctx &cx, XvalScore &sc, const Setup &su, double n_tot, oemb200_result *res) {
    const int nc = sc.nc, P = su.P, L = su.Lmax;
    std::vector<double> h3(3 * (size_t)nc);
    sc.out3.download(h3.data(), h3.size(), cx.stream);
    cx.sync();
    if (cx.distributed()) {
        // cross-rank merge with sum all-reduces only: first (count, sum) -> global mean, then M2 about it
        std::vector<double> a(2 * (size_t)nc);
        for (int c = 0; c < nc; ++c) { a[c] = h3[c]; a[nc + c] = h3[c] * h3[nc + c]; }
        DBuf<double> da(a.size());
        da.upload(a.data(), a.size(), cx.stream);
        cx.all_reduce(da.p, (int64_t)a.size());
        da.download(a.data(), a.size(), cx.stream);
        cx.sync();
        std::vector<double> m2(nc);
        for (int c = 0; c < nc; ++c) {
            const double gm = a[c] > 0 ? a[nc + c] / a[c] : 0.0;
            const double dl = h3[nc + c] - gm;
            m2[c] = h3[2 * nc + c] + h3[c] * dl * dl;
        }
        DBuf<double> dm(nc);
        dm.upload(m2.data(), nc, cx.stream);
        cx.all_reduce(dm.p, nc);
        dm.download(m2.data(), nc, cx.stream);
        cx.sync();
        for (int c = 0; c < nc; ++c) { h3[c] = a[c]; h3[nc + c] = a[c] > 0 ? a[nc + c] / a[c] : 0.0; h3[2 * nc + c] = m2[c]; }
    }
    for (int pp = 0; pp < P; ++pp)
        for (int i = 0; i < L; ++i) {
            const int c = pp * L + i;
            const bool live = i < su.nlam_run[pp];
            res->cvm[c] = live ? h3[nc + c] : 0.0;
            res->cvsd[c] = live ? std::sqrt(h3[2 * nc + c] / (n_tot - 1.0)) / std::sqrt(n_tot) : 0.0;
        }
    if (!sc.loss) return;
    sc.lout3.download(h3.data(), h3.size(), cx.stream);
    cx.sync();
    std::vector<double> tot(nc);
    for (int c = 0; c < nc; ++c) tot[c] = h3[c] * h3[nc + c];
    if (cx.distributed()) {
        DBuf<double> dt(nc);
        dt.upload(tot.data(), nc, cx.stream);
        cx.all_reduce(dt.p, nc);
        dt.download(tot.data(), nc, cx.stream);
        cx.sync();
    }
    for (int pp = 0; pp < P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) res->loss[(size_t)pp * L + i] = tot[pp * L + i];
}

}  // namespace

void fit_xval(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s, int nfolds,
              const int *foldid, const char *type_measure, const oemb200_opts *o, oemb200_result *res) {
    const bool mae = xval_check(n, p, ldx, s, nfolds, foldid, type_measure, o, res);
    const bool weighted = s->n_weights > 0;
    const int icpt = s->intercept ? 1 : 0, q = p + icpt;
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, q, false);

    XvalSystems xs;
    xval_build_systems(cx, x, n, p, ldx, y, weighted ? s->weights : nullptr, nfolds, foldid, icpt, s->standardize != 0, 1.0, xs);
    PathBuffers pb;
    xval_solve(cx, su, s, o, xs, p, icpt, res, pb);
    XvalScore sc;
    xval_score_setup(cx, su, pb, xs, s, res, p, icpt, mae, sc);
    xval_score_chunk(cx, sc, xs.Xs.p, xs.npad, p, xs.npad, xs.ys.p, weighted ? xs.ws.p : nullptr, xs.cnt, xs.off, false);
    xval_score_finish(cx, sc, su, xs.hn[0], res);
    finish_stats(cx, tm, t_total, res);
}

// oemb200_xval_big: fit_xval on an X that is never resident.  Rows are read in chunks of big_chunk_rows() (opts->gigs GB);
// each chunk is bucketed and gathered into a chunk-local fold-sorted block (the layout of xval_build_systems, with its
// own 72-row aligned fold segments) and goes through the same per-block steps as the resident X, which is one block:
//   pre-pass  one fold_count_launch per chunk on foldid, one download: every chunk's fold segments are known on the host;
//   pass 1    per chunk: xval_bundle_chunk into the F fold Grams (accumulate from the second chunk on); then
//             xval_finish_systems and xval_solve as for a resident X;
//   pass 2    per chunk: xval_score_chunk, whose moments merge into the running state in chunk order (cv_merge_kernel's
//             accumulate mode), so the result does not depend on timing.
// Host chunks are staged on a copy stream (CopyLane) into two buffers while the compute stream works on the previous
// chunk: pinned sources are queued two chunks ahead, pageable ones (the pinned bounce ring of h2d_block) one.  A device
// X is read in place.  Neither pass synchronises with the host.  Device memory holds the two staging buffers, one
// fold-sorted block, the bundle, the systems, the path and the coefficient matrices: nothing that grows with n beyond
// F counts per chunk.
void fit_xval_big(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s, int nfolds,
                  const int *foldid, const char *type_measure, const oemb200_opts *o, oemb200_result *res) {
    if (s && s->family && strcmp(s->family, "binomial") == 0)
        fail(OEMB200_EUNSUPPORTED, "streamed xval is gaussian only: a binomial fit makes one pass over X per IRLS round, and "
                                   "each pass of a streamed X would cross the host link again; use oem_xval_logistic_dense "
                                   "on an X that fits on the device");
    if (o && (o->world > 1 || o->comm || o->allreduce))
        fail(OEMB200_EUNSUPPORTED, "streamed xval runs on one GPU; row-sharded cross-validation is oem_xval_dense with each "
                                   "rank's rows resident");
    const bool mae = xval_check(n, p, ldx, s, nfolds, foldid, type_measure, o, res);
    const bool weighted = s->n_weights > 0;
    const int icpt = s->intercept ? 1 : 0, q = p + icpt, F = nfolds;
    const bool host_bucket = F > fold_bucket_max_folds();
    const double *w = weighted ? s->weights : nullptr;
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, q, false);
    const bool dev_x = is_device_ptr(x), dev_y = is_device_ptr(y), dev_w = w && is_device_ptr(w);
    const bool dev_fold = is_device_ptr(foldid);
    if (host_bucket && dev_fold) fail(OEMB200_EUNSUPPORTED, "xval: more than 64 folds needs foldid on the host");

    const int64_t align = 2 * gram_kt();
    const int64_t rows = big_chunk_rows(o, n, p), nchunks = (n + rows - 1) / rows;
    const int64_t cap = rows + (int64_t)F * align;           // rows of a fold-sorted block: every segment pads < 72 rows
    if (cap >= (1ll << 31)) fail(OEMB200_EUNSUPPORTED, "xval: chunks of more than 2^31 rows; lower opts->gigs");
    auto chunk_rows = [&](int64_t c) { return std::min(rows, n - c * rows); };

    // ---- pre-pass: rows per (chunk, fold) ----
    std::vector<int64_t> ccnt((size_t)nchunks * F, 0), coff((size_t)nchunks * (F + 1), 0), cnt(F, 0);
    std::vector<int> hdest, horder;                           // > 64 folds: chunk-local dest / order of every row
    DBuf<int> tcount, err(1), fstage[2];
    DBuf<long long> d_tot, d_base;
    std::vector<long long> hbase((size_t)nchunks * F);
    if (!host_bucket) {
        tcount.alloc((size_t)((rows + fold_gather_tile_rows() - 1) / fold_gather_tile_rows()) * F);
        if (!dev_fold) for (auto &f : fstage) f.alloc(rows);
        d_tot.alloc((size_t)nchunks * F);
        err.zero(cx.stream);
        for (int64_t c = 0; c < nchunks; ++c) {
            const int64_t nr = chunk_rows(c);
            const int *fp = foldid + c * rows;
            if (!dev_fold) {
                OEM_CUDA(cudaMemcpyAsync(fstage[0].p, fp, (size_t)nr * 4, cudaMemcpyHostToDevice, cx.stream));
                cx.st.h2d_bytes += nr * 4;
                fp = fstage[0].p;
            }
            fold_count_launch(cx, fp, nr, F, tcount.p, err.p, d_tot.p + (size_t)c * F);
        }
        std::vector<long long> ht((size_t)nchunks * F);
        int herr = 0;
        d_tot.download(ht.data(), ht.size(), cx.stream);
        err.download(&herr, 1, cx.stream);
        cx.sync();
        if (herr) fail(OEMB200_EINVAL, "foldid has entries outside 1..%d", F);
        for (size_t i = 0; i < ht.size(); ++i) ccnt[i] = ht[i];
    } else {
        hdest.resize(n);
        horder.resize(n);
        std::vector<int64_t> cc, co;
        for (int64_t c = 0; c < nchunks; ++c) {
            xval_bucket_host(foldid + c * rows, chunk_rows(c), F, align, cc, co, hdest.data() + c * rows, horder.data() + c * rows);
            std::copy(cc.begin(), cc.end(), ccnt.begin() + c * F);
        }
    }
    for (int64_t c = 0; c < nchunks; ++c)
        for (int k = 0; k < F; ++k) {
            const int64_t m = ccnt[c * F + k];
            cnt[k] += m;
            coff[c * (F + 1) + k + 1] = coff[c * (F + 1) + k] + (m + align - 1) / align * align;
            hbase[c * F + k] = coff[c * (F + 1) + k];
        }
    // the systems' row counts are known now: refuse before streaming X (xval_solve checks the same counts again)
    if (!(n > p)) fail(OEMB200_EINVAL, "%s", kTooFewRows);
    for (int k = 0; k < F; ++k)
        if (!(n - cnt[k] > p)) fail(OEMB200_EINVAL, "%s", kTooFewRows);
    if (!host_bucket) {
        d_base.alloc(hbase.size());
        d_base.upload(hbase.data(), hbase.size(), cx.stream);
    }

    // ---- the two streamed passes ----
    DBuf<double> stage[2], ystage[2], wstage[2];
    DBuf<int> dest(rows), order(rows);
    for (int b = 0; b < 2; ++b) {
        if (!dev_x) stage[b].alloc((size_t)rows * p);
        if (!dev_y) ystage[b].alloc(rows);
        if (w && !dev_w) wstage[b].alloc(rows);
    }
    DBuf<double> Xs((size_t)cap * p), ys(cap), ws, yws;
    if (weighted) {
        ws.alloc(cap);
        yws.alloc(cap);
    }
    CopyLane lane;
    const bool ahead2 = dev_x || is_pinned_host(x);
    int64_t seq = 0;            // chunks staged so far over both passes: chunk c of the pass starting at s0 uses buffer (s0 + c) & 1
    auto issue_copy = [&](int64_t s0, int64_t c) {
        const int b = (int)((s0 + c) & 1);
        const int64_t r0 = c * rows, nr = chunk_rows(c);
        if (s0 + c >= 2) OEM_CUDA(cudaStreamWaitEvent(lane.s, lane.freed[b], 0));
        if (!dev_x) h2d_block(cx, x + r0, ldx, nr, p, stage[b].p, rows, lane.s);
        if (!dev_y) h2d_block(cx, y + r0, n, nr, 1, ystage[b].p, rows, lane.s);
        if (w && !dev_w) h2d_block(cx, w + r0, n, nr, 1, wstage[b].p, rows, lane.s);
        if (!dev_fold && !host_bucket) {
            OEM_CUDA(cudaMemcpyAsync(fstage[b].p, foldid + r0, (size_t)nr * 4, cudaMemcpyHostToDevice, lane.s));
            cx.st.h2d_bytes += nr * 4;
        }
        OEM_CUDA(cudaEventRecord(lane.ready[b], lane.s));
        seq = s0 + c + 1;
    };
    // one pass: chunk c is staged, bucketed and gathered into Xs / ys / ws / yws, then body(c, cnt_c, off_c, npad_c) queues
    // the chunk's work; once that is queued the staging buffer is released to the copy after next
    auto pass = [&](const std::function<void(int64_t, const std::vector<int64_t> &, const std::vector<int64_t> &, int64_t)> &body) {
        const int64_t s0 = seq;
        issue_copy(s0, 0);
        if (nchunks > 1 && ahead2) issue_copy(s0, 1);
        std::vector<int64_t> cc(F), co(F + 1);
        for (int64_t c = 0; c < nchunks; ++c) {
            const int b = (int)((s0 + c) & 1);
            const int64_t r0 = c * rows, nr = chunk_rows(c);
            OEM_CUDA(cudaStreamWaitEvent(cx.stream, lane.ready[b], 0));
            std::copy(ccnt.begin() + c * F, ccnt.begin() + (c + 1) * F, cc.begin());
            std::copy(coff.begin() + c * (F + 1), coff.begin() + (c + 1) * (F + 1), co.begin());
            if (!host_bucket) {
                const int *fp = dev_fold ? foldid + r0 : fstage[b].p;
                fold_count_launch(cx, fp, nr, F, tcount.p, err.p, d_tot.p);      // tile prefixes (the totals are known)
                fold_rank_launch(cx, fp, nr, F, tcount.p, d_base.p + c * F, dest.p, order.p);
            } else {
                dest.upload(hdest.data() + r0, nr, cx.stream);
                order.upload(horder.data() + r0, nr, cx.stream);
                cx.st.h2d_bytes += nr * 8;
            }
            const int64_t npad = std::max<int64_t>(co[F], align);
            xval_gather(cx, dev_x ? x + r0 : stage[b].p, nr, p, dev_x ? ldx : rows, dev_y ? y + r0 : ystage[b].p,
                        w ? (dev_w ? w + r0 : wstage[b].p) : nullptr, dest.p, order.p, cc, co, npad, Xs.p, cap, ys, ws, yws);
            OEM_CUDA(cudaEventRecord(lane.freed[b], cx.stream));
            body(c, cc, co, npad);
            const int64_t nxt = ahead2 ? c + 2 : c + 1;
            if (nxt < nchunks) issue_copy(s0, nxt);
        }
    };

    XvalSystems xs;
    {
        XvalBundle bundle(cx, F, p, weighted);
        const size_t t_h = tm.start(&cx.st.ms_h2d);      // pass 1 as a whole (the copies overlap the kernels)
        pass([&](int64_t c, const std::vector<int64_t> &, const std::vector<int64_t> &co, int64_t npad) {
            xval_bundle_chunk(cx, Xs.p, npad, cap, ys.p, ws.p, yws.p, co, c > 0, bundle);
        });
        tm.stop(t_h);
        xval_finish_systems(cx, cnt, icpt, s->standardize != 0, 1.0, bundle, xs);
    }
    PathBuffers pb;
    xval_solve(cx, su, s, o, xs, p, icpt, res, pb);
    XvalScore sc;
    xval_score_setup(cx, su, pb, xs, s, res, p, icpt, mae, sc);
    pass([&](int64_t c, const std::vector<int64_t> &cc, const std::vector<int64_t> &co, int64_t npad) {
        xval_score_chunk(cx, sc, Xs.p, npad, p, cap, ys.p, weighted ? ws.p : nullptr, cc, co, c > 0);
    });
    cx.st.data_passes = 2;
    xval_score_finish(cx, sc, su, xs.hn[0], res);
    finish_stats(cx, tm, t_total, res);
}

}  // namespace oemb200
