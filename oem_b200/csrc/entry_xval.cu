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
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include "host_common.h"

namespace oemb200 {

// per-fold bundle scaled for the logistic upper-bound Hessian: G_k, the column sums of stats row 0 and the corner
__global__ void xval_hess_scale_kernel(double *G, size_t ng, double *stats, int F, int p, double *corner, double f) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ng) G[i] *= f;
    if (i < (size_t)F * p) stats[(i / p) * 3 * p + i % p] *= f;
    if (i < (size_t)F) corner[i] *= f;
}

// steps 1-3 (see the top of the file), shared by fit_xval and fit_xval_logistic
void xval_build_systems(Ctx &cx, const double *x, int64_t n, int p, int64_t ldx, const double *y, const double *weights,
                        int F, const int *foldid, int icpt, bool stdz, double hess_scale, XvalSystems &xs) {
    PhaseTimers &tm = *cx.tm;
    const bool weighted = weights != nullptr;
    xs.F = F;
    xs.NG = F + 1;
    const int q = p + icpt;

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
    DBuf<double> &Xs = xs.Xs, &ys = xs.ys, &ws = xs.ws, yws;
    // only the (< 72) padding rows at the end of each fold segment need zeros; the gather writes every other row
    ys.zero(cx.stream);
    if (weighted) {
        ws.alloc(npad);
        yws.alloc(npad);
        ws.zero(cx.stream);
        yws.zero(cx.stream);
    }
    for (int k = 0; k < F; ++k) {
        const int64_t pad0 = off[k] + cnt[k], npadrows = off[k + 1] - pad0;
        if (npadrows > 0)
            OEM_CUDA(cudaMemset2DAsync(Xs.p + pad0, (size_t)npad * 8, 0, (size_t)npadrows * 8, p, cx.stream));
    }
    if (off[F] < npad)
        OEM_CUDA(cudaMemset2DAsync(Xs.p + off[F], (size_t)npad * 8, 0, (size_t)(npad - off[F]) * 8, p, cx.stream));
    fold_gather_launch(cx, X.p, n, p, X.ld, d_dest.p, d_order.p, Xs.p, npad, yv.p, ys.p, weighted ? wv.p : nullptr,
                       ws.p, yws.p);
    X.own.release();          // the fold-sorted copy replaces the uploaded one

    // ---- 2. per-fold sums: bundle = [G F*p*p | stats F*3p | ysum F*2 | nobs F | corner F] ----
    // unweighted: G_k = X_k'X_k, stats = (colsums, X_k'y, sum x^2), ysum = sum y, corner = n_k.
    // weighted:   G_k = X_k'W X_k, stats = (sum w x, X_k'(y*w), UNWEIGHTED sum x^2), ysum = sum y*w, corner = sum w;
    //             nobs stays the row count (oem_xval_dense.h:528-545, 596-624).
    const size_t nb = (size_t)F * p * p + (size_t)F * 3 * p + (size_t)F * 2 + 2 * (size_t)F;
    DBuf<double> bundle(nb);
    double *G = bundle.p, *stats = G + (size_t)F * p * p, *ysum = stats + (size_t)F * 3 * p, *nobs = ysum + (size_t)F * 2;
    double *corner = nobs + F;
    std::vector<RowSegment> segs;
    for (int k = 0; k < F; ++k) segs.push_back(RowSegment{off[k], off[k + 1], k});
    // unweighted: the per-fold column sums / X'y / sum x^2 ride in the Gram launch (diagonal-tile CTAs); weighted: a
    // separate sweep per fold (the Gram launch's statistics are unweighted)
    if (!weighted) gram_launch(cx, Xs.p, npad, p, npad, segs, F, nullptr, nullptr, G, false, ys.p, stats);
    else gram_launch(cx, Xs.p, npad, p, npad, segs, F, nullptr, ws.p, G, false);
    const size_t t_c = tm.start(&cx.st.ms_colstats);
    for (int k = 0; k < F; ++k) {
        const int64_t len = off[k + 1] - off[k];
        if (len > 0) {
            if (weighted)
                colstats_launch(cx, Xs.p + off[k], len, p, npad, ws.p + off[k], yws.p + off[k], nullptr,
                                stats + (size_t)k * 3 * p, false);
            vecsum_launch(cx, (weighted ? yws.p : ys.p) + off[k], len, 0.0, ysum + (size_t)k * 2, false);
        } else {
            if (weighted) OEM_CUDA(cudaMemsetAsync(stats + (size_t)k * 3 * p, 0, 3 * (size_t)p * 8, cx.stream));
            OEM_CUDA(cudaMemsetAsync(ysum + (size_t)k * 2, 0, 16, cx.stream));
        }
    }
    tm.stop(t_c);
    {
        std::vector<double> hc(F);
        for (int k = 0; k < F; ++k) hc[k] = (double)cnt[k];
        OEM_CUDA(cudaMemcpyAsync(nobs, hc.data(), F * sizeof(double), cudaMemcpyHostToDevice, cx.stream));
        if (!weighted)
            OEM_CUDA(cudaMemcpyAsync(corner, hc.data(), F * sizeof(double), cudaMemcpyHostToDevice, cx.stream));
    }
    DBuf<double> wsum2;
    if (weighted) {           // corner_k = sum of the fold's weights (vecsum writes [sum, sum of squares])
        wsum2.alloc(2 * (size_t)F);
        wsum2.zero(cx.stream);
        for (int k = 0; k < F; ++k)
            if (off[k + 1] > off[k]) vecsum_launch(cx, ws.p + off[k], off[k + 1] - off[k], 0.0, wsum2.p + 2 * (size_t)k, false);
        OEM_CUDA(cudaMemcpy2DAsync(corner, 8, wsum2.p, 16, 8, F, cudaMemcpyDeviceToDevice, cx.stream));
    }
    if (hess_scale != 1.0) {
        const size_t ng = (size_t)F * p * p;
        xval_hess_scale_kernel<<<(unsigned)((ng + 255) / 256), 256, 0, cx.stream>>>(G, ng, stats, F, p, corner, hess_scale);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 1;
    }
    const size_t t_ar = tm.start(&cx.st.ms_allreduce);
    cx.all_reduce(bundle.p, (int64_t)nb);
    tm.stop(t_ar);

    // ---- 3. assemble full-data + leave-one-fold-out systems ----
    const int NG = xs.NG;
    const size_t t_as = tm.start(&cx.st.ms_assemble);
    xs.XX.alloc((size_t)NG * q * q);
    xs.XY.alloc((size_t)NG * q);
    xs.cinv.alloc((size_t)NG * p);
    xs.nout.alloc(NG);
    assemble_aug_launch(cx, p, icpt, stdz ? 1 : 0, F, NG, G, stats, ysum, 2, corner, nobs, xs.XX.p, xs.XY.p, xs.cinv.p, xs.nout.p);
    xs.hXY.resize(q);
    xs.hcinv.resize((size_t)NG * p);
    xs.hn.resize(NG);
    xs.XY.download(xs.hXY.data(), q, cx.stream);
    xs.cinv.download(xs.hcinv.data(), xs.hcinv.size(), cx.stream);
    xs.nout.download(xs.hn.data(), NG, cx.stream);
    tm.stop(t_as);
    cx.sync();
}

void fit_xval(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s, int nfolds,
              const int *foldid, const char *type_measure, const oemb200_opts *o, oemb200_result *res) {
    check_common(s, o, res, "gaussian", /*allow_weights=*/true);
    if (n < 1 || p < 1 || ldx < n) fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d ldx=%lld", (long long)n, p, (long long)ldx);
    // observation weights (xval.oem(weights=), R/oem_xval.R:215-222): XtWX_xval[_int], oem_xval_dense.h:489-627
    const bool weighted = s->n_weights > 0;
    if (weighted && s->n_weights != n)
        fail(OEMB200_EINVAL, "length of weights not same as number of observations in x");      // R/oem_xval.R:218-221
    if (nfolds < 2 || !foldid) fail(OEMB200_EINVAL, "xval needs nfolds >= 2 and foldid");
    if (!res->cvm || !res->cvsd) fail(OEMB200_EINVAL, "xval needs cvm / cvsd result buffers");
    bool mae = false;
    if (type_measure && strcmp(type_measure, "mae") == 0) mae = true;
    else if (type_measure && strcmp(type_measure, "mse") != 0 && strcmp(type_measure, "deviance") != 0)
        fail(OEMB200_EINVAL, "type_measure must be \"mse\" or \"mae\" for the gaussian family");
    const int icpt = s->intercept ? 1 : 0, q = p + icpt;
    const int F = nfolds;
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, q, false);

    XvalSystems xs;
    xval_build_systems(cx, x, n, p, ldx, y, weighted ? s->weights : nullptr, F, foldid, icpt, s->standardize != 0, 1.0, xs);
    const int NG = xs.NG;
    const std::vector<int64_t> &cnt = xs.cnt, &off = xs.off;
    const int64_t npad = xs.npad;
    const std::vector<double> &hXY = xs.hXY, &hcinv = xs.hcinv, &hn = xs.hn;
    const DBuf<double> &Xs = xs.Xs, &ys = xs.ys, &ws = xs.ws, &XX = xs.XX, &XY = xs.XY, &cinv = xs.cinv;
    const double n_tot = hn[0];
    for (int g = 0; g < NG; ++g)
        if (!(hn[g] > p)) fail(OEMB200_EINVAL, "dimension of x larger than number of observations");   // oem_xval_dense.h:690

    double lmax = 0.0;      // X entries only (oem_xval_dense.h:1063-1069)
    for (int j = 0; j < p; ++j) lmax = std::max(lmax, std::fabs(hXY[icpt + j]));
    su.build_lambdas(s, lmax, false);

    // ---- 4. all chains in one persistent launch ----
    PenaltyTables tb(cx, su, s, p, icpt);
    PathBuffers pb;
    const size_t t_p = tm.start(&cx.st.ms_path);
    run_paths(cx, su, tb, o, NG, XX.p, XY.p, 1.005, false, nullptr, pb);
    tm.stop(t_p);

    const int L = su.Lmax, P = su.P;
    fill_common_outputs(su, res);
    write_beta(su, pb.h_beta.data(), p, icpt, s->standardize ? hcinv.data() : nullptr, res);   // the full-data chains
    for (int pp = 0; pp < P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) res->niter[(size_t)pp * L + i] = pb.h_niter[(size_t)pp * L + i];
    *res->d = pb.h_d[0];

    // ---- 5. CV scoring: coefficient matrices [fold][p][ncld], intercepts [fold][ncld] ----
    const int nc = P * L, ncld = cv_ncld(nc);
    DBuf<double> dB((size_t)F * p * ncld), db0((size_t)F * ncld), out3(3 * (size_t)nc);
    DBuf<int> d_nlam(P);
    d_nlam.upload(su.nlam_run.data(), P, cx.stream);
    cv_build_coef_launch(cx, pb.beta_out.p, cinv.p, F, P, L, p, q, icpt, s->standardize != 0, d_nlam.p, dB.p, db0.p);
    std::vector<std::array<int64_t, 3>> cs;
    for (int k = 0; k < F; ++k) cs.push_back({off[k], off[k + 1], off[k] + cnt[k]});
    cvscore_launch(cx, Xs.p, npad, p, npad, ys.p, weighted ? ws.p : nullptr, F, cs, dB.p, db0.p, nc, mae, out3.p);
    std::vector<double> h3(3 * (size_t)nc);
    out3.download(h3.data(), h3.size(), cx.stream);
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
    if (s->compute_loss && res->loss) {
        // loss of the full-data fit = sum (y - b0 - x b)^2: the same pass with one coefficient set for every fold
        std::vector<double> hB2((size_t)F * p * ncld, 0.0), hb2((size_t)F * ncld, 0.0);
        for (int k = 0; k < F; ++k)
            for (int pp = 0; pp < P; ++pp)
                for (int i = 0; i < su.nlam_run[pp]; ++i) {
                    const double *bo = res->beta + ((size_t)pp * L + i) * (p + 1);
                    const int c = pp * L + i;
                    hb2[(size_t)k * ncld + c] = bo[0];
                    for (int j = 0; j < p; ++j) hB2[((size_t)k * p + j) * ncld + c] = bo[1 + j];
                }
        dB.upload(hB2.data(), hB2.size(), cx.stream);
        db0.upload(hb2.data(), hb2.size(), cx.stream);
        cvscore_launch(cx, Xs.p, npad, p, npad, ys.p, nullptr, F, cs, dB.p, db0.p, nc, false, out3.p);   // loss is unweighted (.h:1122-1145)
        out3.download(h3.data(), h3.size(), cx.stream);
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
    finish_stats(cx, tm, t_total, res);
}

}  // namespace oemb200
