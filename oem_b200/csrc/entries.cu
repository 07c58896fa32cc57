// entries.cu -- host drivers of the reference's entry points on top of the sm_100a kernels, and
// the extern "C" layer of include/oem_b200.h.
//
//   oemb200_fit_dense   <- oem_fit_dense   src/oem_dense.cpp:30-309  (+ DataStd.h, oem_dense.h)
//   oemb200_xtx         <- oem_xtx         src/oem_xtx.cpp:29-219    (+ oem_xtx.h)
//   oemb200_fit_big     <- oem_fit_big     src/oem_big.cpp:30-258    (+ oem_big.h)
// (logistic: entry_logistic.cu, xval: entry_xval.cu, sparse: entry_sparse.cu)
//
// Each driver owns only bookkeeping: which sums to take over X, the lambda grid (host libm, so it
// is bit-identical to a CPU implementation), the penalty x lambda layout of the result.  All
// arithmetic on X, on the Gram and on beta runs in the CUDA kernels.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include "host_common.h"

namespace oemb200 {

thread_local std::string g_last_error;

void check_common(const oemb200_spec *s, const oemb200_opts *o, const oemb200_result *r, const char *want_family,
                  bool allow_weights) {
    if (!s || !o || !r) fail(OEMB200_EINVAL, "spec / opts / result must not be NULL");
    if (!s->family || strcmp(s->family, want_family) != 0) {
        if (strcmp(want_family, "gaussian") == 0)
            fail(OEMB200_EINVAL, "binomial not available for oem_fit_dense, use oem_fit_logistic_dense");
        fail(OEMB200_EINVAL, "family must be \"%s\"", want_family);
    }
    if (s->n_weights > 0 && !allow_weights) fail(OEMB200_EUNSUPPORTED, "weights not implemented yet.");   // R/oem.R:244
    if (s->n_weights > 0 && !s->weights) fail(OEMB200_EINVAL, "n_weights > 0 but weights is NULL");
    if (!r->beta || !r->lambda || !r->niter || !r->d) fail(OEMB200_EINVAL, "result buffers beta/lambda/niter/d are required");
    if (o->maxit < 1) fail(OEMB200_EINVAL, "maxit must be >= 1");
}

// Bring an n x p column-major matrix to the device (even leading dimension so that the TMA and
// 128-bit paths apply).  Device inputs are used in place.
void to_device_matrix(Ctx &cx, const double *x, int64_t n, int p, int64_t ldx, DevMatrix &m) {
    if (is_device_ptr(x)) { m.p = x; m.ld = ldx; return; }
    size_t free_b = 0, total_b = 0;
    OEM_CUDA(cudaMemGetInfo(&free_b, &total_b));
    m.ld = n + (n & 1);
    const size_t need = (size_t)m.ld * p * 8;
    if (need + (2ull << 30) > free_b)
        fail(OEMB200_EUNSUPPORTED, "x (%.1f GB) does not fit next to the workspace on the device (%.1f GB free); "
             "use oem_fit_big (streams row chunks) or shard the rows over more GPUs", need / 1e9, free_b / 1e9);
    m.own.alloc((size_t)m.ld * p);
    if (m.ld != n) m.own.zero(cx.stream);
    h2d_block(cx, x, ldx, n, p, m.own.p, m.ld, cx.stream);      // pageable sources go through the pinned bounce ring
    m.p = m.own.p;
}
void to_device_vector(Ctx &cx, const double *v, int64_t n, DevVector &d) {
    if (is_device_ptr(v)) { d.p = v; return; }
    d.own.alloc(n + (n & 1));
    d.own.zero(cx.stream);
    d.own.upload(v, n, cx.stream);
    cx.st.h2d_bytes += n * 8;
    d.p = d.own.p;
}

void fill_common_outputs(const Setup &su, oemb200_result *res) {
    const int L = su.Lmax;
    for (int pp = 0; pp < su.P; ++pp) {
        for (int i = 0; i < L; ++i) {
            res->lambda[(size_t)pp * L + i] = i < (int)su.lam[pp].size() ? su.lam[pp][i] : 0.0;
            if (res->loss) res->loss[(size_t)pp * L + i] = 1e99;
        }
        if (res->nlam_out) res->nlam_out[pp] = su.nlam_run[pp];
    }
}

int64_t big_chunk_rows(const oemb200_opts *o, int64_t n, int p) {
    const double gigs = o->gigs > 0 ? o->gigs : 1.0;
    int64_t rows = (int64_t)(gigs * 1e9 / (8.0 * p));
    const int64_t align = 2 * gram_kt();
    rows = std::max<int64_t>(align, rows / align * align);
    return std::min<int64_t>(rows, (n + align - 1) / align * align);
}

void finish_stats(Ctx &cx, PhaseTimers &tm, size_t total_id, oemb200_result *res) {
    tm.stop(total_id);
    cx.finish();
    if (res->stats) *res->stats = cx.st;
}

// ------------------------------------------------------------------------------------------------
// oem_fit_big: one raw pass over X (row chunks, streamed from the host when X lives there)
// ------------------------------------------------------------------------------------------------
static void fit_big(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s,
                    const oemb200_opts *o, oemb200_result *res) {
    check_common(s, o, res, "gaussian");
    if (n < 1 || p < 1 || ldx < n) fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d ldx=%lld", (long long)n, p, (long long)ldx);
    const int icpt = s->intercept ? 1 : 0, q = p + icpt;
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, /*scan=*/p, /*zero_w0=*/false);      // v < nvars quirk: src/oem_big.h:445

    // bundle = [G p*p | stats 3p | sum y, sum y^2 | n]  -> one all-reduce
    const size_t nb = (size_t)p * p + 3 * (size_t)p + 3;
    DBuf<double> bundle(nb);
    bundle.zero(cx.stream);
    double *G = bundle.p, *stats = G + (size_t)p * p, *ysum = stats + 3 * (size_t)p, *nobs = ysum + 2;

    DevVector yv;
    to_device_vector(cx, y, n, yv);
    const size_t t_y = tm.start(&cx.st.ms_colstats);
    vecsum_launch(cx, yv.p, n, 0.0, ysum, false);
    tm.stop(t_y);

    // column sums, X'y and sum x^2 ride in the Gram launch (diagonal-tile CTAs)
    if (is_device_ptr(x)) {
        gram_launch(cx, x, n, p, ldx, {RowSegment{0, n, 0}}, 1, nullptr, nullptr, G, false, yv.p, stats);
    } else {
        // host X: double-buffered row chunks; H2D of chunk c+1 overlaps the kernels of chunk c
        const int64_t rows = big_chunk_rows(o, n, p);
        DBuf<double> stage[2];
        stage[0].alloc((size_t)rows * p);
        stage[1].alloc((size_t)rows * p);
        CopyLane lane;
        cudaStream_t cs = lane.s;
        cudaEvent_t *ready = lane.ready, *freed = lane.freed;
        const int64_t nchunks = (n + rows - 1) / rows;
        const bool pinned_src = is_pinned_host(x);
        auto issue_copy = [&](int64_t c) {
            const int b = (int)(c & 1);
            const int64_t r0 = c * rows, nr = std::min(rows, n - r0);
            if (c >= 2) OEM_CUDA(cudaStreamWaitEvent(cs, freed[b], 0));
            h2d_block(cx, x + r0, ldx, nr, p, stage[b].p, rows, cs);
            OEM_CUDA(cudaEventRecord(ready[b], cs));
        };
        const size_t t_h = tm.start(&cx.st.ms_h2d);   // whole streamed pass (copies overlap the kernels)
        issue_copy(0);
        if (nchunks > 1 && pinned_src) issue_copy(1);
        for (int64_t c = 0; c < nchunks; ++c) {
            const int b = (int)(c & 1);
            const int64_t r0 = c * rows, nr = std::min(rows, n - r0);
            OEM_CUDA(cudaStreamWaitEvent(cx.stream, ready[b], 0));
            gram_launch(cx, stage[b].p, nr, p, rows, {RowSegment{0, nr, 0}}, 1, nullptr, nullptr, G, c > 0, yv.p + r0, stats);
            OEM_CUDA(cudaEventRecord(freed[b], cx.stream));
            // chunk c's kernels are queued: now stage the copy after next (pinned sources: an asynchronous DMA, queued one
            // chunk further ahead; pageable sources: the reader threads fill the bounce ring while those kernels run)
            const int64_t nxt = pinned_src ? c + 2 : c + 1;
            if (nxt < nchunks) issue_copy(nxt);
        }
        tm.stop(t_h);
        cx.sync();
    }
    const double nd = (double)n;
    OEM_CUDA(cudaMemcpyAsync(nobs, &nd, 8, cudaMemcpyHostToDevice, cx.stream));
    const size_t t_ar = tm.start(&cx.st.ms_allreduce);
    cx.all_reduce(bundle.p, (int64_t)nb);
    tm.stop(t_ar);

    double n_tot = 0.0;
    OEM_CUDA(cudaMemcpyAsync(&n_tot, nobs, 8, cudaMemcpyDeviceToHost, cx.stream));
    cx.sync();
    if (!(n_tot > q)) fail(OEMB200_EUNSUPPORTED, "n <= p branch (XX' form, src/oem_big.h:363-366) is outside the hot path");

    const size_t t_as = tm.start(&cx.st.ms_assemble);
    DBuf<double> XX((size_t)q * q), XY(q), cinv(p);
    // corner = n (XX(0,0) = nobs, src/oem_big.h:527), divisor = n
    assemble_aug_launch(cx, p, icpt, s->standardize ? 1 : 0, 1, 1, G, stats, ysum, 1, nobs, nobs, XX.p, XY.p, cinv.p, nullptr);
    std::vector<double> hXY(q), hcinv(p);
    XY.download(hXY.data(), q, cx.stream);
    cinv.download(hcinv.data(), p, cx.stream);
    tm.stop(t_as);
    cx.sync();

    double lmax = 0.0;   // includes the intercept entry: src/oem_big.h:844-848
    for (int j = 0; j < q; ++j) lmax = std::max(lmax, std::fabs(hXY[j]));
    su.build_lambdas(s, lmax, false);

    PenaltyTables tb(cx, su, s, p, icpt);
    PathBuffers pb;
    const size_t t_p = tm.start(&cx.st.ms_path);
    run_paths(cx, su, tb, o, 1, XX.p, XY.p, 1.005, false, nullptr, pb);
    tm.stop(t_p);

    const int L = su.Lmax;
    fill_common_outputs(su, res);
    write_beta(su, pb.h_beta.data(), p, icpt, s->standardize ? hcinv.data() : nullptr, res);
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) res->niter[(size_t)pp * L + i] = pb.h_niter[(size_t)pp * L + i];
    *res->d = pb.h_d[0];
    finish_stats(cx, tm, t_total, res);
}

// ------------------------------------------------------------------------------------------------
// oem_fit_dense
// ------------------------------------------------------------------------------------------------
static void fit_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s,
                      const oemb200_opts *o, oemb200_result *res) {
    check_common(s, o, res, "gaussian");
    if (n < 1 || p < 1 || ldx < n) fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d ldx=%lld", (long long)n, p, (long long)ldx);
    const int flag = (s->standardize ? 1 : 0) + 2 * (s->intercept ? 1 : 0);
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, p, p, false);
    path_check_fits(cx, p, su.P, su.Lmax, su.any_group ? (int)su.unique.size() : 0, (int)su.idx.size());

    const size_t t_h = tm.start(&cx.st.ms_h2d);
    DevMatrix X;
    to_device_matrix(cx, x, n, p, ldx, X);
    DevVector yv;
    to_device_vector(cx, y, n, yv);
    tm.stop(t_h);

    // ---- pass 1: column sums, sum y, n ----
    const size_t nb1 = 3 * (size_t)p + 3;
    DBuf<double> b1(nb1);
    double *stats1 = b1.p, *ysum = stats1 + 3 * (size_t)p, *nobs = ysum + 2;
    const size_t t_c1 = tm.start(&cx.st.ms_colstats);
    if (flag != 0) colstats_launch(cx, X.p, n, p, X.ld, nullptr, nullptr, nullptr, stats1, false);
    else b1.zero(cx.stream);
    vecsum_launch(cx, yv.p, n, 0.0, ysum, false);
    const double nd = (double)n;
    OEM_CUDA(cudaMemcpyAsync(nobs, &nd, 8, cudaMemcpyHostToDevice, cx.stream));
    tm.stop(t_c1);
    cx.all_reduce(b1.p, (int64_t)nb1);
    std::vector<double> h1(nb1);
    b1.download(h1.data(), nb1, cx.stream);
    cx.sync();
    const double n_tot = h1[nb1 - 1];
    // n <= p (src/oem_dense.h:474-483, 515-521): the reference takes d from the n x n matrix XX'/n and iterates
    // u = X'(Y - X beta)/n + d beta.  XX'/n and X'X/n share their non-zero eigenvalues and that u is (dI - X'X/n) beta + X'Y/n
    // term by term, so the p x p Gram route below computes the same path (differences are rounding only); it is kept for
    // every shape instead of a second, GEMV-bound iteration kernel.

    std::vector<double> meanX(p, 0.0), scaleX(p, 1.0);
    double meanY = 0.0, scaleY = 1.0;
    const bool center_x = (flag == 2 || flag == 3);
    if (flag != 0) for (int j = 0; j < p; ++j) meanX[j] = h1[j] / n_tot;
    DBuf<double> d_mean(p);
    d_mean.upload(meanX.data(), p, cx.stream);

    // ---- y standardisation (DataStd.h:102-138; flag 2 falls through into flag 3) ----
    DBuf<double> ys;
    const double *yuse = yv.p;
    if (flag != 0) {
        const double ybar = h1[3 * (size_t)p] / n_tot;
        DBuf<double> yss(2);
        vecsum_launch(cx, yv.p, n, ybar, yss.p, false);
        cx.all_reduce(yss.p, 2);
        double h[2];
        yss.download(h, 2, cx.stream);
        cx.sync();
        const double n_invsqrt = 1.0 / std::sqrt(n_tot);
        if (flag == 1) scaleY = std::sqrt(h[1]) / std::sqrt(n_tot);        // sd_n(Y)
        else { meanY = ybar; scaleY = std::sqrt(h[1]) * n_invsqrt; }       // Y.norm() * n_invsqrt after centring
        ys.alloc(n + (n & 1));
        ys.zero(cx.stream);
        affine_launch(cx, yv.p, n, flag == 1 ? 0.0 : meanY, scaleY, ys.p);
        yuse = ys.p;
    }

    // ---- pass 2: X' ys (centred like X), centred sums of squares; pass 3: the Gram ----
    const size_t nb2 = (size_t)p * p + 2 * (size_t)p;
    DBuf<double> b2(nb2), stats2(3 * (size_t)p);
    double *G = b2.p, *xy = G + (size_t)p * p, *css = xy + p;
    // Uncentred, unscaled fits (flag 0) take X'y and the sums of squares from the Gram launch (diagonal-tile CTAs), which
    // pays for big.oem and xval.oem from p = 500 up.  Centred statistics from the Gram launch do not pay for this entry:
    // masking the tail rows of every fragment slowed the Gram more than the sweep it saved, and measured on a B200 the
    // fused launch lost at both ends -- n = 1e6 x p = 100: 2.84 ms per fit against 2.41 ms; n = 2e6 x p = 512: 28.9 ms
    // against 27.3 ms (Gram 19.9 vs 18.4 ms for a 1.2 ms sweep saved).  Every other fit takes them from a separate HBM sweep.
    const bool fused_stats = flag == 0 && p >= 256 && (double)n * p >= 268435456.0;
    if (fused_stats) {
        gram_launch(cx, X.p, n, p, X.ld, {RowSegment{0, n, 0}}, 1, nullptr, nullptr, G, false, yuse, stats2.p);
        OEM_CUDA(cudaMemcpyAsync(xy, stats2.p + (size_t)p, (size_t)p * 8, cudaMemcpyDeviceToDevice, cx.stream));
        OEM_CUDA(cudaMemcpyAsync(css, stats2.p + 2 * (size_t)p, (size_t)p * 8, cudaMemcpyDeviceToDevice, cx.stream));
    } else {
        const size_t t_c2 = tm.start(&cx.st.ms_colstats);
        colstats_launch(cx, X.p, n, p, X.ld, yuse, nullptr, center_x ? d_mean.p : nullptr, stats2.p, false);
        OEM_CUDA(cudaMemcpyAsync(xy, stats2.p, (size_t)p * 8, cudaMemcpyDeviceToDevice, cx.stream));
        if (flag == 1) {   // sd about the mean although X itself is not centred
            DBuf<double> stats3(3 * (size_t)p);
            colstats_launch(cx, X.p, n, p, X.ld, nullptr, nullptr, d_mean.p, stats3.p, false);
            OEM_CUDA(cudaMemcpyAsync(css, stats3.p + 2 * (size_t)p, (size_t)p * 8, cudaMemcpyDeviceToDevice, cx.stream));
            cx.sync();
        } else {
            OEM_CUDA(cudaMemcpyAsync(css, stats2.p + 2 * (size_t)p, (size_t)p * 8, cudaMemcpyDeviceToDevice, cx.stream));
        }
        tm.stop(t_c2);
        gram_launch(cx, X.p, n, p, X.ld, {RowSegment{0, n, 0}}, 1, center_x ? d_mean.p : nullptr, nullptr, G, false);
    }
    const size_t t_ar = tm.start(&cx.st.ms_allreduce);
    cx.all_reduce(b2.p, (int64_t)nb2);
    tm.stop(t_ar);

    const size_t t_as = tm.start(&cx.st.ms_assemble);
    DBuf<double> XX((size_t)p * p), XY(p), d_scalex(p);
    assemble_dense_launch(cx, p, flag, n_tot, G, xy, css, XX.p, XY.p, d_scalex.p);
    std::vector<double> hXY(p);
    XY.download(hXY.data(), p, cx.stream);
    d_scalex.download(scaleX.data(), p, cx.stream);
    tm.stop(t_as);
    cx.sync();

    double lmax = 0.0;
    for (int j = 0; j < p; ++j) lmax = std::max(lmax, std::fabs(hXY[j]));
    lmax *= scaleY;                                   // src/oem_dense.cpp:176
    su.build_lambdas(s, lmax, false);
    PenaltyTables tb(cx, su, s, p, 0, scaleY);
    PathBuffers pb;
    const size_t t_p = tm.start(&cx.st.ms_path);
    run_paths(cx, su, tb, o, 1, XX.p, XY.p, 1.005, o->accelerate != 0, nullptr, pb);
    tm.stop(t_p);

    // ---- recover (DataStd.h:269-293) ----
    const int L = su.Lmax;
    fill_common_outputs(su, res);
    memset(res->beta, 0, sizeof(double) * (size_t)su.P * (p + 1) * L);
    DBuf<double> d_b, d_eta, d_l2;
    // losses of all (penalty, lambda) columns in ONE pass over X when the TMA can address it (else per-lambda sweeps)
    // (which route a rank takes depends on its local pointer alignment; both routes end in ONE all-reduce of the same P x L
    // vector, so ranks may differ)
    const bool loss_gemm = s->compute_loss && res->loss && !(X.ld & 1) && !(reinterpret_cast<uintptr_t>(X.p) & 15);
    std::vector<double> loss_local((size_t)su.P * L, 0.0);
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const double *raw = &pb.h_beta[((size_t)pp * L + i) * p];
            double *out = res->beta + ((size_t)pp * L + i) * (p + 1);
            double b0 = 0.0;
            for (int j = 0; j < p; ++j) {
                double c = raw[j];
                if (flag == 1 || flag == 3) c /= scaleX[j];
                if (flag != 0) c *= scaleY;
                out[1 + j] = c;
            }
            if (flag == 2 || flag == 3) {
                double acc = 0.0;
                for (int j = 0; j < p; ++j) acc += out[1 + j] * meanX[j];
                b0 = meanY - acc;
            }
            out[0] = b0;
            res->niter[(size_t)pp * L + i] = pb.h_niter[(size_t)pp * L + i];
            if (s->compute_loss && res->loss && !loss_gemm) {
                // get_loss(): ||Y_std - X_std beta_std||^2 (src/oem_dense.h:759-770) as one more X b pass:
                // X_std b = X (b / s) - sum_j m_j b_j / s_j   (sweep fallback for X the TMA cannot address)
                std::vector<double> bs(p);
                double off = 0.0;
                for (int j = 0; j < p; ++j) {
                    bs[j] = (flag == 1 || flag == 3) ? raw[j] / scaleX[j] : raw[j];
                    if (center_x) off -= bs[j] * meanX[j];
                }
                if (!d_b.p) { d_b.alloc(p); d_eta.alloc(n + (n & 1)); d_l2.alloc(2); }
                d_b.upload(bs.data(), p, cx.stream);
                // eta = ys - X_std b  is formed as  -(X bs + off) + ys  via the resid output of the xb epilogue
                xb_launch(cx, X.p, n, p, X.ld, d_b.p, off, nullptr, d_eta.p, nullptr, nullptr, nullptr, false);
                affine_launch(cx, d_eta.p, n, 0.0, -1.0, d_eta.p);
                axpy_launch(cx, n, 1.0, yuse, d_eta.p);
                vecsum_launch(cx, d_eta.p, n, 0.0, d_l2.p, false);
                double h[2];
                d_l2.download(h, 2, cx.stream);
                cx.sync();
                loss_local[(size_t)pp * L + i] = h[1];      // summed over ranks below, in the same one all-reduce as the GEMM route
            }
        }
    if (loss_gemm) {
        // get_loss(): ||Y_std - X_std beta_std||^2 (src/oem_dense.h:759-770).  X_std b = X (b / s) - sum_j m_j b_j / s_j, so
        // every column is (y_std - b0' - X b')^2 summed over rows: the CV-scoring GEMM with its squared-error moments.
        const int nc = su.P * L, ncld = cv_ncld(nc);
        std::vector<double> hB((size_t)p * ncld, 0.0), hb0(ncld, 0.0);
        for (int pp = 0; pp < su.P; ++pp)
            for (int i = 0; i < su.nlam_run[pp]; ++i) {
                const double *raw = &pb.h_beta[((size_t)pp * L + i) * p];
                const int c = pp * L + i;
                double off = 0.0;
                for (int j = 0; j < p; ++j) {
                    const double b = (flag == 1 || flag == 3) ? raw[j] / scaleX[j] : raw[j];
                    hB[(size_t)j * ncld + c] = b;
                    if (center_x) off -= b * meanX[j];
                }
                hb0[c] = off;
            }
        DBuf<double> dB(hB.size()), db0(hb0.size()), out3(3 * (size_t)nc);
        dB.upload(hB.data(), hB.size(), cx.stream);
        db0.upload(hb0.data(), hb0.size(), cx.stream);
        std::vector<std::array<int64_t, 3>> cs{{0, n, n}};
        cvscore_launch(cx, X.p, n, p, X.ld, yuse, nullptr, 1, cs, dB.p, db0.p, nc, false, out3.p);
        std::vector<double> h3(3 * (size_t)nc);
        out3.download(h3.data(), h3.size(), cx.stream);
        cx.sync();
        for (int c = 0; c < nc; ++c) loss_local[c] = h3[c] * h3[nc + c];   // count * mean = sum
    }
    if (s->compute_loss && res->loss) {
        if (cx.distributed()) {
            DBuf<double> dt(loss_local.size());
            dt.upload(loss_local.data(), loss_local.size(), cx.stream);
            cx.all_reduce(dt.p, (int64_t)loss_local.size());
            dt.download(loss_local.data(), loss_local.size(), cx.stream);
            cx.sync();
        }
        for (int pp = 0; pp < su.P; ++pp)
            for (int i = 0; i < su.nlam_run[pp]; ++i) res->loss[(size_t)pp * L + i] = loss_local[(size_t)pp * L + i];
    }
    *res->d = pb.h_d[0];
    finish_stats(cx, tm, t_total, res);
}

// ------------------------------------------------------------------------------------------------
// oem_xtx
// ------------------------------------------------------------------------------------------------
static void fit_xtx(const double *xtx, const double *xty, int p, const oemb200_spec *s, const double *scale_factor,
                    int n_sf, const oemb200_opts *o, oemb200_result *res) {
    check_common(s, o, res, "gaussian");
    if (p < 1 || !xtx || !xty) fail(OEMB200_EINVAL, "xtx / xty missing");
    if (n_sf != 0 && n_sf != p) fail(OEMB200_EINVAL, "scale_factor must have length p");
    if (n_sf != 0 && (!scale_factor || is_device_ptr(scale_factor)))
        fail(OEMB200_EINVAL, "scale_factor must be a host vector (it is read on the host)");
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, p, p, false);
    DBuf<double> XXin, XYin, XX((size_t)p * p), XY(p), sinv;
    const double *pxx = xtx, *pxy = xty;
    if (!is_device_ptr(xtx)) { XXin.alloc((size_t)p * p); XXin.upload(xtx, (size_t)p * p, cx.stream); pxx = XXin.p; cx.st.h2d_bytes += (int64_t)p * p * 8; }
    if (!is_device_ptr(xty)) { XYin.alloc(p); XYin.upload(xty, p, cx.stream); pxy = XYin.p; cx.st.h2d_bytes += p * 8; }
    std::vector<double> hs;
    if (n_sf) {
        hs.resize(p);
        for (int j = 0; j < p; ++j) hs[j] = 1.0 / scale_factor[j];
        sinv.alloc(p);
        sinv.upload(hs.data(), p, cx.stream);
    }
    const size_t t_as = tm.start(&cx.st.ms_assemble);
    scale_sym_launch(cx, p, n_sf ? sinv.p : nullptr, pxx, pxy, XX.p, XY.p);
    std::vector<double> hXY(p);
    XY.download(hXY.data(), p, cx.stream);
    tm.stop(t_as);
    cx.sync();
    double lmax = 0.0;
    for (int j = 0; j < p; ++j) lmax = std::max(lmax, std::fabs(hXY[j]));
    su.build_lambdas(s, lmax, false);
    PenaltyTables tb(cx, su, s, p, 0);
    PathBuffers pb;
    const size_t t_p = tm.start(&cx.st.ms_path);
    run_paths(cx, su, tb, o, 1, XX.p, XY.p, 1.005, false, n_sf ? sinv.p : nullptr, pb);
    tm.stop(t_p);
    const int L = su.Lmax;
    fill_common_outputs(su, res);
    memset(res->beta, 0, sizeof(double) * (size_t)su.P * p * L);
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            memcpy(res->beta + ((size_t)pp * L + i) * p, &pb.h_beta[((size_t)pp * L + i) * p], sizeof(double) * p);
            res->niter[(size_t)pp * L + i] = pb.h_niter[(size_t)pp * L + i];
        }
    *res->d = pb.h_d[0];
    finish_stats(cx, tm, t_total, res);
}

void fit_logistic(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s,
                  const oemb200_opts *o, oemb200_result *res, SlabCache *cache);
void fit_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *y,
                const oemb200_spec *s, const oemb200_opts *o, oemb200_result *res);
void fit_logistic_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *y,
                         const oemb200_spec *s, const oemb200_opts *o, oemb200_result *res);
void predict_sparse_entry(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *beta,
                          int nrows, int L, int type, double *out, int64_t ldo, const oemb200_opts *o, oemb200_stats *stats);
void fit_xval(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s, int nfolds,
              const int *foldid, const char *type_measure, const oemb200_opts *o, oemb200_result *res);
void fit_xval_logistic(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s, int nfolds,
                       const int *foldid, const char *type_measure, const oemb200_opts *o, oemb200_result *res);
void fit_xval_big(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s, int nfolds,
                  const int *foldid, const char *type_measure, const oemb200_opts *o, oemb200_result *res);

template <typename F>
static int guarded(F &&f) {
    try {
        f();
        return OEMB200_OK;
    } catch (const Error &e) {
        g_last_error = e.what();
        cudaGetLastError();
        return e.code;
    } catch (const std::exception &e) {
        g_last_error = e.what();
        return OEMB200_EINVAL;
    } catch (...) {
        g_last_error = "unknown error";
        return OEMB200_EINVAL;
    }
}

}  // namespace oemb200

using namespace oemb200;

// ------------------------------------------------------------------------------------------------
// predict.oem (R/methods.R:48-119, 346-366): newx %*% nbeta (+ intercept row), optional logistic response
// ------------------------------------------------------------------------------------------------
static void predict_entry(const double *x, int64_t n, int p, int64_t ldx, const double *beta, int nrows, int L, int type,
                          double *out, int64_t ldo, const oemb200_opts *o, oemb200_stats *stats) {
    if (!x || !beta || !out || !o) fail(OEMB200_EINVAL, "x / beta / out / opts must not be NULL");
    if (n < 1 || p < 1 || ldx < n || L < 1 || ldo < n)
        fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d ldx=%lld L=%d ldo=%lld", (long long)n, p, (long long)ldx, L, (long long)ldo);
    if (nrows != p && nrows != p + 1)
        fail(OEMB200_EINVAL, "beta has %d rows; newx has %d columns (expected %d or %d)", nrows, p, p, p + 1);   // R/methods.R:115-116
    if (type != 0 && type != 1) fail(OEMB200_EINVAL, "type must be 0 (link) or 1 (response)");
    if (is_device_ptr(beta)) fail(OEMB200_EINVAL, "beta must be a host pointer");
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    const size_t t_h = tm.start(&cx.st.ms_h2d);
    DevMatrix X;
    to_device_matrix(cx, x, n, p, ldx, X);
    if ((X.ld & 1) || (reinterpret_cast<uintptr_t>(X.p) & 15)) {
        // device-resident newx that the TMA descriptor cannot address (odd leading dimension / unaligned base): repack
        const int64_t ld2 = n + (n & 1);
        X.own.alloc((size_t)ld2 * p);
        if (ld2 != n) X.own.zero(cx.stream);
        OEM_CUDA(cudaMemcpy2DAsync(X.own.p, (size_t)ld2 * 8, X.p, (size_t)X.ld * 8, (size_t)n * 8, p, cudaMemcpyDeviceToDevice,
                                   cx.stream));
        X.p = X.own.p;
        X.ld = ld2;
    }
    tm.stop(t_h);
    const int icpt = nrows - p, ncld = cv_ncld(L);
    std::vector<double> hB((size_t)p * ncld, 0.0), hb0(ncld, 0.0);
    for (int c = 0; c < L; ++c) {
        const double *col = beta + (size_t)c * nrows;
        if (icpt) hb0[c] = col[0];
        for (int j = 0; j < p; ++j) hB[(size_t)j * ncld + c] = col[icpt + j];
    }
    DBuf<double> dB(hB.size()), db0(hb0.size()), dout;
    dB.upload(hB.data(), hB.size(), cx.stream);
    db0.upload(hb0.data(), hb0.size(), cx.stream);
    const bool out_dev = is_device_ptr(out);
    double *po = out;
    int64_t ldp = ldo;
    if (!out_dev) {
        dout.alloc((size_t)n * L);
        po = dout.p;
        ldp = n;
    }
    predict_launch(cx, X.p, n, p, X.ld, dB.p, db0.p, L, type == 1, po, ldp);
    if (!out_dev) {
        OEM_CUDA(cudaMemcpy2DAsync(out, (size_t)ldo * 8, po, (size_t)n * 8, (size_t)n * 8, L, cudaMemcpyDeviceToHost, cx.stream));
        cx.st.d2h_bytes += (int64_t)n * L * 8;
    }
    tm.stop(t_total);
    cx.finish();
    if (stats) *stats = cx.st;
}

extern "C" {

const char *oemb200_last_error(void) { return g_last_error.c_str(); }
const char *oemb200_version(void) { return "oem_b200 0.2 (sm_100a)"; }
int oemb200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
void oemb200_default_opts(oemb200_opts *o) {
    if (!o) return;
    memset(o, 0, sizeof *o);
    o->maxit = 500; o->tol = 1e-7; o->irls_maxit = 100; o->irls_tol = 1e-3; o->ncores = -1;
    o->hessian_full = 0; o->accelerate = 0; o->gigs = 4.0; o->device = -1; o->world = 1;
}
int oemb200_penalty_id(const char *name) { return penalty_id(name); }
int oemb200_nlambda_max(const oemb200_spec *s) {
    if (!s) return 0;
    if (s->n_lambda && s->lambda && s->n_lambda[0] >= 1) return s->n_lambda[0];
    return s->nlambda;
}

int oemb200_lambda_grid(double lmax, int nlambda, double lambda_min_ratio, double *out) {
    return guarded([&] {
        if (nlambda < 1 || !out) fail(OEMB200_EINVAL, "lambda_grid: nlambda < 1 or NULL output");
        const std::vector<double> v = lambda_base(lmax, nlambda, lambda_min_ratio);
        memcpy(out, v.data(), sizeof(double) * v.size());
    });
}
int oemb200_stop_rule(const double *cur, const double *prev, int q, double tol) {
    std::vector<double> a(cur, cur + q), b(prev, prev + q);
    return stop_rule_host(a, b, tol) ? 1 : 0;
}
void oemb200_release_cache(void) { pool_release_all(); release_host_stager(); }

int oemb200_fit_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *spec,
                      const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] { fit_dense(x, n, p, ldx, y, spec, opts, res); });
}
int oemb200_xtx(const double *xtx, const double *xty, int p, const oemb200_spec *spec, const double *scale_factor,
                int n_scale_factor, const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] { fit_xtx(xtx, xty, p, spec, scale_factor, n_scale_factor, opts, res); });
}
int oemb200_fit_big(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *spec,
                    const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] { fit_big(x, n, p, ldx, y, spec, opts, res); });
}
int oemb200_fit_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *y,
                       const oemb200_spec *spec, const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] { fit_sparse(row_idx, col_ptr, values, n, p, y, spec, opts, res); });
}
int oemb200_fit_logistic_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *y,
                                const oemb200_spec *spec, const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] { fit_logistic_sparse(row_idx, col_ptr, values, n, p, y, spec, opts, res); });
}
int oemb200_fit_logistic_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y,
                               const oemb200_spec *spec, const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] { fit_logistic(x, n, p, ldx, y, spec, opts, res, nullptr); });
}
int oemb200_xval_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *spec,
                       int nfolds, const int *foldid, const char *type_measure, const oemb200_opts *opts,
                       oemb200_result *res) {
    return guarded([&] { fit_xval(x, n, p, ldx, y, spec, nfolds, foldid, type_measure, opts, res); });
}
int oemb200_xval_big(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *spec, int nfolds,
                     const int *foldid, const char *type_measure, const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] { fit_xval_big(x, n, p, ldx, y, spec, nfolds, foldid, type_measure, opts, res); });
}
int oemb200_xval_logistic_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *spec,
                                int nfolds, const int *foldid, const char *type_measure, const oemb200_opts *opts,
                                oemb200_result *res) {
    return guarded([&] { fit_xval_logistic(x, n, p, ldx, y, spec, nfolds, foldid, type_measure, opts, res); });
}

int oemb200_predict(const double *x, int64_t n, int p, int64_t ldx, const double *beta, int beta_rows, int nlambda, int type,
                    double *out, int64_t ldo, const oemb200_opts *opts, oemb200_stats *stats) {
    return guarded([&] { predict_entry(x, n, p, ldx, beta, beta_rows, nlambda, type, out, ldo, opts, stats); });
}

int oemb200_predict_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *beta,
                           int beta_rows, int nlambda, int type, double *out, int64_t ldo, const oemb200_opts *opts,
                           oemb200_stats *stats) {
    return guarded([&] { predict_sparse_entry(row_idx, col_ptr, values, n, p, beta, beta_rows, nlambda, type, out, ldo, opts, stats); });
}

// ---------------- device-resident matrix handle ----------------
}  // extern "C"

struct oemb200_matrix {
    double *dev = nullptr;
    int64_t n = 0, ld = 0;
    int p = 0, device = 0;
    int64_t h2d_bytes = 0;
    double ms_upload = 0.0;
    mutable SlabCache slab;      // built by the first logistic fit on the handle
};

namespace {
oemb200_matrix *matrix_alloc(Ctx &cx, int64_t n, int p) {
    if (n < 1 || p < 1) fail(OEMB200_EINVAL, "matrix: bad dimensions n=%lld p=%d", (long long)n, p);
    oemb200_matrix *m = new oemb200_matrix();
    m->n = n; m->p = p; m->ld = n + (n & 1); m->device = cx.device;
    const size_t bytes = (size_t)m->ld * p * 8;
    if (cudaMalloc(reinterpret_cast<void **>(&m->dev), bytes) != cudaSuccess) {
        cudaGetLastError();
        pool_release_all();
        if (cudaMalloc(reinterpret_cast<void **>(&m->dev), bytes) != cudaSuccess) {
            cudaGetLastError();
            delete m;
            fail(OEMB200_ECUDA, "matrix: cudaMalloc of %.2f GB failed", bytes / 1e9);
        }
    }
    if (m->ld != n) OEM_CUDA(cudaMemsetAsync(m->dev, 0, bytes, cx.stream));
    return m;
}
// upload in row chunks of `gigs` GB so that the bounce ring (pageable sources) overlaps its DMA with the next fill
void matrix_upload(Ctx &cx, oemb200_matrix *m, const double *x, int64_t ldx, double gigs) {
    cudaEvent_t e0, e1;
    OEM_CUDA(cudaEventCreate(&e0)); OEM_CUDA(cudaEventCreate(&e1));
    OEM_CUDA(cudaEventRecord(e0, cx.stream));
    if (is_device_ptr(x)) {
        OEM_CUDA(cudaMemcpy2DAsync(m->dev, (size_t)m->ld * 8, x, (size_t)ldx * 8, (size_t)m->n * 8, m->p, cudaMemcpyDeviceToDevice, cx.stream));
    } else {
        int64_t rows = (int64_t)((gigs > 0 ? gigs : 1.0) * 1e9 / (8.0 * m->p));
        rows = std::max<int64_t>(1024, rows);
        for (int64_t r0 = 0; r0 < m->n; r0 += rows)
            h2d_block(cx, x + r0, ldx, std::min(rows, m->n - r0), m->p, m->dev + r0, m->ld, cx.stream);
    }
    OEM_CUDA(cudaEventRecord(e1, cx.stream));
    cx.sync();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    m->ms_upload = ms;
    m->h2d_bytes = cx.st.h2d_bytes;
}
void check_handle(const oemb200_matrix *m) {
    if (!m || !m->dev) fail(OEMB200_EINVAL, "matrix handle is NULL or destroyed");
}
// the *_h entries run on the handle's device
struct HandleOpts {
    oemb200_opts o;
    HandleOpts(const oemb200_matrix *m, const oemb200_opts *in) {
        if (!in) fail(OEMB200_EINVAL, "opts must not be NULL");
        o = *in;
        if (o.device >= 0 && o.device != m->device)
            fail(OEMB200_EINVAL, "opts.device = %d but the matrix lives on device %d", o.device, m->device);
        o.device = m->device;
    }
};
}  // namespace

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

extern "C" {

int oemb200_matrix_create(const double *x, int64_t n, int p, int64_t ldx, const oemb200_opts *opts, oemb200_matrix **out) {
    return guarded([&] {
        if (!x || !out || !opts) fail(OEMB200_EINVAL, "matrix_create: x / opts / out must not be NULL");
        if (ldx < n) fail(OEMB200_EINVAL, "matrix_create: ldx < n");
        Ctx cx(opts);
        oemb200_matrix *m = matrix_alloc(cx, n, p);
        try {
            matrix_upload(cx, m, x, ldx, opts->gigs);
        } catch (...) {
            cudaFree(m->dev);
            delete m;
            throw;
        }
        *out = m;
    });
}

int oemb200_matrix_create_from_file(const char *bk_path, int64_t n, int p, const oemb200_opts *opts, oemb200_matrix **out) {
    return guarded([&] {
        if (!bk_path || !out || !opts) fail(OEMB200_EINVAL, "matrix_create_from_file: path / opts / out must not be NULL");
        if (n < 1 || p < 1) fail(OEMB200_EINVAL, "matrix_create_from_file: bad dimensions n=%lld p=%d", (long long)n, p);
        // the backing file of a bigmemory file-backed matrix: raw column-major doubles, no header (R/big_oem.R:87-90)
        const int fd = open(bk_path, O_RDONLY);
        if (fd < 0) fail(OEMB200_EINVAL, "cannot open %s", bk_path);
        struct stat sb;
        const size_t need = (size_t)n * p * 8;
        if (fstat(fd, &sb) != 0 || (size_t)sb.st_size < need) {
            close(fd);
            fail(OEMB200_EINVAL, "%s holds %lld bytes, an %lld x %d matrix of doubles needs %zu", bk_path,
                 (long long)sb.st_size, (long long)n, p, need);
        }
        void *map = mmap(nullptr, need, PROT_READ, MAP_SHARED, fd, 0);
        close(fd);
        if (map == MAP_FAILED) fail(OEMB200_EINVAL, "cannot map %s", bk_path);
        madvise(map, need, MADV_SEQUENTIAL);
        oemb200_matrix *m = nullptr;
        try {
            Ctx cx(opts);
            m = matrix_alloc(cx, n, p);
            matrix_upload(cx, m, static_cast<const double *>(map), n, opts->gigs);
        } catch (...) {
            munmap(map, need);
            if (m) { cudaFree(m->dev); delete m; }
            throw;
        }
        munmap(map, need);
        *out = m;
    });
}

int oemb200_matrix_destroy(oemb200_matrix *m) {
    return guarded([&] {
        if (!m) return;
        int prev = -1;
        cudaGetDevice(&prev);
        cudaSetDevice(m->device);
        if (m->slab.slabs) cudaFree(m->slab.slabs);
        if (m->dev) cudaFree(m->dev);
        if (prev >= 0) cudaSetDevice(prev);
        cudaGetLastError();
        delete m;
    });
}

int oemb200_matrix_info(const oemb200_matrix *m, int64_t *n, int *p, int64_t *ld, const double **dev_ptr, int64_t *h2d_bytes,
                        double *ms_upload) {
    return guarded([&] {
        check_handle(m);
        if (n) *n = m->n;
        if (p) *p = m->p;
        if (ld) *ld = m->ld;
        if (dev_ptr) *dev_ptr = m->dev;
        if (h2d_bytes) *h2d_bytes = m->h2d_bytes;
        if (ms_upload) *ms_upload = m->ms_upload;
    });
}

int oemb200_fit_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec, const oemb200_opts *opts,
                        oemb200_result *res) {
    return guarded([&] { check_handle(x); HandleOpts h(x, opts); fit_dense(x->dev, x->n, x->p, x->ld, y, spec, &h.o, res); });
}
int oemb200_fit_big_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec, const oemb200_opts *opts,
                      oemb200_result *res) {
    return guarded([&] { check_handle(x); HandleOpts h(x, opts); fit_big(x->dev, x->n, x->p, x->ld, y, spec, &h.o, res); });
}
int oemb200_fit_logistic_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec, const oemb200_opts *opts,
                                 oemb200_result *res) {
    return guarded([&] {
        check_handle(x);
        HandleOpts h(x, opts);
        fit_logistic(x->dev, x->n, x->p, x->ld, y, spec, &h.o, res, &x->slab);
    });
}
int oemb200_xval_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec, int nfolds, const int *foldid,
                         const char *type_measure, const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] {
        check_handle(x);
        HandleOpts h(x, opts);
        fit_xval(x->dev, x->n, x->p, x->ld, y, spec, nfolds, foldid, type_measure, &h.o, res);
    });
}
int oemb200_xval_logistic_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec, int nfolds,
                                  const int *foldid, const char *type_measure, const oemb200_opts *opts, oemb200_result *res) {
    return guarded([&] {
        check_handle(x);
        HandleOpts h(x, opts);
        fit_xval_logistic(x->dev, x->n, x->p, x->ld, y, spec, nfolds, foldid, type_measure, &h.o, res);
    });
}
int oemb200_predict_h(const oemb200_matrix *x, const double *beta, int beta_rows, int nlambda, int type, double *out,
                      int64_t ldo, const oemb200_opts *opts, oemb200_stats *stats) {
    return guarded([&] {
        check_handle(x);
        HandleOpts h(x, opts);
        predict_entry(x->dev, x->n, x->p, x->ld, beta, beta_rows, nlambda, type, out, ldo, &h.o, stats);
    });
}

// ---------------- phase-level entries ----------------
static void phase_ctx_opts(oemb200_opts &o, void *stream) {
    oemb200_default_opts(&o);
    o.stream = stream;
}
static double elapsed_ms(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}
#define OEM_PHASE_TIMED(body)                                                    \
    oemb200_opts o_; phase_ctx_opts(o_, stream);                                 \
    Ctx cx(&o_);                                                                 \
    cudaEvent_t ea, eb;                                                          \
    OEM_CUDA(cudaEventCreate(&ea)); OEM_CUDA(cudaEventCreate(&eb));              \
    OEM_CUDA(cudaEventRecord(ea, cx.stream));                                    \
    body;                                                                        \
    OEM_CUDA(cudaEventRecord(eb, cx.stream));                                    \
    cx.sync();                                                                   \
    if (ms_out) *ms_out = elapsed_ms(ea, eb);                                    \
    cudaEventDestroy(ea); cudaEventDestroy(eb);

int oemb200_gram(const double *x_dev, int64_t n, int p, int64_t ldx, const double *mean_dev, const double *row_w_dev,
                 double *g_dev, void *stream, double *ms_out) {
    return guarded([&] {
        OEM_PHASE_TIMED(gram_launch(cx, x_dev, n, p, ldx, {RowSegment{0, n, 0}}, 1, mean_dev, row_w_dev, g_dev, false));
    });
}
int oemb200_colstats(const double *x_dev, int64_t n, int p, int64_t ldx, const double *v0_dev, const double *v1_dev,
                     double *out_dev, void *stream, double *ms_out) {
    return guarded([&] { OEM_PHASE_TIMED(colstats_launch(cx, x_dev, n, p, ldx, v0_dev, v1_dev, nullptr, out_dev, false)); });
}
int oemb200_xb_logistic(const double *x_dev, int64_t n, int p, int64_t ldx, const double *b_dev, double b0,
                        const double *y_dev, double *prob_dev, double *resid_dev, double *w_dev, void *stream,
                        double *ms_out) {
    return guarded([&] {
        OEM_PHASE_TIMED(xb_launch(cx, x_dev, n, p, ldx, b_dev, b0, y_dev, nullptr, prob_dev, resid_dev, w_dev, true));
    });
}
int oemb200_logit_slab_pass(const double *x_dev, int64_t n, int p, int64_t ldx, const double *b_dev, double b0,
                            const double *y_dev, double *prob_dev, double *w_dev, double *grad_dev, int reps, void *stream,
                            double *ms_out, double *ms_relayout_out) {
    return guarded([&] {
        if (!x_dev || !b_dev || !y_dev || !grad_dev || n < 1 || p < 1 || ldx < n) fail(OEMB200_EINVAL, "logit_slab_pass: bad arguments");
        if (!logit_slab_rows(p)) fail(OEMB200_EUNSUPPORTED, "the slab kernel covers 8 <= p <= 2048 (p = %d)", p);
        oemb200_opts o_; phase_ctx_opts(o_, stream);
        Ctx cx(&o_);
        cudaEvent_t e0, e1, e2;
        OEM_CUDA(cudaEventCreate(&e0)); OEM_CUDA(cudaEventCreate(&e1)); OEM_CUDA(cudaEventCreate(&e2));
        DBuf<double> slabs(logit_slab_doubles(n, p)), d_b0(1);
        OEM_CUDA(cudaMemcpyAsync(d_b0.p, &b0, 8, cudaMemcpyHostToDevice, cx.stream));
        OEM_CUDA(cudaEventRecord(e0, cx.stream));
        logit_slab_relayout(cx, x_dev, n, p, ldx, slabs.p);
        OEM_CUDA(cudaEventRecord(e1, cx.stream));
        const int nrep = reps < 1 ? 1 : reps;
        for (int r = 0; r < nrep; ++r) logit_slab_launch(cx, slabs.p, n, p, b_dev, d_b0.p, y_dev, prob_dev, w_dev, grad_dev);
        OEM_CUDA(cudaEventRecord(e2, cx.stream));
        cx.sync();
        if (ms_relayout_out) *ms_relayout_out = elapsed_ms(e0, e1);
        if (ms_out) *ms_out = elapsed_ms(e1, e2) / nrep;
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
    });
}
int oemb200_logit_fold_pass(const double *x_dev, int64_t n, int p, int64_t ldx, const double *b_dev, const double *b0_dev,
                            const double *y_dev, const int *fold_dev, int M, const int *conv_dev, double *grad_dev, int reps,
                            void *stream, double *ms_out, double *ms_relayout_out, int *sweeps_out) {
    return guarded([&] {
        if (!x_dev || !b_dev || !b0_dev || !y_dev || !fold_dev || !grad_dev || n < 1 || p < 1 || ldx < n || M < 1)
            fail(OEMB200_EINVAL, "logit_fold_pass: bad arguments");
        if (!logit_fold_models(p)) fail(OEMB200_EUNSUPPORTED, "the fused fold pass covers 8 <= p <= 2048 (p = %d)", p);
        oemb200_opts o_; phase_ctx_opts(o_, stream);
        Ctx cx(&o_);
        cudaEvent_t e0, e1, e2;
        OEM_CUDA(cudaEventCreate(&e0)); OEM_CUDA(cudaEventCreate(&e1)); OEM_CUDA(cudaEventCreate(&e2));
        DBuf<double> slabs(logit_fold_doubles(n, p));
        OEM_CUDA(cudaEventRecord(e0, cx.stream));
        logit_fold_relayout(cx, x_dev, n, p, ldx, slabs.p);
        OEM_CUDA(cudaEventRecord(e1, cx.stream));
        const int nrep = reps < 1 ? 1 : reps;
        int sweeps = 0;
        for (int r = 0; r < nrep; ++r)
            sweeps = logit_fold_launch(cx, slabs.p, n, p, b_dev, b0_dev, y_dev, fold_dev, M, conv_dev, nullptr, nullptr, grad_dev);
        OEM_CUDA(cudaEventRecord(e2, cx.stream));
        cx.sync();
        if (ms_relayout_out) *ms_relayout_out = elapsed_ms(e0, e1);
        if (ms_out) *ms_out = elapsed_ms(e1, e2) / nrep;
        if (sweeps_out) *sweeps_out = sweeps;
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
    });
}
int oemb200_top_eig(const double *xx_dev, int q, double *lambda_max_out, int *steps_out, void *stream) {
    return guarded([&] {
        oemb200_opts o_; phase_ctx_opts(o_, stream);
        Ctx cx(&o_);
        DBuf<double> d(1), xy(q);
        DBuf<int> lz(1);
        xy.zero(cx.stream);
        PathProblem pp;
        pp.q = q; pp.ngram = 1; pp.XX = xx_dev; pp.XY = xy.p; pp.d = d.p; pp.compute_eig = true;
        pp.eig_factor = 1.0; pp.Lmax = 1; pp.lanczos_steps = lz.p;
        path_launch(cx, pp);
        double h; int k;
        d.download(&h, 1, cx.stream);
        lz.download(&k, 1, cx.stream);
        cx.sync();
        if (lambda_max_out) *lambda_max_out = h;
        if (steps_out) *steps_out = k;
    });
}

}  // extern "C"
