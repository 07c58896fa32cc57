// entry_logistic.cu -- host drivers of oem_fit_logistic_dense (src/oem_logistic_dense.cpp:29-313, solver
// src/oem_logistic_dense.h:721-1036) and oem_fit_logistic_sparse (below) on the sm_100a kernels.
//
// Per IRLS iteration the reference makes two passes over X:
//   prob = sigma(X (beta o w) + beta0)        (oem_logistic_dense.h:864-949)
//   grad = [sum(y-prob), X'(y-prob) o w] / n  (oem_logistic_dense.h:970-992)
// Here both come out of ONE sweep of a row-slab copy of X (logit_slab.cu; built once per fit), or, for shapes the
// slab kernel does not cover, out of the two HBM-bound sweeps xb_kernel + colstats_kernel.  When the Hessian bound is
// (re)built, X'WX runs on the FP64 tensor pipe (gram_syrk_kernel; the row weight fused into the fragment load for
// hessian.type = "full") and the Lanczos eigenvalue inside the path kernel.
//
// The IRLS state never leaves the device.  An iteration of the dense driver is three launches on one stream: the data pass
// (+ its partial-sum kernel), in row-sharded runs the sum of the (p+1)-vector gradient (comm.cu), and the path launch, which
// forms XY = XX beta + grad, runs the inner OEM loop, applies the outer stop rule and leaves the next pass's coefficients
// (IrlsLoop::path_step); their phase clocks are kept on the device.  The only host round trip per IRLS iteration is ONE
// event synchronisation that reads the stop-rule verdict from pinned memory (IrlsLoop, host_common.h, which the sparse
// and the binomial xval drivers share), and it is hidden behind the next iteration, which is enqueued one ahead and
// predicated on the device-side verdict.  logistic_init (host_common.h) is the init step of both drivers of this file.
// The reference's quirks are kept (SURVEY.md Appendix B item 5): the data pass is skipped on the first IRLS
// iteration of a warm lambda, W is clamped at index = IRLS counter, eigen factor 1.0005.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include "host_common.h"

namespace oemb200 {

__global__ void clamp_one_kernel(double *w, long long idx, double lo, const int *skip) {
    if (skip && *skip) return;
    if (w[idx] < lo) w[idx] = lo;
}

// loss of get_loss(): src/oem_logistic_dense.h:1057-1088 (uses whatever prob currently holds)
__global__ void logistic_loss_kernel(const double *__restrict__ y, const double *__restrict__ prob, long long n,
                                     double *__restrict__ partial) {
    double s = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double pr = prob[i];
        if (y[i] == 1.0) s += (pr > 1e-5) ? log(1.0 / pr) : log(1.0 / 1e-5);
        else s += (pr <= 1.0 - 1e-5) ? log(1.0 / (1.0 - pr)) : log(1.0 / 1e-5);
    }
    __shared__ double red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        partial[blockIdx.x] = t;
    }
}

double logistic_loss(Ctx &cx, const double *y, const double *prob, int64_t n) {
    DBuf<double> buf(1024 + 2);        // per-block partial sums, then their [sum, sum of squares]
    logistic_loss_kernel<<<1024, 256, 0, cx.stream>>>(y, prob, n, buf.p);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
    vecsum_launch(cx, buf.p, 1024, 0.0, buf.p + 1024, false);
    cx.all_reduce(buf.p + 1024, 2);
    double h[2];
    OEM_CUDA(cudaMemcpyAsync(h, buf.p + 1024, sizeof h, cudaMemcpyDeviceToHost, cx.stream));
    cx.sync();
    return h[0];
}

__global__ void scale_inplace_kernel(double *v, size_t n, double f) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] *= f;
}

// X'r (p values at xr) and sum r (at sr) of the column sweeps -> the (p+1)-vector [sum r, X'r] the slab kernel emits
__global__ void irls_pack_grad_kernel(const double *__restrict__ xr, const double *__restrict__ sr, int p, double *__restrict__ g) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < p) g[1 + j] = xr[j];
    if (j == 0) g[0] = sr[0];
}

namespace {
// OEMB200_TIMING=1: host wall-clock marks of the driver on stderr (where does time go outside the stream?)
struct WallMarks {
    bool on = getenv("OEMB200_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void mark(const char *what) {
        if (!on) return;
        fprintf(stderr, "[timing] %-28s %9.3f ms\n", what,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    }
};
}  // namespace

void fit_logistic(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s,
                  const oemb200_opts *o, oemb200_result *res, SlabCache *cache) {
    check_common(s, o, res, "binomial");
    if (n < 1 || p < 1 || ldx < n) fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d ldx=%lld", (long long)n, p, (long long)ldx);
    const int icpt = s->intercept ? 1 : 0, q = p + icpt;
    const bool stdz = s->standardize != 0;
    WallMarks wm;
    struct ExitMark { WallMarks &w; ~ExitMark() { w.mark("scope exit (buffers freed)"); } } exit_mark{wm};
    Ctx cx(o);
    wm.mark("context");
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, q, /*zero_w0=*/true);

    const size_t t_h = tm.start(&cx.st.ms_h2d);
    DevMatrix X;
    to_device_matrix(cx, x, n, p, ldx, X);
    DevVector yv;
    to_device_vector(cx, y, n, yv);
    tm.stop(t_h);

    // ---- init_oem: colsq, X'y (oem_logistic_dense.h:721-793) ----
    const LogisticInit in = logistic_init(
        cx, n, p, q, stdz, [&](double *out) { colstats_launch(cx, X.p, n, p, X.ld, nullptr, yv.p, nullptr, out, false); },
        "oem_fit_logistic_dense with n <= p + intercept: the reference takes least-squares steps on the 0/1 "
        "response there, with a step matrix its d does not bound (src/oem_logistic_dense.h:478-483, 530-568; "
        "restated in oracle/oracle.py:_logistic_wide, which diverges) -- not built");
    const double n_tot = in.n_tot;
    su.build_lambdas(s, in.lmax, /*logistic_fudge=*/true);

    // ---- data-pass route.  Every route ends in the same (p+1)-vector all-reduce, so ranks may differ in their choice.
    //      slab (default where it applies): X re-laid out once, one HBM sweep per pass (logit_slab.cu)
    //      sweeps: xb_kernel + colstats_kernel, two HBM sweeps per pass (small / very wide p, or no room for the copy)
    const char *route_env = getenv("OEMB200_LOGIT_ROUTE");
    bool slab = logit_slab_rows(p) != 0 && !(route_env && strcmp(route_env, "sweeps") == 0) &&
                (logit_slab_preferred(n, p) || (route_env && strcmp(route_env, "slab") == 0));
    DBuf<double> slabs_own;
    const double *slabs_p = nullptr;
    if (slab && cache && cache->slabs && cache->rt == logit_slab_rows(p)) {
        slabs_p = cache->slabs;                                                       // built by an earlier fit on this handle
    } else if (slab) {
        size_t free_b = 0, total_b = 0;
        OEM_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t need = logit_slab_doubles(n, p) * 8;
        if (need + 3 * (size_t)(n + 2) * 8 + (1ull << 30) > free_b) slab = false;      // no room for the second copy of X
    }
    if (slab && !slabs_p) {
        const size_t t_r = tm.start(&cx.st.ms_relayout);
        double *dst = nullptr;
        if (cache) {       // the handle owns the copy (plain cudaMalloc: it outlives this call and this thread's pool)
            if (cache->slabs) { cudaFree(cache->slabs); cache->slabs = nullptr; }
            OEM_CUDA(cudaMalloc(reinterpret_cast<void **>(&dst), logit_slab_doubles(n, p) * 8));
            cache->slabs = dst;
            cache->rt = logit_slab_rows(p);
        } else {
            slabs_own.alloc(logit_slab_doubles(n, p));
            dst = slabs_own.p;
        }
        logit_slab_relayout(cx, X.p, n, p, X.ld, dst);
        slabs_p = dst;
        tm.stop(t_r);
    }

    // ---- device state ----
    PenaltyTables tb(cx, su, s, p, icpt);
    DBuf<double> d_cinv(p), d_g((size_t)p + 2), d_XY(q), d_XX((size_t)q * q), d_d(1);
    DBuf<double> d_prob(n + (n & 1)), d_res, d_W(n + (n & 1));
    if (!slab) d_res.alloc(n + (n & 1));
    d_prob.zero(cx.stream);
    d_W.zero(cx.stream);
    d_cinv.upload(in.cinv.data(), p, cx.stream);
    // Hessian bundle: [G p*p | stats 3p | sum W, sum W^2]
    const size_t nbh = (size_t)p * p + 3 * (size_t)p + 2;
    DBuf<double> bh(nbh), d_nobs(1);
    d_nobs.upload(&n_tot, 1, cx.stream);
    DBuf<double> gradb(3 * (size_t)p + 2);   // two-sweep route: [stats 3p | sum r, sum r^2]
    fill_common_outputs(su, res);

    // Phase clocks of the per-iteration kernels live on the device (%globaltimer, accumulated by the kernels themselves): a
    // pair of event records around each of them cost ~21 us of stream time per IRLS iteration, 6 % of a sharded fit.
    //   [0] data passes (slab kernel start -> end of its partial-sum kernel), [1] scratch, [2] path launches, [3] all-reduces
    DBuf<unsigned long long> d_clk(4);
    d_clk.zero(cx.stream);
    const bool clk_allreduce = cx.comm != nullptr && cx.all_reduce_can_skip((int64_t)p + 1);     // the peer-memory kernel
    // Speculation (IrlsLoop) needs every kernel of the chain to be predicated: slab route, upper-bound Hessian (the Gram
    // launch cannot), and a cross-rank sum that runs on the peer-memory transport (an NCCL collective cannot be predicated
    // from the device).
    const bool speculate = slab && !o->hessian_full && cx.all_reduce_can_skip((int64_t)p + 1) &&
                           getenv("OEMB200_IRLS_NO_SPECULATION") == nullptr;
    IrlsLoop loop(cx, su, tb, o, 1, icpt, speculate);
    loop.set_model(0, d_XX.p, d_XY.p, d_d.p, stdz ? d_cinv.p : nullptr, d_clk.p + 2);
    wm.mark("setup (stats, slabs, buffers)");

    // One IRLS iteration as a chain of kernels on the stream (k = IRLS counter of this lambda).  Every kernel of the chain
    // takes the model's `conv` flag as its predicate, so an iteration enqueued AFTER the loop has converged costs a few
    // empty launches.
    const int *skip = loop.conv.p;
    auto enqueue_round = [&](int i, int k, bool pass) {
        bool rebuilt = false;
        if (pass) {
            const bool need_w = (k == 0 && i == 0) || o->hessian_full;
            if (slab) {
                // one kernel, one HBM sweep: prob, W and the gradient sums [sum r, X'r] (timed on the device: d_clk)
                logit_slab_launch(cx, slabs_p, n, p, loop.b.p, loop.b0.p, yv.p, d_prob.p, d_W.p, d_g.p, skip, d_clk.p + 0);
                cx.st.gemv_bytes += 8.0 * n * p + 8.0 * (3.0 * n + 2.0 * p);
            } else {
                const size_t t1 = tm.start(&cx.st.ms_irls_xb);
                xb_launch(cx, X.p, n, p, X.ld, loop.b.p, 0.0, yv.p, nullptr, d_prob.p, d_res.p, d_W.p, true, loop.b0.p);
                tm.stop(t1);
                cx.st.gemv_bytes += 8.0 * n * p + 8.0 * (n + p);
                cx.st.data_passes += 1;
            }
            // W(i) clamp, sic (oem_logistic_dense.h:953-959).  W is consumed by the Hessian build alone (the next data pass
            // recomputes it from scratch), so the clamp only has to happen in front of one
            if (need_w && cx.rank == 0 && k < n) {
                clamp_one_kernel<<<1, 1, 0, cx.stream>>>(d_W.p, k, 1e-5, skip);
                cx.st.kernel_launches += 1;
            }
            if (need_w) {
                // X'WX / n with the intercept border (oem_logistic_dense.h:458-522)
                double *G = bh.p, *st = G + (size_t)p * p, *ws = st + 3 * (size_t)p;
                // The upper-bound Hessian is built on the first pass of a penalty, at beta = 0 (b = 0, b0 = 0): every
                // row has eta = 0, prob = 1/2 and W = prob (1 - prob) = 1/4 exactly.  A power-of-two weight commutes
                // with every rounding of the Gram, so X'WX == X'X / 4 to the bit, and the unweighted DMMA variant (no
                // multiply in the fragment load: 34.7 against 31 TFLOP/s) followed by one scaling pass over p x p
                // gives the identical matrix.
                gram_launch(cx, X.p, n, p, X.ld, {RowSegment{0, n, 0}}, 1, nullptr, o->hessian_full ? d_W.p : nullptr, G, false);
                if (!o->hessian_full) {
                    scale_inplace_kernel<<<(unsigned)(((size_t)p * p + 255) / 256), 256, 0, cx.stream>>>(G, (size_t)p * p, 0.25);
                    cx.st.kernel_launches += 1;
                }
                const size_t tc = tm.start(&cx.st.ms_colstats);
                colstats_launch(cx, X.p, n, p, X.ld, d_W.p, nullptr, nullptr, st, false);
                vecsum_launch(cx, d_W.p, n, 0.0, ws, false);
                tm.stop(tc);
                const size_t t_ar = tm.start(&cx.st.ms_allreduce);
                cx.all_reduce(bh.p, (int64_t)nbh);
                tm.stop(t_ar);
                // border = (W'X) o w, corner = sum W, divisor n; uncentred scale from the DATA colsq:
                // assemble_aug derives w from stats row 2, so put sum x^2 there
                OEM_CUDA(cudaMemcpyAsync(st + 2 * (size_t)p, in.stats.p + 2 * (size_t)p, (size_t)p * 8,
                                         cudaMemcpyDeviceToDevice, cx.stream));
                assemble_aug_launch(cx, p, icpt, stdz ? 1 : 0, 1, 1, G, st, ws, 1, ws, d_nobs.p, d_XX.p, nullptr,
                                    nullptr, nullptr);
                rebuilt = true;
            }
            if (!slab) {
                const size_t t2 = tm.start(&cx.st.ms_irls_xtr);
                colstats_launch(cx, X.p, n, p, X.ld, d_res.p, nullptr, nullptr, gradb.p, false);
                vecsum_launch(cx, d_res.p, n, 0.0, gradb.p + 3 * (size_t)p, false);
                irls_pack_grad_kernel<<<(p + 255) / 256, 256, 0, cx.stream>>>(gradb.p, gradb.p + 3 * (size_t)p, p, d_g.p);
                tm.stop(t2);
                cx.st.kernel_launches += 1;
                cx.st.gemv_bytes += 8.0 * n * p + 8.0 * (n + p);
            }
            if (cx.distributed()) {
                if (clk_allreduce) {
                    cx.all_reduce(d_g.p, (int64_t)p + 1, speculate ? skip : nullptr, d_clk.p + 3);
                } else {
                    const size_t t_ar = tm.start(&cx.st.ms_allreduce);
                    cx.all_reduce(d_g.p, (int64_t)p + 1, speculate ? skip : nullptr);
                    tm.stop(t_ar);
                }
            }
        }
        // XY = XX beta + grad (:999) after a data pass: formed by the path launch
        loop.path_step(0, rebuilt, pass ? d_g.p : nullptr, n_tot);
    };
    loop.run(res, enqueue_round, [&](int pp, int i) {
        if (s->compute_loss && res->loss) res->loss[(size_t)pp * su.Lmax + i] = logistic_loss(cx, yv.p, d_prob.p, n);
    });
    wm.mark("IRLS loops enqueued");
    // ---- bring the path back, un-scale (get_beta, oem_logistic_dense.h:1038-1055) ----
    unsigned long long hclk[4] = {0, 0, 0, 0};
    d_clk.download(hclk, 4, cx.stream);
    loop.write_path(stdz ? in.cinv.data() : nullptr, res);
    cx.st.ms_irls_xb += (double)hclk[0] * 1e-6;
    cx.st.ms_path += (double)hclk[2] * 1e-6;
    cx.st.ms_allreduce += (double)hclk[3] * 1e-6;
    wm.mark("path downloaded");
    finish_stats(cx, tm, t_total, res);
    wm.mark("stats collected");
}

// ================================================================================================
// oem_fit_logistic_sparse  (src/oem_logistic_sparse.cpp:30-330, solver src/oem_logistic_sparse.h:458-545, 727-1100)
// ================================================================================================
// dgCMatrix design, n > p, the reference's `ncores <= 1` code path.  Same IRLS skeleton as the dense entry, with the
// sparse solver's own conventions (restated in oracle.oem_fit_logistic_sparse):
//   * X'WX and d are rebuilt on EVERY data pass (compute_XtX_d_update_A is unconditional, :958-961);
//   * the intercept column is the constant `intval`, fixed at the first pass (:470-491): xxdiag = mean(diag(X block)),
//     intval = sqrt((xxdiag / sum W) / n), XX(0,0) = xxdiag, border = (X'W o colsq_inv) * intval;
//   * eta of the (standardize, intercept) branch adds beta(0) without intval (:875-876); grad(0) = sum(y - prob) / n;
//   * get_beta() multiplies the member beta(0) by intval in place (:1040-1043).
// intercept && !standardize multiplies beta by a colsq_inv that the reference never initialised (:880 vs :737-751):
// there is no behaviour to match, so that combination is rejected.
// Data passes: CSR SpMV with the logistic epilogue, the weighted sparse Gram (or densified DMMA tiles from ~6 % density),
// per-column sums over the CSC slots; one all-reduce of [X'WX | X'W | sum W | X'r | sum r] per pass in sharded runs.

__global__ void diag_gather_kernel(const double *__restrict__ G, int p, double *__restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < p) out[j] = G[(size_t)j * p + j];
}

// XX (q x q) = [[xxdiag, ((X'W) o cinv) intval], [., cinv G cinv]] / n
__global__ void logit_sparse_assemble_kernel(int p, int icpt, const double *__restrict__ G, const double *__restrict__ xw,
                                             const double *__restrict__ cinv, double intval, double xxdiag, double n_tot,
                                             double *__restrict__ XX) {
    const int q = p + icpt;
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)q * q) return;
    const int r = (int)(e % q), c = (int)(e / q);
    double v;
    if (icpt && r == 0 && c == 0) v = xxdiag;
    else if (icpt && (r == 0 || c == 0)) {
        const int j = (r == 0 ? c : r) - 1;
        double t = xw[j];
        if (cinv) t *= cinv[j];
        v = t * intval;
    } else {
        const int jr = r - icpt, jc = c - icpt;
        v = G[(size_t)jc * p + jr];
        if (cinv) v = (cinv[jr] * v) * cinv[jc];
    }
    XX[e] = v / n_tot;
}

__global__ void scale_first_kernel(double *v, double f) { v[0] *= f; }

void fit_logistic_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *y,
                         const oemb200_spec *s, const oemb200_opts *o, oemb200_result *res) {
    check_common(s, o, res, "binomial");
    if (n < 1 || p < 1 || !col_ptr || !y) fail(OEMB200_EINVAL, "bad sparse input: n=%lld p=%d", (long long)n, p);
    if (n >= (1ll << 31)) fail(OEMB200_EINVAL, "sparse: more than 2^31-1 rows per call; shard the rows");
    const int icpt = s->intercept ? 1 : 0, q = p + icpt;
    const bool stdz = s->standardize != 0;
    if (icpt && !stdz)
        fail(OEMB200_EUNSUPPORTED, "oem_fit_logistic_sparse with intercept = TRUE and standardize = FALSE reads an uninitialised "
                                   "colsq_inv in the reference (src/oem_logistic_sparse.h:880): no defined behaviour to reproduce");
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, q, /*zero_w0=*/true);

    const size_t t_h = tm.start(&cx.st.ms_h2d);
    std::unique_ptr<SparseDesign, void (*)(SparseDesign *)> sd(nullptr, sparse_design_destroy);
    collective_guard(cx, [&] { sd.reset(sparse_design_create(cx, row_idx, col_ptr, values, n, p)); });   // dgCMatrix checks are per rank
    DevVector yv;
    to_device_vector(cx, y, n, yv);
    tm.stop(t_h);

    // ---- init_oem: colsq, X'y (:727-806); compute_lambda_zero: the X entries of XY = (X'y o colsq_inv) / n (:808-818) ----
    const LogisticInit in = logistic_init(
        cx, n, p, q, stdz, [&](double *out) { sparse_colstats_launch(cx, sd.get(), yv.p, out); },
        "oem_fit_logistic_sparse with n <= p + intercept: the reference takes least-squares steps on the 0/1 "
        "response there, with a step matrix its d does not bound (src/oem_logistic_sparse.h:503-509, 534-580; "
        "restated in oracle/oracle.py:_logistic_wide, which diverges) -- not built");
    const double n_tot = in.n_tot;
    su.build_lambdas(s, in.lmax, /*logistic_fudge=*/true);

    // ---- device state ----
    PenaltyTables tb(cx, su, s, p, icpt);
    const size_t pp2 = (size_t)p * p;
    // per-pass bundle: [G p*p | statsW 3p | sum W, sum W^2 | statsR 3p | sum r, sum r^2]
    const size_t nbp = pp2 + 6 * (size_t)p + 4;
    DBuf<double> bundle(nbp);
    double *G = bundle.p, *statsW = G + pp2, *ws = statsW + 3 * (size_t)p, *statsR = ws + 2, *rs = statsR + 3 * (size_t)p;
    DBuf<double> d_cinv(p), d_g((size_t)p + 2), d_XY(q), d_XX((size_t)q * q), d_d(1), d_diag(p);
    DBuf<double> d_prob(n + 2), d_res(n + 2), d_W(n + 2);
    d_prob.zero(cx.stream);
    d_cinv.upload(in.cinv.data(), p, cx.stream);
    fill_common_outputs(su, res);
    const double *cinv_dev = stdz ? d_cinv.p : nullptr;
    double xxdiag = 0.0, intval = 0.0;
    IrlsLoop loop(cx, su, tb, o, 1, icpt, /*speculate=*/false);          // the sparse Gram launch cannot be predicated
    loop.set_model(0, d_XX.p, d_XY.p, d_d.p, cinv_dev);

    auto enqueue_round = [&](int, int k, bool pass) {
        if (pass) {
            const size_t t1 = tm.start(&cx.st.ms_irls_xb);
            sparse_xb_logistic_launch(cx, sd.get(), loop.b.p, loop.b0.p, yv.p, d_prob.p, d_res.p, d_W.p);
            tm.stop(t1);
            cx.st.data_passes += 1;
            if (cx.rank == 0 && k < n) {             // W(i) clamp, sic (:948-954)
                clamp_one_kernel<<<1, 1, 0, cx.stream>>>(d_W.p, k, 1e-5, nullptr);
                cx.st.kernel_launches += 1;
            }
            sparse_gram_launch(cx, sd.get(), d_W.p, G);                                   // X'WX
            const size_t t2 = tm.start(&cx.st.ms_irls_xtr);
            sparse_colstats_launch(cx, sd.get(), d_W.p, statsW);                          // row 1: X'W
            vecsum_launch(cx, d_W.p, n, 0.0, ws, false);
            sparse_colstats_launch(cx, sd.get(), d_res.p, statsR);                        // row 1: X'(y - prob)
            vecsum_launch(cx, d_res.p, n, 0.0, rs, false);
            tm.stop(t2);
            if (cx.distributed()) {
                const size_t t_ar = tm.start(&cx.st.ms_allreduce);
                cx.all_reduce(bundle.p, (int64_t)nbp);
                tm.stop(t_ar);
            }
            if (icpt && xxdiag <= 0.0) {
                // fixed once, from the first X'WX: xxdiag = mean(diag(scaled X block)), intval (:485-489)
                diag_gather_kernel<<<(p + 255) / 256, 256, 0, cx.stream>>>(G, p, d_diag.p);
                cx.st.kernel_launches += 1;
                std::vector<double> hd(p);
                double hws[2];
                d_diag.download(hd.data(), p, cx.stream);
                OEM_CUDA(cudaMemcpyAsync(hws, ws, 16, cudaMemcpyDeviceToHost, cx.stream));
                cx.sync();
                double tr = 0.0;
                for (int j = 0; j < p; ++j) tr += stdz ? (in.cinv[j] * hd[j]) * in.cinv[j] : hd[j];
                xxdiag = tr / p;
                intval = std::sqrt((xxdiag / hws[0]) / n_tot);
            }
            logit_sparse_assemble_kernel<<<(unsigned)(((size_t)q * q + 255) / 256), 256, 0, cx.stream>>>(
                p, icpt, G, statsW + (size_t)p, cinv_dev, intval, xxdiag, n_tot, d_XX.p);
            irls_pack_grad_kernel<<<(p + 255) / 256, 256, 0, cx.stream>>>(statsR + (size_t)p, rs, p, d_g.p);
            cx.st.kernel_launches += 2;
        }
        // X'WX is rebuilt on every pass, so the eigenvalue is too; XY = XX beta + grad is formed by the launch
        const size_t t3 = tm.start(&cx.st.ms_path);
        loop.path_step(0, pass, pass ? d_g.p : nullptr, n_tot);
        tm.stop(t3);
    };
    loop.run(res, enqueue_round, [&](int pp, int i) {
        if (icpt) {
            // get_beta(): beta(0) *= intval, in place (:1040-1043).  The next lambda starts without a data pass, and its
            // path launch derives the following pass's b0 from its own output
            scale_first_kernel<<<1, 1, 0, cx.stream>>>(loop.final_iterate(0), intval);
            cx.st.kernel_launches += 1;
        }
        if (s->compute_loss && res->loss) res->loss[(size_t)pp * su.Lmax + i] = logistic_loss(cx, yv.p, d_prob.p, n);
    });
    loop.write_path(stdz ? in.cinv.data() : nullptr, res);
    finish_stats(cx, tm, t_total, res);
}

}  // namespace oemb200
