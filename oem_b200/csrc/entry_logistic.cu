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
// (irls_path_problem); their phase clocks are kept on the device.  The only host round trip per IRLS iteration is ONE
// event synchronisation that reads the stop-rule verdict from pinned memory (IrlsLoop, shared with the sparse driver),
// and it is hidden behind the next iteration, which is enqueued one ahead and predicated on the device-side verdict.
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

// b = beta[icpt:] o colsq_inv, b0 = beta[0]: the coefficients the data pass multiplies raw X with (:875-890)
__global__ void irls_coef_kernel(const double *__restrict__ beta, const double *__restrict__ cinv, int p, int icpt,
                                 double *__restrict__ b, double *__restrict__ b0, const int *__restrict__ skip) {
    if (skip && *skip) return;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < p) b[j] = cinv ? beta[icpt + j] * cinv[j] : beta[icpt + j];
    if (j == 0) *b0 = icpt ? beta[0] : 0.0;
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
// 1 / sd of every column from its sum of squares h0[2p + j] (uncentred, divisor n - 1, a zero column keeps scale 1);
// ones when the fit is not standardised
std::vector<double> logistic_cinv(const std::vector<double> &h0, int p, double n_tot, bool stdz) {
    std::vector<double> cinv(p, 1.0);
    if (stdz)
        for (int j = 0; j < p; ++j) {
            double sq = h0[2 * (size_t)p + j] / (n_tot - 1.0);
            if (sq == 0.0) sq = 1.0;
            cinv[j] = 1.0 / std::sqrt(sq);
        }
    return cinv;
}

// The outer IRLS loop of one lambda (src/oem_logistic_dense.h:1000-1035) around a driver's enqueue(k, verdict), which puts
// iteration k of the lambda on the stream: it starts from the iterate in slot (par0 + k) & 1, writes the other slot, and
// its path launch writes the stop rule's verdict to *verdict and to the device flag that predicates every later kernel of
// the lambda.  The host's one round trip per iteration is an event wait and a read of that verdict.  With `speculate`
// iteration k + 1 is enqueued before iteration k's verdict is read, so the GPU never waits for the host (the gap was
// ~100 us per iteration: 5 % of a dense fit on one GPU, 25 % row-sharded over eight); an iteration enqueued after
// convergence is a few empty launches, and its counters are rolled back.  Only a driver whose every kernel of the chain
// can be predicated may speculate.
struct IrlsLoop {
    bool speculate;
    PinnedFlags flag{4};                  // verdict slots: the host reads slot (gi & 3) after that iteration's event
    cudaEvent_t ev[2] = {event_acquire(), event_acquire()};
    long long gi = 0;                     // global IRLS iteration counter (verdict slot = gi & 3, event = gi & 1)
    explicit IrlsLoop(bool speculate_) : speculate(speculate_) {}
    IrlsLoop(const IrlsLoop &) = delete;
    ~IrlsLoop() { event_release(ev[0]); event_release(ev[1]); }

    // Returns niter as the reference reports it: executed iterations + 1 on convergence, irls_maxit + 1 at the cap.  par0
    // moves to the slot of the iterate the last EXECUTED iteration wrote.
    template <typename F>
    int run(Ctx &cx, int irls_maxit, int &par0, F &&enqueue_iteration) {
        auto enqueue = [&](int k) {
            enqueue_iteration(k, flag.p + (gi & 3));
            OEM_CUDA(cudaEventRecord(ev[gi & 1], cx.stream));
            ++gi;
        };
        int it = 0;
        bool broke = false;
        enqueue(0);
        for (;;) {
            // iteration `it` is in the stream (event (gi - 1) & 1 if nothing was enqueued after it)
            const bool ahead = speculate && it + 1 < irls_maxit;
            const oemb200_stats before = cx.st;
            if (ahead) enqueue(it + 1);
            const long long gi_it = gi - 1 - (ahead ? 1 : 0);
            cx.st.host_syncs += 1;
            OEM_CUDA(cudaEventSynchronize(ev[gi_it & 1]));
            if (flag.p[gi_it & 3]) {
                broke = true;
                if (ahead) {           // the speculative iteration found the lambda converged: nothing of it ran
                    cx.st.data_passes = before.data_passes; cx.st.xb_launches = before.xb_launches;
                    cx.st.gemv_bytes = before.gemv_bytes; cx.st.allreduce_calls = before.allreduce_calls;
                    cx.st.allreduce_doubles = before.allreduce_doubles;
                }
                break;
            }
            ++it;
            if (it >= irls_maxit) { it = irls_maxit - 1; break; }
            if (!ahead) enqueue(it);
        }
        par0 = (par0 + it + 1) & 1;
        return (broke ? it : irls_maxit) + 1;
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

    // ---- init_oem: colsq, X'y, sum y (oem_logistic_dense.h:721-793) ----
    const size_t nb0 = 3 * (size_t)p + 3;
    DBuf<double> b0(nb0);
    double *stats0 = b0.p, *ysum = stats0 + 3 * (size_t)p, *nobs = ysum + 2;
    const size_t t_c = tm.start(&cx.st.ms_colstats);
    colstats_launch(cx, X.p, n, p, X.ld, nullptr, yv.p, nullptr, stats0, false);
    vecsum_launch(cx, yv.p, n, 0.0, ysum, false);
    tm.stop(t_c);
    const double nd = (double)n;
    OEM_CUDA(cudaMemcpyAsync(nobs, &nd, 8, cudaMemcpyHostToDevice, cx.stream));
    {
        const size_t t_ar = tm.start(&cx.st.ms_allreduce);
        cx.all_reduce(b0.p, (int64_t)nb0);
        tm.stop(t_ar);
    }
    std::vector<double> h0(nb0);
    b0.download(h0.data(), nb0, cx.stream);
    cx.sync();
    const double n_tot = h0[nb0 - 1];
    if (!(n_tot > q)) fail(OEMB200_EUNSUPPORTED, "oem_fit_logistic_dense with n <= p + intercept: the reference takes least-squares steps on the 0/1 "
                                          "response there, with a step matrix its d does not bound (src/oem_logistic_dense.h:478-483, 530-568; "
                                          "restated in oracle/oracle.py:_logistic_wide, which diverges) -- not built");
    const std::vector<double> cinv = logistic_cinv(h0, p, n_tot, stdz);
    std::vector<double> XY0(q, 0.0);
    if (icpt) XY0[0] = h0[3 * (size_t)p];
    for (int j = 0; j < p; ++j) XY0[icpt + j] = stdz ? h0[(size_t)p + j] * cinv[j] : h0[(size_t)p + j];
    for (auto &v : XY0) v /= n_tot;
    double lmax = 0.0;
    for (int j = 0; j < p; ++j) lmax = std::max(lmax, std::fabs(XY0[icpt + j]));
    su.build_lambdas(s, lmax, /*logistic_fudge=*/true);

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
    const int L = su.Lmax;
    PenaltyTables tb(cx, su, s, p, icpt);
    DBuf<double> d_cinv(p), d_b(p), d_b0(2), d_g((size_t)p + 2), d_XY(q), d_XX((size_t)q * q), d_d(1);
    DBuf<double> d_iter(2 * (size_t)q), d_path((size_t)su.P * L * q);
    DBuf<double> d_prob(n + (n & 1)), d_res, d_W(n + (n & 1));
    DBuf<long long> d_iters_total(1);
    DBuf<int> d_niter(1), d_lz(1);
    if (!slab) d_res.alloc(n + (n & 1));
    d_prob.zero(cx.stream);
    d_W.zero(cx.stream);
    d_iters_total.zero(cx.stream);
    d_path.zero(cx.stream);
    d_cinv.upload(cinv.data(), p, cx.stream);
    // Hessian bundle: [G p*p | stats 3p | sum W, sum W^2]
    const size_t nbh = (size_t)p * p + 3 * (size_t)p + 2;
    DBuf<double> bh(nbh), d_nobs(1);
    d_nobs.upload(&n_tot, 1, cx.stream);
    DBuf<double> gradb(3 * (size_t)p + 2);   // two-sweep route: [stats 3p | sum r, sum r^2]
    PathScratches scratch(1);
    wm.mark("setup (stats, slabs, buffers)");

    fill_common_outputs(su, res);
    const double *cinv_dev = stdz ? d_cinv.p : nullptr;

    // One IRLS iteration as a chain of kernels on the stream (k = IRLS counter of this lambda).  Every kernel of the chain
    // takes `d_conv` as its predicate, so an iteration enqueued AFTER the loop has converged costs a few empty launches.
    DBuf<int> d_conv(1);
    // Phase clocks of the per-iteration kernels live on the device (%globaltimer, accumulated by the kernels themselves): a
    // pair of event records around each of them cost ~21 us of stream time per IRLS iteration, 6 % of a sharded fit.
    //   [0] data passes (slab kernel start -> end of its partial-sum kernel), [1] scratch, [2] path launches, [3] all-reduces
    DBuf<unsigned long long> d_clk(4);
    d_clk.zero(cx.stream);
    IrlsModel md;
    md.XX = d_XX.p; md.XY = d_XY.p; md.d = d_d.p; md.niter = d_niter.p; md.lz = d_lz.p; md.scratch = scratch.s[0];
    md.conv = d_conv.p; md.iters_total = d_iters_total.p; md.icpt = icpt; md.cinv = cinv_dev; md.b = d_b.p; md.b0 = d_b0.p;
    md.t_acc = d_clk.p + 2;
    const bool clk_allreduce = cx.comm != nullptr && cx.all_reduce_can_skip((int64_t)p + 1);     // the peer-memory kernel
    // Speculation (IrlsLoop) needs every kernel of the chain to be predicated: slab route, upper-bound Hessian (the Gram
    // launch cannot), and a cross-rank sum that runs on the peer-memory transport (an NCCL collective cannot be predicated
    // from the device).
    const bool speculate = slab && !o->hessian_full && cx.all_reduce_can_skip((int64_t)p + 1) &&
                           getenv("OEMB200_IRLS_NO_SPECULATION") == nullptr;
    IrlsLoop loop(speculate);

    for (int pp = 0; pp < su.P; ++pp) {
        int par0 = 0;                            // d_iter.p + par0 * q holds the iterate the next iteration starts from
        OEM_CUDA(cudaMemsetAsync(d_iter.p, 0, sizeof(double) * q, cx.stream));      // init(): beta = 0, on_lam_1 = true
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const bool on_lam_1 = (i == 0);
            OEM_CUDA(cudaMemsetAsync(d_conv.p, 0, sizeof(int), cx.stream));
            const int *skip = d_conv.p;

            auto enqueue_iteration = [&](int k, volatile int *verdict) {
                double *cur = d_iter.p + (size_t)((par0 + k) & 1) * q, *nxt = d_iter.p + (size_t)((par0 + k + 1) & 1) * q;
                bool rebuilt = false, form_xy = false;
                if (!(k == 0 && !on_lam_1)) {
                    const bool need_w = (k == 0 && on_lam_1) || o->hessian_full;
                    if (k == 0) {      // later passes of this lambda get b from the previous iteration's path launch (IRLS epilogue)
                        irls_coef_kernel<<<(p + 255) / 256, 256, 0, cx.stream>>>(cur, cinv_dev, p, icpt, d_b.p, d_b0.p, skip);
                        cx.st.kernel_launches += 1;
                    }
                    if (slab) {
                        // one kernel, one HBM sweep: prob, W and the gradient sums [sum r, X'r] (timed on the device: d_clk)
                        logit_slab_launch(cx, slabs_p, n, p, d_b.p, d_b0.p, yv.p, d_prob.p, d_W.p, d_g.p, skip, d_clk.p + 0);
                        cx.st.gemv_bytes += 8.0 * n * p + 8.0 * (3.0 * n + 2.0 * p);
                    } else {
                        const size_t t1 = tm.start(&cx.st.ms_irls_xb);
                        xb_launch(cx, X.p, n, p, X.ld, d_b.p, 0.0, yv.p, nullptr, d_prob.p, d_res.p, d_W.p, true, d_b0.p);
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
                        OEM_CUDA(cudaMemcpyAsync(st + 2 * (size_t)p, stats0 + 2 * (size_t)p, (size_t)p * 8,
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
                    form_xy = true;           // XY = XX beta + grad (:999): formed by the path launch below
                }
                path_launch(cx, irls_path_problem(tb, su, pp, i, o, md, cur, nxt, verdict, rebuilt, form_xy ? d_g.p : nullptr, n_tot));
            };

            res->niter[(size_t)pp * L + i] = loop.run(cx, o->irls_maxit, par0, enqueue_iteration);
            OEM_CUDA(cudaMemcpyAsync(d_path.p + ((size_t)pp * L + i) * q, d_iter.p + (size_t)par0 * q, sizeof(double) * q,
                                     cudaMemcpyDeviceToDevice, cx.stream));
            if (s->compute_loss && res->loss) res->loss[(size_t)pp * L + i] = logistic_loss(cx, yv.p, d_prob.p, n);
        }
    }
    wm.mark("IRLS loops enqueued");
    // ---- bring the path back, un-scale (get_beta, oem_logistic_dense.h:1038-1055) ----
    unsigned long long hclk[4] = {0, 0, 0, 0};
    d_clk.download(hclk, 4, cx.stream);
    irls_write_path(cx, su, p, icpt, d_path.p, d_iters_total.p, d_d.p, stdz ? cinv.data() : nullptr, res);
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

    // ---- init_oem: colsq, X'y (:727-806) ----
    const size_t nb0 = 3 * (size_t)p + 1;
    DBuf<double> b0(nb0);
    const size_t t_c = tm.start(&cx.st.ms_colstats);
    sparse_colstats_launch(cx, sd.get(), yv.p, b0.p);
    tm.stop(t_c);
    const double nd = (double)n;
    OEM_CUDA(cudaMemcpyAsync(b0.p + 3 * (size_t)p, &nd, 8, cudaMemcpyHostToDevice, cx.stream));
    {
        const size_t t_ar = tm.start(&cx.st.ms_allreduce);
        cx.all_reduce(b0.p, (int64_t)nb0);
        tm.stop(t_ar);
    }
    std::vector<double> h0(nb0);
    b0.download(h0.data(), nb0, cx.stream);
    cx.sync();
    const double n_tot = h0[nb0 - 1];
    if (!(n_tot > q)) fail(OEMB200_EUNSUPPORTED, "oem_fit_logistic_sparse with n <= p + intercept: the reference takes least-squares steps on the 0/1 "
                                          "response there, with a step matrix its d does not bound (src/oem_logistic_sparse.h:503-509, 534-580; "
                                          "restated in oracle/oracle.py:_logistic_wide, which diverges) -- not built");
    const std::vector<double> cinv = logistic_cinv(h0, p, n_tot, stdz);
    double lmax = 0.0;      // compute_lambda_zero: the X entries of XY = (X'y o colsq_inv) / n only (:808-818)
    for (int j = 0; j < p; ++j) {
        double v = h0[(size_t)p + j];
        if (stdz) v *= cinv[j];
        lmax = std::max(lmax, std::fabs(v / n_tot));
    }
    su.build_lambdas(s, lmax, /*logistic_fudge=*/true);

    // ---- device state ----
    const int L = su.Lmax;
    PenaltyTables tb(cx, su, s, p, icpt);
    const size_t pp2 = (size_t)p * p;
    // per-pass bundle: [G p*p | statsW 3p | sum W, sum W^2 | statsR 3p | sum r, sum r^2]
    const size_t nbp = pp2 + 6 * (size_t)p + 4;
    DBuf<double> bundle(nbp);
    double *G = bundle.p, *statsW = G + pp2, *ws = statsW + 3 * (size_t)p, *statsR = ws + 2, *rs = statsR + 3 * (size_t)p;
    DBuf<double> d_cinv(p), d_b(p), d_b0(2), d_g((size_t)p + 2), d_XY(q), d_XX((size_t)q * q), d_d(1), d_diag(p);
    DBuf<double> d_iter(2 * (size_t)q), d_path((size_t)su.P * L * q);
    DBuf<double> d_prob(n + 2), d_res(n + 2), d_W(n + 2);
    DBuf<long long> d_iters_total(1);
    DBuf<int> d_niter(1), d_lz(1), d_conv(1);
    d_prob.zero(cx.stream);
    d_iters_total.zero(cx.stream);
    d_path.zero(cx.stream);
    d_cinv.upload(cinv.data(), p, cx.stream);
    PathScratches scratch(1);
    fill_common_outputs(su, res);
    const double *cinv_dev = stdz ? d_cinv.p : nullptr;
    double xxdiag = 0.0, intval = 0.0;
    IrlsModel md;
    md.XX = d_XX.p; md.XY = d_XY.p; md.d = d_d.p; md.niter = d_niter.p; md.lz = d_lz.p; md.scratch = scratch.s[0];
    md.conv = d_conv.p; md.iters_total = d_iters_total.p; md.icpt = icpt; md.cinv = cinv_dev; md.b = d_b.p; md.b0 = d_b0.p;
    IrlsLoop loop(false);          // the sparse Gram launch cannot be predicated

    for (int pp = 0; pp < su.P; ++pp) {
        int par0 = 0;                            // d_iter.p + par0 * q holds the iterate the next iteration starts from
        OEM_CUDA(cudaMemsetAsync(d_iter.p, 0, sizeof(double) * q, cx.stream));
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const bool on_lam_1 = (i == 0);
            OEM_CUDA(cudaMemsetAsync(d_conv.p, 0, sizeof(int), cx.stream));
            auto enqueue_iteration = [&](int k, volatile int *verdict) {
                double *cur = d_iter.p + (size_t)((par0 + k) & 1) * q, *nxt = d_iter.p + (size_t)((par0 + k + 1) & 1) * q;
                const bool pass = !(k == 0 && !on_lam_1);
                if (pass) {
                    if (k == 0) {      // later passes of this lambda get b from the previous iteration's path launch (IRLS epilogue)
                        irls_coef_kernel<<<(p + 255) / 256, 256, 0, cx.stream>>>(cur, cinv_dev, p, icpt, d_b.p, d_b0.p, nullptr);
                        cx.st.kernel_launches += 1;
                    }
                    const size_t t1 = tm.start(&cx.st.ms_irls_xb);
                    sparse_xb_logistic_launch(cx, sd.get(), d_b.p, d_b0.p, yv.p, d_prob.p, d_res.p, d_W.p);
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
                        for (int j = 0; j < p; ++j) tr += stdz ? (cinv[j] * hd[j]) * cinv[j] : hd[j];
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
                path_launch(cx, irls_path_problem(tb, su, pp, i, o, md, cur, nxt, verdict, pass, pass ? d_g.p : nullptr, n_tot));
                tm.stop(t3);
            };

            res->niter[(size_t)pp * L + i] = loop.run(cx, o->irls_maxit, par0, enqueue_iteration);
            double *fin = d_iter.p + (size_t)par0 * q;
            if (icpt) {
                // get_beta(): beta(0) *= intval, in place (:1040-1043).  The next lambda starts without a data pass, and its
                // path launch derives the following pass's b0 from its own output
                scale_first_kernel<<<1, 1, 0, cx.stream>>>(fin, intval);
                cx.st.kernel_launches += 1;
            }
            OEM_CUDA(cudaMemcpyAsync(d_path.p + ((size_t)pp * L + i) * q, fin, sizeof(double) * q, cudaMemcpyDeviceToDevice,
                                     cx.stream));
            if (s->compute_loss && res->loss) res->loss[(size_t)pp * L + i] = logistic_loss(cx, yv.p, d_prob.p, n);
        }
    }
    irls_write_path(cx, su, p, icpt, d_path.p, d_iters_total.p, d_d.p, stdz ? cinv.data() : nullptr, res);
    finish_stats(cx, tm, t_total, res);
}

}  // namespace oemb200
