// entry_logistic.cu -- host driver of oem_fit_logistic_dense (src/oem_logistic_dense.cpp:29-313,
// solver src/oem_logistic_dense.h:721-1036) on the sm_100a kernels.
//
// Per IRLS iteration the reference makes two passes over X:
//   prob = sigma(X (beta o w) + beta0)        (oem_logistic_dense.h:864-949)
//   grad = [sum(y-prob), X'(y-prob) o w] / n  (oem_logistic_dense.h:970-992)
// Here both come out of ONE sweep of a row-slab copy of X (logit_slab.cu; built once per fit), or, for shapes the
// slab kernel does not cover, out of the two HBM-bound sweeps xb_kernel + colstats_kernel.  When the Hessian bound is
// (re)built, X'WX runs on the FP64 tensor pipe with the row weight fused into the fragment load
// (gram_syrk_kernel<WEIGHT>) and the Lanczos eigenvalue inside the path kernel.
//
// The IRLS state never leaves the device.  An iteration of the dense driver is three launches on one stream: the data pass
// (+ its partial-sum kernel), in row-sharded runs the sum of the (p+1)-vector gradient (comm.cu), and the path launch, which
// forms XY = XX beta + grad from the XX slice its members load anyway, runs the inner OEM loop, applies the outer stop rule
// and leaves the next pass's coefficients (PathProblem::xy_grad / irls_*); their phase clocks are kept on the device.  The
// only host round trip per IRLS iteration is ONE event synchronisation that reads the stop-rule flag from pinned memory,
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

void logistic_loss_launch(Ctx &cx, const double *y, const double *prob, int64_t n, double *partial, double *tot2) {
    logistic_loss_kernel<<<1024, 256, 0, cx.stream>>>(y, prob, n, partial);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
    vecsum_launch(cx, partial, 1024, 0.0, tot2, false);
}

// per-block min / max of v (partial[2 b], partial[2 b + 1]); the host folds the blocks
__global__ void __launch_bounds__(256) minmax_kernel(const double *__restrict__ v, long long n, double *__restrict__ partial) {
    double lo = INFINITY, hi = -INFINITY;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double x = v[i];
        lo = fmin(lo, x); hi = fmax(hi, x);
    }
    __shared__ double slo[8], shi[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0) { slo[threadIdx.x >> 5] = lo; shi[threadIdx.x >> 5] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { lo = fmin(lo, slo[w]); hi = fmax(hi, shi[w]); }
        partial[2 * blockIdx.x] = lo; partial[2 * blockIdx.x + 1] = hi;
    }
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

// stopRule(beta_new, beta_prev, irls_tol) (src/utils.cpp:537-549) on the device; the verdict goes to pinned host
// memory, the inner loop's iteration count is accumulated for the statistics.  One CTA.
// `conv` (device) is the predicate of speculatively enqueued work: once an IRLS loop has converged, every later kernel
// of that lambda -- this one included -- returns at once, so the host may enqueue iteration it + 1 before it has read
// iteration it's verdict.
// With `b` given it also prepares the NEXT data pass: b = beta_new[icpt:] o colsq_inv, b0 = beta_new[0] (what
// irls_coef_kernel computes).  The dense driver no longer launches this kernel -- the same steps are the last thing its
// path launch does (oem_path_kernel, "IRLS epilogue") -- the sparse driver does.
__global__ void irls_stop_kernel(const double *__restrict__ cur, const double *__restrict__ prev, int q, double tol,
                                 const int *__restrict__ niter, long long *__restrict__ iters_total,
                                 volatile int *__restrict__ host_flag, int *__restrict__ conv,
                                 const double *__restrict__ cinv = nullptr, int p = 0, int icpt = 0, double *__restrict__ b = nullptr,
                                 double *__restrict__ b0 = nullptr) {
    if (conv && *conv) return;
    if (b) {
        for (int j = threadIdx.x; j < p; j += blockDim.x) b[j] = cinv ? cur[icpt + j] * cinv[j] : cur[icpt + j];
        if (threadIdx.x == 0) *b0 = icpt ? cur[0] : 0.0;
    }
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    int v = 0;
    for (int i = threadIdx.x; i < q; i += blockDim.x) {
        const double ac = fabs(cur[i]), ap = fabs(prev[i]);
        if ((ac > 1e-13 && ap <= 1e-13) || (ac <= 1e-13 && ap > 1e-13)) v = 1;
        else if (ac > 1e-13 && ap > 1e-13 && fabs((cur[i] - prev[i]) / prev[i]) > tol) v = 1;
    }
    if (v) bad = 1;
    __syncthreads();
    if (threadIdx.x == 0) {
        *iters_total += niter[0];
        if (conv && !bad) *conv = 1;
        *host_flag = bad ? 0 : 1;
        __threadfence_system();
    }
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
struct PinnedFlag {          // four verdict slots: the host reads slot (iteration & 3) after that iteration's event
    int *p = nullptr;
    PinnedFlag() { OEM_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&p), 64, cudaHostAllocMapped)); memset(p, 0, 64); }
    ~PinnedFlag() { if (p) cudaFreeHost(p); }
};
struct ScratchHolder {
    PathScratch *s;
    ScratchHolder() : s(path_scratch_create()) {}
    ~ScratchHolder() { path_scratch_destroy(s); }
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
    std::vector<double> cinv(p, 1.0);
    if (stdz)
        for (int j = 0; j < p; ++j) {
            double sq = h0[2 * (size_t)p + j] / (n_tot - 1.0);
            if (sq == 0.0) sq = 1.0;
            cinv[j] = 1.0 / std::sqrt(sq);
        }
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
    std::vector<double> pf(q, 0.0);
    for (int j = 0; j < p; ++j) pf[icpt + j] = s->penalty_factor[j];
    const int L = su.Lmax;
    DBuf<double> d_pf(q), d_cinv(p), d_b(p), d_b0(2), d_g((size_t)p + 2), d_XY(q), d_XX((size_t)q * q), d_d(1);
    DBuf<double> d_iter(2 * (size_t)q), d_path((size_t)su.P * L * q), d_lams((size_t)su.P * L);
    DBuf<double> d_prob(n + (n & 1)), d_res, d_W(n + (n & 1));
    DBuf<long long> d_iters_total(1);
    DBuf<int> d_niter(1), d_lz(1);
    if (!slab) d_res.alloc(n + (n & 1));
    d_prob.zero(cx.stream);
    d_W.zero(cx.stream);
    d_iters_total.zero(cx.stream);
    d_path.zero(cx.stream);
    d_pf.upload(pf.data(), q, cx.stream);
    d_cinv.upload(cinv.data(), p, cx.stream);
    {
        std::vector<double> lam_flat((size_t)su.P * L, 0.0);
        for (int pp = 0; pp < su.P; ++pp)
            for (size_t i = 0; i < su.lam[pp].size() && (int)i < L; ++i) lam_flat[(size_t)pp * L + i] = su.lam[pp][i];
        d_lams.upload(lam_flat.data(), lam_flat.size(), cx.stream);
        cx.sync();                                  // lam_flat is a host temporary
    }
    DBuf<int> g_unique, g_ptr, g_idx, g_cover;
    DBuf<double> g_w;
    if (su.any_group) {
        g_unique.alloc(su.unique.size()); g_unique.upload(su.unique.data(), su.unique.size(), cx.stream);
        g_ptr.alloc(su.ptr.size());       g_ptr.upload(su.ptr.data(), su.ptr.size(), cx.stream);
        g_idx.alloc(std::max<size_t>(1, su.idx.size()));
        if (!su.idx.empty()) g_idx.upload(su.idx.data(), su.idx.size(), cx.stream);
        g_w.alloc(su.gw.size());          g_w.upload(su.gw.data(), su.gw.size(), cx.stream);
        g_cover.alloc(q);                 g_cover.upload(su.cover.data(), q, cx.stream);
    }
    // Hessian bundle: [G p*p | stats 3p | sum W, sum W^2]
    const size_t nbh = (size_t)p * p + 3 * (size_t)p + 2;
    DBuf<double> bh(nbh), d_nobs(1);
    d_nobs.upload(&n_tot, 1, cx.stream);
    DBuf<double> gradb(3 * (size_t)p + 2);   // two-sweep route: [stats 3p | sum r, sum r^2]
    DBuf<double> d_losspart(1024);
    PinnedFlag flag;
    ScratchHolder scratch;
    wm.mark("setup (stats, slabs, buffers)");

    fill_common_outputs(su, res);
    memset(res->beta, 0, sizeof(double) * (size_t)su.P * (p + 1) * L);
    double dval = 0.0;
    const double *cinv_dev = stdz ? d_cinv.p : nullptr;

    // One IRLS iteration as a chain of kernels on the stream (k = IRLS counter of this lambda).  Every kernel of the chain
    // takes `d_conv` as its predicate, so an iteration enqueued AFTER the loop has converged costs a few empty launches.
    DBuf<int> d_conv(1);
    // Phase clocks of the per-iteration kernels live on the device (%globaltimer, accumulated by the kernels themselves): a
    // pair of event records around each of them cost ~21 us of stream time per IRLS iteration, 6 % of a sharded fit.
    //   [0] data passes (slab kernel start -> end of its partial-sum kernel), [1] scratch, [2] path launches, [3] all-reduces
    DBuf<unsigned long long> d_clk(4);
    d_clk.zero(cx.stream);
    const bool clk_allreduce = cx.comm != nullptr && cx.all_reduce_can_skip((int64_t)p + 1);     // the peer-memory kernel
    // Speculation: enqueue iteration k + 1 before reading iteration k's verdict, so the GPU never waits for the host round
    // trip (the gap was ~100 us per iteration: 5 % of the fit on one GPU, 25 % row-sharded over eight).  Possible when every
    // kernel of the chain can be predicated: slab route, upper-bound Hessian (the Gram launch cannot), and a cross-rank sum
    // that runs on the peer-memory transport (an NCCL collective cannot be predicated from the device).
    const bool speculate = slab && !o->hessian_full && cx.all_reduce_can_skip((int64_t)p + 1) &&
                           getenv("OEMB200_IRLS_NO_SPECULATION") == nullptr;
    cudaEvent_t ev_done[2] = {event_acquire(), event_acquire()};
    struct EvGuard { cudaEvent_t *e; ~EvGuard() { event_release(e[0]); event_release(e[1]); } } ev_guard{ev_done};
    long long gi = 0;                            // global IRLS iteration counter (verdict slot = gi & 3, event = gi & 1)

    for (int pp = 0; pp < su.P; ++pp) {
        int par0 = 0;                            // d_iter.p + par0 * q holds the iterate the next iteration starts from
        OEM_CUDA(cudaMemsetAsync(d_iter.p, 0, sizeof(double) * q, cx.stream));      // init(): beta = 0, on_lam_1 = true
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const bool on_lam_1 = (i == 0);
            OEM_CUDA(cudaMemsetAsync(d_conv.p, 0, sizeof(int), cx.stream));
            const int *skip = d_conv.p;

            auto enqueue_iteration = [&](int k) {
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
                        // The upper-bound Hessian is built at beta = 0, where every W_i is prob (1 - prob) = 0.25 exactly.
                        // A uniform power-of-two weight commutes with every rounding of the Gram, so X'WX == w0 * X'X to the
                        // bit, and the unweighted DMMA variant (no multiply in the fragment load: 34.7 against 31 TFLOP/s)
                        // followed by one scaling pass over p x p gives the identical matrix.  Decided per rank from its own
                        // rows; the all-reduced bundle has the same shape either way.
                        double w_uniform = 0.0;
                        if (!o->hessian_full) {
                            const int nblk = 1024;
                            DBuf<double> mm(2 * (size_t)nblk);
                            minmax_kernel<<<nblk, 256, 0, cx.stream>>>(d_W.p, n, mm.p);
                            cx.st.kernel_launches += 1;
                            std::vector<double> hmm(2 * (size_t)nblk);
                            mm.download(hmm.data(), hmm.size(), cx.stream);
                            cx.sync();
                            double lo = hmm[0], hi = hmm[1];
                            for (int b2 = 1; b2 < nblk; ++b2) { lo = std::min(lo, hmm[2 * b2]); hi = std::max(hi, hmm[2 * b2 + 1]); }
                            int ex = 0;
                            if (lo == hi && lo > 0.0 && std::frexp(lo, &ex) == 0.5) w_uniform = lo;      // exact power of two
                        }
                        gram_launch(cx, X.p, n, p, X.ld, {RowSegment{0, n, 0}}, 1, nullptr, w_uniform > 0.0 ? nullptr : d_W.p, G, false);
                        if (w_uniform > 0.0 && w_uniform != 1.0) {
                            scale_inplace_kernel<<<(unsigned)(((size_t)p * p + 255) / 256), 256, 0, cx.stream>>>(G, (size_t)p * p, w_uniform);
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
                // inner OEM loop: one chain, one lambda, warm start (oem_logistic_dense.h:1010-1022)
                PathProblem pr;
                pr.q = q; pr.ngram = 1; pr.XX = d_XX.p; pr.XY = d_XY.p; pr.d = d_d.p;
                pr.compute_eig = rebuilt; pr.eig_factor = 1.0005; pr.eig_tol = 1e-10;
                ChainDesc c;
                c.gram = 0; c.penalty = su.pen[pp]; c.nlam = 1; c.lam_off = 0; c.alpha = su.alpha;
                c.gamma = su.gamma[pp]; c.tau = su.tau; c.out_off = 0;
                pr.chains.push_back(c);
                pr.lambdas = d_lams.p + (size_t)pp * L + i; pr.Lmax = 1; pr.pen_fact = d_pf.p;
                pr.ngroups = su.any_group ? (int)su.unique.size() : 0;
                pr.ngidx = su.any_group ? (int)su.idx.size() : 0;
                pr.unique_groups = g_unique.p; pr.grp_ptr = g_ptr.p; pr.grp_idx = g_idx.p;
                pr.group_weights = g_w.p; pr.grp_cover = g_cover.p;
                pr.beta_init = cur; pr.beta_final = nullptr;
                pr.maxit = o->maxit; pr.tol = o->tol;
                pr.beta_out = nxt; pr.niter_out = d_niter.p; pr.lanczos_steps = d_lz.p;
                pr.scratch = scratch.s;
                pr.skip = skip;
                if (form_xy) { pr.xy_grad = d_g.p; pr.xy_cinv = cinv_dev; pr.xy_n = n_tot; pr.xy_icpt = icpt; pr.xy_out = d_XY.p; }
                pr.t_acc = d_clk.p + 2;
                // the outer loop's stop rule, its verdicts and the next pass's coefficients are the launch's last step
                pr.irls_conv = d_conv.p; pr.irls_host_flag = flag.p + (gi & 3); pr.irls_iters_total = d_iters_total.p;
                pr.irls_tol = o->irls_tol; pr.irls_cinv = cinv_dev; pr.irls_p = p; pr.irls_icpt = icpt;
                pr.irls_b = d_b.p; pr.irls_b0 = d_b0.p;
                path_launch(cx, pr);
                OEM_CUDA(cudaEventRecord(ev_done[gi & 1], cx.stream));
                ++gi;
            };

            int it = 0;
            bool broke = false;
            enqueue_iteration(0);
            for (;;) {
                // iteration `it` is in the stream (event (gi - 1) & 1 if nothing was enqueued after it)
                const bool ahead = speculate && it + 1 < o->irls_maxit;
                const oemb200_stats before = cx.st;
                if (ahead) enqueue_iteration(it + 1);
                const long long gi_it = gi - 1 - (ahead ? 1 : 0);
                cx.st.host_syncs += 1;
                OEM_CUDA(cudaEventSynchronize(ev_done[gi_it & 1]));          // the one host round trip of the IRLS iteration
                if (flag.p[gi_it & 3]) {
                    broke = true;
                    if (ahead) {           // the speculative iteration found d_conv set: nothing of it ran
                        cx.st.data_passes = before.data_passes; cx.st.xb_launches = before.xb_launches;
                        cx.st.gemv_bytes = before.gemv_bytes; cx.st.allreduce_calls = before.allreduce_calls;
                        cx.st.allreduce_doubles = before.allreduce_doubles;
                    }
                    break;
                }
                ++it;
                if (it >= o->irls_maxit) { it = o->irls_maxit - 1; break; }
                if (!ahead) enqueue_iteration(it);
            }
            res->niter[(size_t)pp * L + i] = (broke ? it : o->irls_maxit) + 1;
            par0 = (par0 + it + 1) & 1;                      // the iterate the last EXECUTED iteration produced
            double *fin = d_iter.p + (size_t)par0 * q;
            OEM_CUDA(cudaMemcpyAsync(d_path.p + ((size_t)pp * L + i) * q, fin, sizeof(double) * q, cudaMemcpyDeviceToDevice,
                                     cx.stream));
            if (s->compute_loss && res->loss) {
                logistic_loss_kernel<<<1024, 256, 0, cx.stream>>>(yv.p, d_prob.p, n, d_losspart.p);
                cx.st.kernel_launches += 1;
                DBuf<double> tot(2);
                vecsum_launch(cx, d_losspart.p, 1024, 0.0, tot.p, false);
                cx.all_reduce(tot.p, 2);
                double h[2];
                tot.download(h, 2, cx.stream);
                cx.sync();
                res->loss[(size_t)pp * L + i] = h[0];
            }
        }
    }
    wm.mark("IRLS loops enqueued");
    // ---- bring the path back, un-scale (get_beta, oem_logistic_dense.h:1038-1055) ----
    std::vector<double> hpath((size_t)su.P * L * q);
    long long iters_total = 0;
    d_path.download(hpath.data(), hpath.size(), cx.stream);
    d_iters_total.download(&iters_total, 1, cx.stream);
    d_d.download(&dval, 1, cx.stream);
    unsigned long long hclk[4] = {0, 0, 0, 0};
    d_clk.download(hclk, 4, cx.stream);
    cx.sync();
    cx.st.ms_irls_xb += (double)hclk[0] * 1e-6;
    cx.st.ms_path += (double)hclk[2] * 1e-6;
    cx.st.ms_allreduce += (double)hclk[3] * 1e-6;
    cx.st.d2h_bytes += (int64_t)hpath.size() * 8;
    cx.st.total_oem_iters += iters_total;
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const double *raw = &hpath[((size_t)pp * L + i) * q];
            double *out = res->beta + ((size_t)pp * L + i) * (p + 1);
            if (icpt) out[0] = raw[0];
            for (int j = 0; j < p; ++j) out[1 + j] = stdz ? raw[icpt + j] * cinv[j] : raw[icpt + j];
        }
    *res->d = dval;
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
    std::vector<double> cinv(p, 1.0);
    if (stdz)
        for (int j = 0; j < p; ++j) {
            double sq = h0[2 * (size_t)p + j] / (n_tot - 1.0);
            if (sq == 0.0) sq = 1.0;
            cinv[j] = 1.0 / std::sqrt(sq);
        }
    double lmax = 0.0;      // compute_lambda_zero: the X entries of XY = (X'y o colsq_inv) / n only (:808-818)
    for (int j = 0; j < p; ++j) {
        double v = h0[(size_t)p + j];
        if (stdz) v *= cinv[j];
        lmax = std::max(lmax, std::fabs(v / n_tot));
    }
    su.build_lambdas(s, lmax, /*logistic_fudge=*/true);

    // ---- device state ----
    std::vector<double> pf(q, 0.0);
    for (int j = 0; j < p; ++j) pf[icpt + j] = s->penalty_factor[j];
    const int L = su.Lmax;
    const size_t pp2 = (size_t)p * p;
    // per-pass bundle: [G p*p | statsW 3p | sum W, sum W^2 | statsR 3p | sum r, sum r^2]
    const size_t nbp = pp2 + 6 * (size_t)p + 4;
    DBuf<double> bundle(nbp);
    double *G = bundle.p, *statsW = G + pp2, *ws = statsW + 3 * (size_t)p, *statsR = ws + 2, *rs = statsR + 3 * (size_t)p;
    DBuf<double> d_pf(q), d_cinv(p), d_b(p), d_b0(2), d_g((size_t)p + 2), d_XY(q), d_XX((size_t)q * q), d_d(1), d_diag(p);
    DBuf<double> d_iter(2 * (size_t)q), d_path((size_t)su.P * L * q), d_lams((size_t)su.P * L);
    DBuf<double> d_prob(n + 2), d_res(n + 2), d_W(n + 2), d_losspart(1024);
    DBuf<long long> d_iters_total(1);
    DBuf<int> d_niter(1), d_lz(1);
    d_prob.zero(cx.stream);
    d_iters_total.zero(cx.stream);
    d_path.zero(cx.stream);
    d_pf.upload(pf.data(), q, cx.stream);
    d_cinv.upload(cinv.data(), p, cx.stream);
    {
        std::vector<double> lam_flat((size_t)su.P * L, 0.0);
        for (int pp = 0; pp < su.P; ++pp)
            for (size_t i = 0; i < su.lam[pp].size() && (int)i < L; ++i) lam_flat[(size_t)pp * L + i] = su.lam[pp][i];
        d_lams.upload(lam_flat.data(), lam_flat.size(), cx.stream);
        cx.sync();
    }
    DBuf<int> g_unique, g_ptr, g_idx, g_cover;
    DBuf<double> g_w;
    if (su.any_group) {
        g_unique.alloc(su.unique.size()); g_unique.upload(su.unique.data(), su.unique.size(), cx.stream);
        g_ptr.alloc(su.ptr.size());       g_ptr.upload(su.ptr.data(), su.ptr.size(), cx.stream);
        g_idx.alloc(std::max<size_t>(1, su.idx.size()));
        if (!su.idx.empty()) g_idx.upload(su.idx.data(), su.idx.size(), cx.stream);
        g_w.alloc(su.gw.size());          g_w.upload(su.gw.data(), su.gw.size(), cx.stream);
        g_cover.alloc(q);                 g_cover.upload(su.cover.data(), q, cx.stream);
    }
    PinnedFlag flag;
    ScratchHolder scratch;
    fill_common_outputs(su, res);
    memset(res->beta, 0, sizeof(double) * (size_t)su.P * (p + 1) * L);
    const double *cinv_dev = stdz ? d_cinv.p : nullptr;
    double xxdiag = 0.0, intval = 0.0;

    for (int pp = 0; pp < su.P; ++pp) {
        double *cur = d_iter.p, *nxt = d_iter.p + q;
        OEM_CUDA(cudaMemsetAsync(cur, 0, sizeof(double) * q, cx.stream));
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const bool on_lam_1 = (i == 0);
            int it = 0;
            bool broke = false;
            for (it = 0; it < o->irls_maxit; ++it) {
                bool rebuilt = false;
                if (!(it == 0 && !on_lam_1)) {
                    irls_coef_kernel<<<(p + 255) / 256, 256, 0, cx.stream>>>(cur, cinv_dev, p, icpt, d_b.p, d_b0.p, nullptr);
                    cx.st.kernel_launches += 1;
                    const size_t t1 = tm.start(&cx.st.ms_irls_xb);
                    sparse_xb_logistic_launch(cx, sd.get(), d_b.p, d_b0.p, yv.p, d_prob.p, d_res.p, d_W.p);
                    tm.stop(t1);
                    cx.st.data_passes += 1;
                    if (cx.rank == 0 && it < n) {            // W(i) clamp, sic (:948-954)
                        clamp_one_kernel<<<1, 1, 0, cx.stream>>>(d_W.p, it, 1e-5, nullptr);
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
                    path_xy_launch(cx, q, icpt, d_XX.p, cur, d_g.p, cinv_dev, n_tot, d_XY.p, nullptr);
                    rebuilt = true;
                }
                PathProblem pr;
                pr.q = q; pr.ngram = 1; pr.XX = d_XX.p; pr.XY = d_XY.p; pr.d = d_d.p;
                pr.compute_eig = rebuilt; pr.eig_factor = 1.0005; pr.eig_tol = 1e-10;
                ChainDesc c;
                c.gram = 0; c.penalty = su.pen[pp]; c.nlam = 1; c.lam_off = 0; c.alpha = su.alpha;
                c.gamma = su.gamma[pp]; c.tau = su.tau; c.out_off = 0;
                pr.chains.push_back(c);
                pr.lambdas = d_lams.p + (size_t)pp * L + i; pr.Lmax = 1; pr.pen_fact = d_pf.p;
                pr.ngroups = su.any_group ? (int)su.unique.size() : 0;
                pr.ngidx = su.any_group ? (int)su.idx.size() : 0;
                pr.unique_groups = g_unique.p; pr.grp_ptr = g_ptr.p; pr.grp_idx = g_idx.p;
                pr.group_weights = g_w.p; pr.grp_cover = g_cover.p;
                pr.beta_init = cur; pr.beta_final = nullptr;
                pr.maxit = o->maxit; pr.tol = o->tol;
                pr.beta_out = nxt; pr.niter_out = d_niter.p; pr.lanczos_steps = d_lz.p;
                pr.scratch = scratch.s;
                const size_t t3 = tm.start(&cx.st.ms_path);
                path_launch(cx, pr);
                tm.stop(t3);
                irls_stop_kernel<<<1, 256, 0, cx.stream>>>(nxt, cur, q, o->irls_tol, d_niter.p, d_iters_total.p, flag.p, nullptr);
                cx.st.kernel_launches += 1;
                cx.sync();
                std::swap(cur, nxt);
                if (*flag.p) { broke = true; break; }
            }
            res->niter[(size_t)pp * L + i] = (broke ? it : o->irls_maxit) + 1;
            if (icpt) {                                      // get_beta(): beta(0) *= intval, in place (:1040-1043)
                scale_first_kernel<<<1, 1, 0, cx.stream>>>(cur, intval);
                cx.st.kernel_launches += 1;
            }
            OEM_CUDA(cudaMemcpyAsync(d_path.p + ((size_t)pp * L + i) * q, cur, sizeof(double) * q, cudaMemcpyDeviceToDevice,
                                     cx.stream));
            if (s->compute_loss && res->loss) {
                logistic_loss_kernel<<<1024, 256, 0, cx.stream>>>(yv.p, d_prob.p, n, d_losspart.p);
                cx.st.kernel_launches += 1;
                DBuf<double> tot(2);
                vecsum_launch(cx, d_losspart.p, 1024, 0.0, tot.p, false);
                cx.all_reduce(tot.p, 2);
                double h[2];
                tot.download(h, 2, cx.stream);
                cx.sync();
                res->loss[(size_t)pp * L + i] = h[0];
            }
        }
    }
    std::vector<double> hpath((size_t)su.P * L * q);
    long long iters_total = 0;
    double dval = 0.0;
    d_path.download(hpath.data(), hpath.size(), cx.stream);
    d_iters_total.download(&iters_total, 1, cx.stream);
    d_d.download(&dval, 1, cx.stream);
    cx.sync();
    cx.st.d2h_bytes += (int64_t)hpath.size() * 8;
    cx.st.total_oem_iters += iters_total;
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const double *raw = &hpath[((size_t)pp * L + i) * q];
            double *out = res->beta + ((size_t)pp * L + i) * (p + 1);
            if (icpt) out[0] = raw[0];
            for (int j = 0; j < p; ++j) out[1 + j] = stdz ? raw[icpt + j] * cinv[j] : raw[icpt + j];
        }
    *res->d = dval;
    finish_stats(cx, tm, t_total, res);
}

}  // namespace oemb200
