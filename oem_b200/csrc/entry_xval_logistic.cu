// entry_xval_logistic.cu -- binomial cross-validation (oemb200_xval_logistic_dense).  The reference has no such entry:
// xval.oem stops on the binomial family (R/oem_xval.R:160-163) and cv.oem refits K + 1 times.  Meaning:
//   model 0     = oem_fit_logistic_dense on all rows (its beta / lambda / niter / loss / d are the result);
//   model k > 0 = the same fit on the rows with foldid != k, at model 0's lambda sequence (the grid its solver saw);
//   cvm / cvsd  = mean and sqrt(M2 / (n - 1)) / sqrt(n) over all rows of cv.oem's binomial measure of the held-out
//                 fold model (R/cv_oem.R:288-330), the ungrouped convention of fit_xval.
//
// The M = K + 1 IRLS loops run in lockstep on shared passes over X:
//   1. steps 1-3 of fit_xval (xval_build_systems): fold-sorted copy, ONE segmented Gram launch for all fold Grams, and
//      assemble_aug for the M systems.  The upper-bound Hessian of a logistic fit is X'WX / n at beta = 0, where
//      W = 1/4 exactly, so each model's Hessian is its Gram, border and corner scaled by 1/4 (unscaled sum x^2 for the
//      standardisation): one Gram launch instead of M;
//   2. per penalty, lambda and IRLS round: ONE fused data pass for all still-active models (logit_fold_launch; a pass
//      is ceil(M / logit_fold_models(p)) sweeps), then one single-chain path launch per active model, which forms
//      XY = XX beta + grad, runs the inner OEM loop, applies the outer stop rule and leaves the model's next
//      coefficients (PathProblem::irls_*).  The host waits once per round and reads the M verdicts; a converged model
//      idles until lambda advances, so every model does exactly the arithmetic of a separate fit;
//   3. one fold-segmented scoring GEMM with the binomial epilogue (cvscore_binomial_launch).
// The reference's logistic quirks come along: no data pass on the first IRLS iteration of every lambda after the first,
// eigenvalue factor 1.0005, uncentred standardisation from each model's own rows.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include "host_common.h"

namespace oemb200 {

namespace {
struct PinnedFlags {          // one verdict slot per model, written by its path launch
    int *p = nullptr;
    explicit PinnedFlags(int m) {
        OEM_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&p), sizeof(int) * (size_t)m, cudaHostAllocMapped));
        memset(p, 0, sizeof(int) * (size_t)m);
    }
    ~PinnedFlags() { if (p) cudaFreeHost(p); }
};
struct Scratches {
    std::vector<PathScratch *> s;
    explicit Scratches(int m) { for (int i = 0; i < m; ++i) s.push_back(path_scratch_create()); }
    ~Scratches() { for (auto *x : s) path_scratch_destroy(x); }
};
}  // namespace

void fit_xval_logistic(const double *x, int64_t n, int p, int64_t ldx, const double *y, const oemb200_spec *s, int nfolds,
                       const int *foldid, const char *type_measure, const oemb200_opts *o, oemb200_result *res) {
    check_common(s, o, res, "binomial");
    if (o->hessian_full)
        fail(OEMB200_EUNSUPPORTED, "binomial xval builds the upper-bound Hessian X'X / 4 once for all fold models; "
                                   "hessian.type = \"full\" needs a new X'WX per model and IRLS iteration: use cv_oem");
    if (o->world > 1 || o->comm || o->allreduce)
        fail(OEMB200_EUNSUPPORTED, "binomial xval runs on one GPU: a row-sharded run would need an all-reduce of the "
                                   "M x (p + 1) gradient block per pass, which is not built");
    if (n < 1 || p < 1 || ldx < n) fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d ldx=%lld", (long long)n, p, (long long)ldx);
    if (!logit_fold_models(p))
        fail(OEMB200_EUNSUPPORTED, "binomial xval runs on the fused slab pass, which covers 8 <= p <= 2048 (p = %d)", p);
    if (nfolds < 2 || !foldid) fail(OEMB200_EINVAL, "xval needs nfolds >= 2 and foldid");
    if (!res->cvm || !res->cvsd) fail(OEMB200_EINVAL, "xval needs cvm / cvsd result buffers");
    int measure = 0;
    if (!type_measure || strcmp(type_measure, "deviance") == 0) measure = 0;
    else if (strcmp(type_measure, "class") == 0) measure = 1;
    else if (strcmp(type_measure, "mse") == 0) measure = 2;
    else if (strcmp(type_measure, "mae") == 0) measure = 3;
    else if (strcmp(type_measure, "auc") == 0)
        fail(OEMB200_EINVAL, "type_measure \"auc\" needs per-fold ranks: use cv_oem");
    else fail(OEMB200_EINVAL, "type_measure must be \"deviance\", \"class\", \"mse\" or \"mae\" for the binomial family");
    const int icpt = s->intercept ? 1 : 0, q = p + icpt;
    const bool stdz = s->standardize != 0;
    const int F = nfolds, M = F + 1;
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, q, /*zero_w0=*/true);

    XvalSystems xs;
    xval_build_systems(cx, x, n, p, ldx, y, nullptr, F, foldid, icpt, stdz, 0.25, xs);
    for (int g = 0; g < M; ++g)
        if (!(xs.hn[g] > q)) fail(OEMB200_EINVAL, "dimension of x larger than number of observations");
    const int64_t npad = xs.npad;
    double lmax = 0.0;      // init_oem: the X entries of XY = (X'y o colsq_inv) / n of the full data
    for (int j = 0; j < p; ++j) lmax = std::max(lmax, std::fabs(xs.hXY[icpt + j]));
    su.build_lambdas(s, lmax, /*logistic_fudge=*/true);

    // ---- slab copy of the fold-sorted X and the fold of every sorted row (0 = padding) ----
    DBuf<double> slabs(logit_fold_doubles(npad, p));
    {
        const size_t t_r = tm.start(&cx.st.ms_relayout);
        logit_fold_relayout(cx, xs.Xs.p, npad, p, npad, slabs.p);
        tm.stop(t_r);
    }
    DBuf<int> d_rowfold(npad);
    {
        std::vector<int> hf(npad, 0);
        for (int k = 0; k < F; ++k) std::fill(hf.begin() + xs.off[k], hf.begin() + xs.off[k] + xs.cnt[k], k + 1);
        d_rowfold.upload(hf.data(), npad, cx.stream);
        cx.sync();                                  // hf is a host temporary
    }

    // ---- device state: one slice per model ----
    const int L = su.Lmax, P = su.P;
    std::vector<double> pf(q, 0.0);
    for (int j = 0; j < p; ++j) pf[icpt + j] = s->penalty_factor[j];
    DBuf<double> d_pf(q), d_B((size_t)M * p), d_b0(M), d_G((size_t)M * (p + 1)), d_XY((size_t)M * q), d_d(M);
    DBuf<double> d_iter((size_t)M * 2 * q), d_path((size_t)M * P * L * q), d_lams((size_t)P * L), d_prob(npad);
    DBuf<double> d_losspart(1024), d_losstot(2);
    DBuf<long long> d_iters_total(1);
    DBuf<int> d_niter(M), d_lz(M), d_conv(M);
    DBuf<unsigned long long> d_clk(1);
    d_prob.zero(cx.stream);
    d_path.zero(cx.stream);
    d_iters_total.zero(cx.stream);
    d_clk.zero(cx.stream);
    d_pf.upload(pf.data(), q, cx.stream);
    {
        std::vector<double> lam_flat((size_t)P * L, 0.0);
        for (int pp = 0; pp < P; ++pp)
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
    PinnedFlags flags(M);
    Scratches scratch(M);
    fill_common_outputs(su, res);
    memset(res->beta, 0, sizeof(double) * (size_t)P * (p + 1) * L);
    const double *cinv_all = stdz ? xs.cinv.p : nullptr;
    const bool want_loss = s->compute_loss && res->loss;

    std::vector<int> par0(M), it_m(M);
    std::vector<char> active(M), broke(M);
    for (int pp = 0; pp < P; ++pp) {
        // init(): beta = 0 for every model, so the first pass multiplies X with b = 0, b0 = 0
        OEM_CUDA(cudaMemsetAsync(d_iter.p, 0, d_iter.n * sizeof(double), cx.stream));
        OEM_CUDA(cudaMemsetAsync(d_B.p, 0, d_B.n * sizeof(double), cx.stream));
        OEM_CUDA(cudaMemsetAsync(d_b0.p, 0, d_b0.n * sizeof(double), cx.stream));
        std::fill(par0.begin(), par0.end(), 0);
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            OEM_CUDA(cudaMemsetAsync(d_conv.p, 0, sizeof(int) * M, cx.stream));
            std::fill(active.begin(), active.end(), 1);
            std::fill(broke.begin(), broke.end(), 0);
            for (int k = 0;; ++k) {
                const bool pass = !(k == 0 && i > 0);      // the reference skips the data pass on a warm lambda's first iteration
                if (pass) {
                    const size_t t1 = tm.start(&cx.st.ms_irls_xb);
                    const int sweeps = logit_fold_launch(cx, slabs.p, npad, p, d_B.p, d_b0.p, xs.ys.p, d_rowfold.p, M,
                                                         d_conv.p, &active, want_loss ? d_prob.p : nullptr, d_G.p);
                    tm.stop(t1);
                    cx.st.gemv_bytes += 8.0 * (double)npad * p * sweeps;
                }
                for (int m = 0; m < M; ++m) {
                    if (!active[m]) continue;
                    const size_t qm = (size_t)m * q;
                    double *base = d_iter.p + 2 * qm;
                    double *cur = base + (size_t)((par0[m] + k) & 1) * q, *nxt = base + (size_t)((par0[m] + k + 1) & 1) * q;
                    const double *cinv_m = cinv_all ? cinv_all + (size_t)m * p : nullptr;
                    PathProblem pr;
                    pr.q = q; pr.ngram = 1; pr.XX = xs.XX.p + qm * q; pr.XY = d_XY.p + qm; pr.d = d_d.p + m;
                    pr.compute_eig = (k == 0 && i == 0); pr.eig_factor = 1.0005; pr.eig_tol = 1e-10;
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
                    pr.beta_out = nxt; pr.niter_out = d_niter.p + m; pr.lanczos_steps = d_lz.p + m;
                    pr.scratch = scratch.s[m];
                    pr.skip = d_conv.p + m;
                    if (pass) {
                        pr.xy_grad = d_G.p + (size_t)m * (p + 1); pr.xy_cinv = cinv_m; pr.xy_n = xs.hn[m];
                        pr.xy_icpt = icpt; pr.xy_out = d_XY.p + qm;
                    }
                    pr.t_acc = d_clk.p;
                    pr.irls_conv = d_conv.p + m; pr.irls_host_flag = flags.p + m; pr.irls_iters_total = d_iters_total.p;
                    pr.irls_tol = o->irls_tol; pr.irls_cinv = cinv_m; pr.irls_p = p; pr.irls_icpt = icpt;
                    pr.irls_b = d_B.p + (size_t)m * p; pr.irls_b0 = d_b0.p + m;
                    path_launch(cx, pr);
                }
                cx.sync();                                   // the one host round trip of the round
                int left = 0;
                for (int m = 0; m < M; ++m) {
                    if (!active[m]) continue;
                    if (flags.p[m]) { active[m] = 0; broke[m] = 1; it_m[m] = k; }
                    else left++;
                }
                if (!left) break;
                if (k + 1 >= o->irls_maxit) {
                    for (int m = 0; m < M; ++m)
                        if (active[m]) { active[m] = 0; it_m[m] = o->irls_maxit - 1; }
                    break;
                }
            }
            for (int m = 0; m < M; ++m) {
                if (m == 0) res->niter[(size_t)pp * L + i] = (broke[0] ? it_m[0] : o->irls_maxit) + 1;
                par0[m] = (par0[m] + it_m[m] + 1) & 1;       // the iterate the model's last executed iteration produced
                const double *fin = d_iter.p + (size_t)m * 2 * q + (size_t)par0[m] * q;
                OEM_CUDA(cudaMemcpyAsync(d_path.p + (((size_t)m * P + pp) * L + i) * q, fin, sizeof(double) * q,
                                         cudaMemcpyDeviceToDevice, cx.stream));
            }
            if (want_loss) {          // padding rows hold prob = 0 and y = 0: their terms are log(1) = 0
                logistic_loss_launch(cx, xs.ys.p, d_prob.p, npad, d_losspart.p, d_losstot.p);
                double h[2];
                d_losstot.download(h, 2, cx.stream);
                cx.sync();
                res->loss[(size_t)pp * L + i] = h[0];
            }
        }
    }

    // ---- full model back to the host, un-scaled (get_beta) ----
    std::vector<double> hpath((size_t)P * L * q);
    long long iters_total = 0;
    double dval = 0.0;
    unsigned long long hclk = 0;
    OEM_CUDA(cudaMemcpyAsync(hpath.data(), d_path.p, hpath.size() * 8, cudaMemcpyDeviceToHost, cx.stream));
    d_iters_total.download(&iters_total, 1, cx.stream);
    d_d.download(&dval, 1, cx.stream);
    d_clk.download(&hclk, 1, cx.stream);
    cx.sync();
    cx.st.ms_path += (double)hclk * 1e-6;
    cx.st.d2h_bytes += (int64_t)hpath.size() * 8;
    cx.st.total_oem_iters += iters_total;
    for (int pp = 0; pp < P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const double *raw = &hpath[((size_t)pp * L + i) * q];
            double *out = res->beta + ((size_t)pp * L + i) * (p + 1);
            if (icpt) out[0] = raw[0];
            for (int j = 0; j < p; ++j) out[1 + j] = stdz ? raw[icpt + j] * xs.hcinv[j] : raw[icpt + j];
        }
    *res->d = dval;

    // ---- CV scoring: fold k's rows against fold model k ----
    const int nc = P * L, ncld = cv_ncld(nc);
    DBuf<double> dB((size_t)F * p * ncld), db0((size_t)F * ncld), out3(3 * (size_t)nc);
    DBuf<int> d_nlam(P);
    d_nlam.upload(su.nlam_run.data(), P, cx.stream);
    cv_build_coef_launch(cx, d_path.p, xs.cinv.p, F, P, L, p, q, icpt, stdz, d_nlam.p, dB.p, db0.p);
    std::vector<std::array<int64_t, 3>> cs;
    for (int k = 0; k < F; ++k) cs.push_back({xs.off[k], xs.off[k + 1], xs.off[k] + xs.cnt[k]});
    cvscore_binomial_launch(cx, xs.Xs.p, npad, p, npad, xs.ys.p, F, cs, dB.p, db0.p, nc, measure, out3.p);
    std::vector<double> h3(3 * (size_t)nc);
    out3.download(h3.data(), h3.size(), cx.stream);
    cx.sync();
    const double n_tot = xs.hn[0];
    for (int pp = 0; pp < P; ++pp)
        for (int i = 0; i < L; ++i) {
            const int c = pp * L + i;
            const bool live = i < su.nlam_run[pp];
            res->cvm[c] = live ? h3[nc + c] : 0.0;
            res->cvsd[c] = live ? std::sqrt(h3[2 * nc + c] / (n_tot - 1.0)) / std::sqrt(n_tot) : 0.0;
        }
    finish_stats(cx, tm, t_total, res);
}

}  // namespace oemb200
