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
//      coefficients (PathProblem::irls_*).  The rounds are IrlsLoop's (host_common.h), the outer loop of the dense and
//      sparse drivers, with M models and no speculation: the host waits once per round and reads the M verdicts; a
//      converged model idles until lambda advances, so every model does exactly the arithmetic of a separate fit;
//   3. one fold-segmented scoring GEMM with the binomial epilogue (cvscore_binomial_launch).
// The reference's logistic quirks come along: no data pass on the first IRLS iteration of every lambda after the first,
// eigenvalue factor 1.0005, uncentred standardisation from each model's own rows.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include "host_common.h"

namespace oemb200 {

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
    PenaltyTables tb(cx, su, s, p, icpt);
    DBuf<double> d_G((size_t)M * (p + 1)), d_XY((size_t)M * q), d_d(M), d_prob(npad);
    DBuf<unsigned long long> d_clk(1);
    d_prob.zero(cx.stream);
    d_clk.zero(cx.stream);
    IrlsLoop loop(cx, su, tb, o, M, icpt, /*speculate=*/false);
    for (int m = 0; m < M; ++m)
        loop.set_model(m, xs.XX.p + (size_t)m * q * q, d_XY.p + (size_t)m * q, d_d.p + m,
                       stdz ? xs.cinv.p + (size_t)m * p : nullptr, d_clk.p);
    fill_common_outputs(su, res);
    const bool want_loss = s->compute_loss && res->loss;

    loop.run(res, [&](int i, int k, bool pass) {
        if (pass) {
            const size_t t1 = tm.start(&cx.st.ms_irls_xb);
            const int sweeps = logit_fold_launch(cx, slabs.p, npad, p, loop.b.p, loop.b0.p, xs.ys.p, d_rowfold.p, M,
                                                 loop.conv.p, &loop.active, want_loss ? d_prob.p : nullptr, d_G.p);
            tm.stop(t1);
            cx.st.gemv_bytes += 8.0 * (double)npad * p * sweeps;
        }
        for (int m = 0; m < M; ++m)
            if (loop.active[m])
                loop.path_step(m, k == 0 && i == 0, pass ? d_G.p + (size_t)m * (p + 1) : nullptr, xs.hn[m]);
    }, [&](int pp, int i) {
        // padding rows hold prob = 0 and y = 0: their terms are log(1) = 0
        if (want_loss) res->loss[(size_t)pp * L + i] = logistic_loss(cx, xs.ys.p, d_prob.p, npad);
    });

    // ---- full model back to the host, un-scaled (get_beta) ----
    unsigned long long hclk = 0;
    d_clk.download(&hclk, 1, cx.stream);
    loop.write_path(stdz ? xs.hcinv.data() : nullptr, res);
    cx.st.ms_path += (double)hclk * 1e-6;

    // ---- CV scoring: fold k's rows against fold model k ----
    const int nc = P * L, ncld = cv_ncld(nc);
    DBuf<double> dB((size_t)F * p * ncld), db0((size_t)F * ncld), out3(3 * (size_t)nc);
    DBuf<int> d_nlam(P);
    d_nlam.upload(su.nlam_run.data(), P, cx.stream);
    cv_build_coef_launch(cx, loop.path.p, xs.cinv.p, F, P, L, p, q, icpt, stdz, d_nlam.p, dB.p, db0.p);
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
