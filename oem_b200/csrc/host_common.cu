// host_common.cu -- see host_common.h.  Host logic only (no kernels): penalty / group / lambda
// bookkeeping restated from the reference's entry functions, its device tables, the path-kernel round trip, the
// write-back of the raw iterates into the reported beta, and the logistic init step and IRLS loop.
#include <algorithm>
#include <cstring>
#include "host_common.h"

namespace oemb200 {

static const char *const kPenaltyNames[] = {"lasso", "ols", "elastic.net", "scad", "scad.net", "mcp", "mcp.net",
                                            "grp.lasso", "grp.lasso.net", "grp.mcp", "grp.scad", "grp.mcp.net",
                                            "grp.scad.net", "sparse.grp.lasso"};

int penalty_id(const char *name) {
    if (!name) return -1;
    for (int i = 0; i < 14; ++i)
        if (strcmp(name, kPenaltyNames[i]) == 0) return i;
    return -1;
}
bool penalty_is_net(int id) { return id >= 0 && strstr(kPenaltyNames[id], ".net") != nullptr; }
bool penalty_is_group(int id) { return id >= 0 && strstr(kPenaltyNames[id], "grp") != nullptr; }

std::vector<double> linspace_eigen(int N, double lo, double hi) {
    std::vector<double> v((size_t)std::max(N, 0));
    if (N <= 0) return v;
    if (N == 1) { v[0] = lo; return v; }
    const double step = (hi - lo) / double(N - 1);
    if (std::fabs(hi) < std::fabs(lo)) {
        for (int i = 0; i < N; ++i) v[i] = hi - double(N - 1 - i) * step;
        v[0] = lo;
    } else {
        for (int i = 0; i < N; ++i) v[i] = lo + double(i) * step;
        v[N - 1] = hi;
    }
    return v;
}

std::vector<double> lambda_base(double lmax, int nl, double lmin_ratio) {
    const double lmin = lmin_ratio * lmax;
    std::vector<double> v = linspace_eigen(nl, std::log(lmax), std::log(lmin));
    for (auto &x : v) x = std::exp(x);
    return v;
}

bool stop_rule_host(const std::vector<double> &cur, const std::vector<double> &prev, double tol) {
    for (size_t i = 0; i < cur.size(); ++i) {
        const double ac = std::fabs(cur[i]), ap = std::fabs(prev[i]);
        if ((ac > 1e-13 && ap <= 1e-13) || (ac <= 1e-13 && ap > 1e-13)) return false;
        if (ac > 1e-13 && ap > 1e-13 && std::fabs((cur[i] - prev[i]) / prev[i]) > tol) return false;
    }
    return true;
}

void Setup::parse(const oemb200_spec *s, int q, int scan, bool zero_w0) {
    if (!s) fail(OEMB200_EINVAL, "spec is NULL");
    if (s->n_penalty < 1 || !s->penalty) fail(OEMB200_EINVAL, "no penalty given");
    P = s->n_penalty;
    alpha = s->alpha;
    tau = s->tau;
    pen.resize(P);
    gamma.resize(P);
    any_group = false;
    for (int i = 0; i < P; ++i) {
        pen[i] = penalty_id(s->penalty[i]);
        if (pen[i] < 0) fail(OEMB200_EINVAL, "unknown penalty '%s'", s->penalty[i] ? s->penalty[i] : "(null)");
        if (!s->gamma || s->n_gamma < 1) fail(OEMB200_EINVAL, "gamma missing");
        if (s->n_gamma != 1 && s->n_gamma != P) fail(OEMB200_EINVAL, "gamma must have length 1 or one per penalty");
        gamma[i] = s->n_gamma == 1 ? s->gamma[0] : s->gamma[i];
        any_group = any_group || penalty_is_group(pen[i]);
    }
    if (!s->penalty_factor) fail(OEMB200_EINVAL, "penalty_factor is NULL");
    lambda_given = s->n_lambda && s->lambda && s->n_lambda[0] >= 1;
    if (lambda_given) {
        for (int i = 0; i < P; ++i)
            if (s->n_lambda[i] != s->n_lambda[0] || !s->lambda[i])
                fail(OEMB200_EINVAL, "user lambda sequences must have one equal-length vector per penalty");
        Lmax = s->n_lambda[0];
    } else {
        if (s->nlambda < 1) fail(OEMB200_EINVAL, "nlambda must be >= 1");
        Lmax = s->nlambda;
    }
    // get_group_indexes(): src/oem_dense.h:421-456
    unique.clear(); ptr.assign(1, 0); idx.clear(); gw.clear();
    cover.assign(q, 0);
    if (any_group) {
        if (!s->groups || !s->unique_groups || s->n_unique_groups < 1)
            fail(OEMB200_EINVAL, "group penalties need groups and unique_groups");
        const int ns = std::min(scan, s->n_groups);
        for (int g = 0; g < s->n_unique_groups; ++g) {
            unique.push_back(s->unique_groups[g]);
            for (int v = 0; v < ns && v < q; ++v)
                if (s->groups[v] == s->unique_groups[g]) { idx.push_back(v); cover[v] = 1; }
            ptr.push_back((int)idx.size());
        }
        if (s->n_group_weights >= 1) {
            if (s->n_group_weights != s->n_unique_groups)
                fail(OEMB200_EINVAL, "group_weights must have one entry per unique group");
            gw.assign(s->group_weights, s->group_weights + s->n_group_weights);
        } else {
            for (int g = 0; g < s->n_unique_groups; ++g) {
                double w = std::sqrt(double(ptr[g + 1] - ptr[g]));
                if (zero_w0 && unique[g] == 0) w = 0.0;
                gw.push_back(w);
            }
        }
    }
}

void Setup::build_lambdas(const oemb200_spec *s, double lmax, bool logistic_fudge) {
    lam.assign(P, {});
    nlam_run.assign(P, 0);
    std::vector<double> base;
    if (!lambda_given) base = lambda_base(lmax, s->nlambda, s->lambda_min_ratio);
    for (int pp = 0; pp < P; ++pp) {
        if (lambda_given) lam[pp].assign(s->lambda[pp], s->lambda[pp] + s->n_lambda[pp]);
        else if (penalty_is_net(pen[pp])) {
            lam[pp] = base;
            const bool ncv = pen[pp] == OEMB200_PEN_MCP_NET || pen[pp] == OEMB200_PEN_SCAD_NET ||
                             pen[pp] == OEMB200_PEN_GRP_MCP_NET || pen[pp] == OEMB200_PEN_GRP_SCAD_NET;
            if (logistic_fudge && ncv) {
                // src/oem_logistic_dense.cpp:214-219 (gamma is the scalar gamma of the call)
                const double fact = 3.5 - std::min(3.5, gamma[0]) * 5.71425 / 8.0;
                const double a8 = std::pow(s->alpha, 0.8);
                for (auto &x : lam[pp]) x = fact * x / a8;
            } else {
                for (auto &x : lam[pp]) x = x / s->alpha;
            }
        } else lam[pp] = base;
        nlam_run[pp] = (pen[pp] == OEMB200_PEN_OLS) ? 1 : (int)lam[pp].size();
    }
}

PenaltyTables::PenaltyTables(Ctx &cx, const Setup &su, const oemb200_spec *s, int p, int icpt, double lam_scale)
    : q(p + icpt), Lmax(su.Lmax), ngroups(su.any_group ? (int)su.unique.size() : 0),
      ngidx(su.any_group ? (int)su.idx.size() : 0), h_pf(q, 0.0) {
    for (int pp = 0; pp < su.P; ++pp)
        for (double x : su.lam[pp]) h_lam.push_back(x / lam_scale);
    for (int j = 0; j < p; ++j) h_pf[icpt + j] = s->penalty_factor[j];
    lambdas.alloc(h_lam.size());
    lambdas.upload(h_lam.data(), h_lam.size(), cx.stream);
    pen_fact.alloc(q);
    pen_fact.upload(h_pf.data(), q, cx.stream);
    if (su.any_group) {
        unique.alloc(su.unique.size()); unique.upload(su.unique.data(), su.unique.size(), cx.stream);
        ptr.alloc(su.ptr.size());       ptr.upload(su.ptr.data(), su.ptr.size(), cx.stream);
        idx.alloc(std::max<size_t>(1, su.idx.size()));
        if (!su.idx.empty()) idx.upload(su.idx.data(), su.idx.size(), cx.stream);
        gw.alloc(su.gw.size());         gw.upload(su.gw.data(), su.gw.size(), cx.stream);
        cover.alloc(q);                 cover.upload(su.cover.data(), q, cx.stream);
    }
}

// the penalty-factor and group fields of a path launch
static void use_tables(PathProblem &pr, const PenaltyTables &tb) {
    pr.pen_fact = tb.pen_fact.p;
    pr.ngroups = tb.ngroups;
    pr.ngidx = tb.ngidx;
    pr.unique_groups = tb.unique.p; pr.grp_ptr = tb.ptr.p; pr.grp_idx = tb.idx.p;
    pr.group_weights = tb.gw.p; pr.grp_cover = tb.cover.p;
}

void run_paths(Ctx &cx, const Setup &su, const PenaltyTables &tb, const oemb200_opts *o, int ngram, const double *XX,
               const double *XY, double eig_factor, bool accelerate, const double *post_scale_dev, PathBuffers &pb) {
    const int P = su.P, L = su.Lmax, q = tb.q;
    const int nchains = ngram * P;
    pb.beta_out.alloc((size_t)nchains * L * q);
    pb.beta_out.zero(cx.stream);
    pb.niter.alloc((size_t)nchains * L);
    pb.niter.zero(cx.stream);
    pb.d.alloc(ngram);
    pb.lz.alloc(ngram);
    pb.lz.zero(cx.stream);

    PathProblem pp;
    pp.q = q; pp.ngram = ngram; pp.XX = XX; pp.XY = XY; pp.d = pb.d.p;
    pp.compute_eig = true; pp.eig_factor = eig_factor;
    for (int g = 0; g < ngram; ++g)
        for (int k = 0; k < P; ++k) {
            ChainDesc c;
            c.gram = g; c.penalty = su.pen[k]; c.nlam = su.nlam_run[k]; c.lam_off = k * L;
            c.alpha = su.alpha; c.gamma = su.gamma[k]; c.tau = su.tau; c.out_off = g * P + k;
            pp.chains.push_back(c);
        }
    pp.lambdas = tb.lambdas.p; pp.Lmax = L;
    use_tables(pp, tb);
    pp.post_scale = post_scale_dev;
    pp.maxit = o->maxit; pp.tol = o->tol; pp.accelerate = accelerate;
    pp.beta_out = pb.beta_out.p; pp.niter_out = pb.niter.p; pp.lanczos_steps = pb.lz.p;

    path_launch(cx, pp);

    pb.h_beta.resize((size_t)nchains * L * q);
    pb.h_niter.resize((size_t)nchains * L);
    pb.h_d.resize(ngram);
    pb.h_lz.resize(ngram);
    pb.beta_out.download(pb.h_beta.data(), pb.h_beta.size(), cx.stream);
    pb.niter.download(pb.h_niter.data(), pb.h_niter.size(), cx.stream);
    pb.d.download(pb.h_d.data(), ngram, cx.stream);
    pb.lz.download(pb.h_lz.data(), ngram, cx.stream);
    cx.sync();
    cx.st.d2h_bytes += (int64_t)(pb.h_beta.size() * 8 + pb.h_niter.size() * 4);
    for (int v : pb.h_niter) cx.st.total_oem_iters += v;
    for (int v : pb.h_lz) cx.st.lanczos_steps += v;
}

// One IRLS iteration's path launch (src/oem_logistic_dense.h:999-1033) for model m: lambda i of penalty pp, one chain, warm
// started from cur, eigenvalue factor 1.0005 (recomputed when compute_eig), predicated on *m.conv.  Its last step is the
// outer stop rule on (nxt, cur), whose verdict goes to *m.conv and *verdict, and b / b0 from nxt.  With grad (device,
// [sum r, X'r] over n_rows rows) it first forms XY = XX cur + grad / n_rows (scaled by cinv); without, it keeps the XY of
// the model's previous data pass.
static PathProblem irls_path_problem(const PenaltyTables &tb, const Setup &su, int pp, int i, const oemb200_opts *o,
                                     const IrlsModel &m, const double *cur, double *nxt, volatile int *verdict,
                                     bool compute_eig, const double *grad, double n_rows) {
    PathProblem pr;
    pr.q = tb.q; pr.ngram = 1;
    pr.XX = m.XX; pr.XY = m.XY; pr.d = m.d;
    pr.compute_eig = compute_eig; pr.eig_factor = 1.0005;
    ChainDesc c;
    c.gram = 0; c.penalty = su.pen[pp]; c.nlam = 1; c.lam_off = 0; c.alpha = su.alpha;
    c.gamma = su.gamma[pp]; c.tau = su.tau; c.out_off = 0;
    pr.chains.push_back(c);
    pr.lambdas = tb.lambdas.p + (size_t)pp * tb.Lmax + i; pr.Lmax = 1;
    use_tables(pr, tb);
    pr.beta_init = cur; pr.beta_out = nxt;
    pr.maxit = o->maxit; pr.tol = o->tol;
    pr.niter_out = m.niter; pr.lanczos_steps = m.lz; pr.scratch = m.scratch;
    pr.skip = m.conv;
    pr.t_acc = m.t_acc;
    pr.irls_conv = m.conv; pr.irls_host_flag = verdict; pr.irls_iters_total = m.iters_total;
    pr.irls_tol = o->irls_tol; pr.irls_cinv = m.cinv; pr.irls_p = tb.q - m.icpt; pr.irls_icpt = m.icpt;
    pr.irls_b = m.b; pr.irls_b0 = m.b0;
    if (grad) { pr.xy_grad = grad; pr.xy_cinv = m.cinv; pr.xy_n = n_rows; pr.xy_icpt = m.icpt; pr.xy_out = m.XY; }
    return pr;
}

void write_beta(const Setup &su, const double *raw, int p, int icpt, const double *cinv, oemb200_result *res) {
    const int L = su.Lmax, q = p + icpt;
    memset(res->beta, 0, sizeof(double) * (size_t)su.P * (p + 1) * L);
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) {
            const double *r = raw + ((size_t)pp * L + i) * q;
            double *out = res->beta + ((size_t)pp * L + i) * (p + 1);
            if (icpt) out[0] = r[0];
            for (int j = 0; j < p; ++j) out[1 + j] = cinv ? r[icpt + j] * cinv[j] : r[icpt + j];
        }
}

LogisticInit logistic_init(Ctx &cx, int64_t n, int p, int q, bool stdz, const std::function<void(double *)> &colstats,
                           const char *refusal) {
    LogisticInit r;
    const size_t nb = 3 * (size_t)p + 1;
    r.stats.alloc(nb);
    PhaseTimers &tm = *cx.tm;
    const size_t t_c = tm.start(&cx.st.ms_colstats);
    colstats(r.stats.p);
    tm.stop(t_c);
    const double nd = (double)n;
    OEM_CUDA(cudaMemcpyAsync(r.stats.p + 3 * (size_t)p, &nd, 8, cudaMemcpyHostToDevice, cx.stream));
    const size_t t_ar = tm.start(&cx.st.ms_allreduce);
    cx.all_reduce(r.stats.p, (int64_t)nb);
    tm.stop(t_ar);
    std::vector<double> h(nb);
    r.stats.download(h.data(), nb, cx.stream);
    cx.sync();
    r.n_tot = h[3 * (size_t)p];
    if (!(r.n_tot > q)) fail(OEMB200_EUNSUPPORTED, "%s", refusal);
    // 1 / sd of every column from its sum of squares (uncentred, divisor n - 1, a zero column keeps scale 1)
    r.cinv.assign(p, 1.0);
    for (int j = 0; j < p; ++j) {
        if (stdz) {
            double sq = h[2 * (size_t)p + j] / (r.n_tot - 1.0);
            if (sq == 0.0) sq = 1.0;
            r.cinv[j] = 1.0 / std::sqrt(sq);
        }
        double v = h[(size_t)p + j];
        if (stdz) v *= r.cinv[j];
        r.lmax = std::max(r.lmax, std::fabs(v / r.n_tot));
    }
    return r;
}

IrlsLoop::IrlsLoop(Ctx &cx, const Setup &su, const PenaltyTables &tb, const oemb200_opts *o, int M, int icpt, bool speculate)
    : b((size_t)M * (tb.q - icpt)), b0(M), conv(M), path((size_t)M * su.P * su.Lmax * tb.q), active(M), cx_(cx), su_(su),
      tb_(tb), o_(o), M_(M), q_(tb.q), speculate_(speculate), iter_((size_t)M * 2 * tb.q), niter_(M), lz_(M),
      iters_total_(1), scratch_(M), md_(M), flag_(4 * M), par0_(M), last_(M), niter_h_(M) {
    if (speculate && M > 1) fail(OEMB200_EINVAL, "IRLS loop: only a single model may be enqueued ahead (M = %d)", M);
    ev_[0] = event_acquire();
    ev_[1] = event_acquire();
    iters_total_.zero(cx.stream);
    path.zero(cx.stream);
    for (int m = 0; m < M; ++m) {
        IrlsModel &d = md_[m];
        d.niter = niter_.p + m; d.lz = lz_.p + m; d.scratch = scratch_.s[m]; d.conv = conv.p + m;
        d.iters_total = iters_total_.p; d.icpt = icpt; d.b = b.p + (size_t)m * (q_ - icpt); d.b0 = b0.p + m;
    }
}

IrlsLoop::~IrlsLoop() { event_release(ev_[0]); event_release(ev_[1]); }

void IrlsLoop::set_model(int m, const double *XX, double *XY, double *d, const double *cinv, unsigned long long *t_acc) {
    md_[m].XX = XX; md_[m].XY = XY; md_[m].d = d; md_[m].cinv = cinv; md_[m].t_acc = t_acc;
}

void IrlsLoop::path_step(int m, bool compute_eig, const double *grad, double n_rows) {
    double *slots = iter_.p + (size_t)m * 2 * q_;
    const int cur = (par0_[m] + k_) & 1;
    path_launch(cx_, irls_path_problem(tb_, su_, pp_, i_, o_, md_[m], slots + (size_t)cur * q_, slots + (size_t)(cur ^ 1) * q_,
                                       flag_.p + (gi_ & 3) * M_ + m, compute_eig, grad, n_rows));
}

double *IrlsLoop::final_iterate(int m) { return iter_.p + ((size_t)m * 2 + par0_[m]) * q_; }

// Waits for round g (iteration k of the lambda) and reads the verdicts of the models it ran; false once none is left.
// Without speculation nothing is enqueued behind round g, and a stream sync is cheaper than an event record per round.
bool IrlsLoop::wait_round(long long g, int k) {
    if (speculate_) {
        cx_.st.host_syncs += 1;
        OEM_CUDA(cudaEventSynchronize(ev_[g & 1]));
    } else {
        cx_.sync();
    }
    const int *verdict = flag_.p + (g & 3) * M_;
    bool left = false;
    for (int m = 0; m < M_; ++m) {
        if (!active[m]) continue;
        if (verdict[m]) { active[m] = 0; last_[m] = k; niter_h_[m] = k + 1; }
        else left = true;
    }
    return left;
}

// niter as the reference reports it: executed iterations + 1 on convergence, irls_maxit + 1 at the cap
void IrlsLoop::run(oemb200_result *res, const std::function<void(int, int, bool)> &round,
                   const std::function<void(int, int)> &lambda_end) {
    const int maxit = o_->irls_maxit, L = su_.Lmax;
    auto enqueue = [&](int k) {
        k_ = k;
        round(i_, k, !(k == 0 && i_ > 0));
        if (speculate_) OEM_CUDA(cudaEventRecord(ev_[gi_ & 1], cx_.stream));
        ++gi_;
    };
    for (pp_ = 0; pp_ < su_.P; ++pp_) {
        iter_.zero(cx_.stream);                          // init(): beta = 0, on_lam_1 = true
        b.zero(cx_.stream);
        b0.zero(cx_.stream);
        std::fill(par0_.begin(), par0_.end(), 0);
        for (i_ = 0; i_ < su_.nlam_run[pp_]; ++i_) {
            conv.zero(cx_.stream);
            std::fill(active.begin(), active.end(), 1);
            int it = 0;
            enqueue(0);
            for (;;) {
                // round `it` is in the stream (the last one, unless round it + 1 is enqueued ahead of its verdict)
                const bool ahead = speculate_ && it + 1 < maxit;
                const oemb200_stats before = cx_.st;
                if (ahead) enqueue(it + 1);
                if (!wait_round(gi_ - 1 - (ahead ? 1 : 0), it)) {
                    if (ahead) {           // the speculative round found the lambda converged: nothing of it ran
                        cx_.st.data_passes = before.data_passes; cx_.st.xb_launches = before.xb_launches;
                        cx_.st.gemv_bytes = before.gemv_bytes; cx_.st.allreduce_calls = before.allreduce_calls;
                        cx_.st.allreduce_doubles = before.allreduce_doubles;
                    }
                    break;
                }
                if (++it >= maxit) {
                    for (int m = 0; m < M_; ++m)
                        if (active[m]) { active[m] = 0; last_[m] = maxit - 1; niter_h_[m] = maxit + 1; }
                    break;
                }
                if (!ahead) enqueue(it);
            }
            for (int m = 0; m < M_; ++m) par0_[m] = (par0_[m] + last_[m] + 1) & 1;
            lambda_end(pp_, i_);
            for (int m = 0; m < M_; ++m)
                OEM_CUDA(cudaMemcpyAsync(path.p + (((size_t)m * su_.P + pp_) * L + i_) * q_, final_iterate(m),
                                         sizeof(double) * q_, cudaMemcpyDeviceToDevice, cx_.stream));
            res->niter[(size_t)pp_ * L + i_] = niter_h_[0];
        }
    }
}

void IrlsLoop::write_path(const double *cinv, oemb200_result *res) {
    const int icpt = md_[0].icpt, p = q_ - icpt;
    std::vector<double> hpath((size_t)su_.P * su_.Lmax * q_);
    long long iters_total = 0;
    double dval = 0.0;
    OEM_CUDA(cudaMemcpyAsync(hpath.data(), path.p, hpath.size() * 8, cudaMemcpyDeviceToHost, cx_.stream));
    OEM_CUDA(cudaMemcpyAsync(&iters_total, iters_total_.p, sizeof iters_total, cudaMemcpyDeviceToHost, cx_.stream));
    OEM_CUDA(cudaMemcpyAsync(&dval, md_[0].d, sizeof dval, cudaMemcpyDeviceToHost, cx_.stream));
    cx_.sync();
    cx_.st.d2h_bytes += (int64_t)hpath.size() * 8;
    cx_.st.total_oem_iters += iters_total;
    write_beta(su_, hpath.data(), p, icpt, cinv, res);
    *res->d = dval;
}

}  // namespace oemb200
