// host_common.cu -- see host_common.h.  Host logic only (no kernels): penalty / group / lambda
// bookkeeping restated from the reference's entry functions, its device tables, the path-kernel round trip and the
// write-back of the raw iterates into the reported beta.
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

PathProblem irls_path_problem(const PenaltyTables &tb, const Setup &su, int pp, int i, const oemb200_opts *o, const IrlsModel &m,
                              const double *cur, double *nxt, volatile int *verdict, bool compute_eig, const double *grad,
                              double n_rows) {
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

void irls_write_path(Ctx &cx, const Setup &su, int p, int icpt, const double *path_dev, const long long *iters_total_dev,
                     const double *d_dev, const double *cinv, oemb200_result *res) {
    std::vector<double> hpath((size_t)su.P * su.Lmax * (p + icpt));
    long long iters_total = 0;
    double dval = 0.0;
    OEM_CUDA(cudaMemcpyAsync(hpath.data(), path_dev, hpath.size() * 8, cudaMemcpyDeviceToHost, cx.stream));
    OEM_CUDA(cudaMemcpyAsync(&iters_total, iters_total_dev, sizeof iters_total, cudaMemcpyDeviceToHost, cx.stream));
    OEM_CUDA(cudaMemcpyAsync(&dval, d_dev, sizeof dval, cudaMemcpyDeviceToHost, cx.stream));
    cx.sync();
    cx.st.d2h_bytes += (int64_t)hpath.size() * 8;
    cx.st.total_oem_iters += iters_total;
    write_beta(su, hpath.data(), p, icpt, cinv, res);
    *res->d = dval;
}

}  // namespace oemb200
