// host_common.h -- host-side bookkeeping shared by the five entry points: penalty / group / lambda
// setup (the part of the reference's entry functions that is not arithmetic on X), and the helper
// that runs a set of chains through the path kernel and brings the raw iterates back.
#pragma once
#include <cmath>
#include <string>
#include <vector>
#include "runtime.h"

namespace oemb200 {

int penalty_id(const char *name);
bool penalty_is_net(int id);     // name contains ".net"  (src/oem_dense.cpp:220: penalty.find("net"))
bool penalty_is_group(int id);

// Eigen >= 3.3 LinSpaced (see SURVEY.md A.1) and the lambda grid of src/oem_dense.cpp:179-186
std::vector<double> linspace_eigen(int N, double lo, double hi);
std::vector<double> lambda_base(double lmax, int nl, double lmin_ratio);

// stopRule, src/utils.cpp:537-549 (used on the host for the IRLS outer loop)
bool stop_rule_host(const std::vector<double> &cur, const std::vector<double> &prev, double tol);

struct Setup {
    int P = 0;
    int Lmax = 0;                         // result stride
    std::vector<int> pen;                 // penalty ids
    std::vector<double> gamma;            // per penalty
    double alpha = 1.0, tau = 0.5;        // call-wide scalars
    std::vector<std::vector<double>> lam; // per penalty (filled by build_lambdas)
    std::vector<int> nlam_run;            // lambdas actually run (ols: 1)
    bool lambda_given = false;
    // groups (CSR over unique groups)
    std::vector<int> unique, ptr, idx, cover;
    std::vector<double> gw;
    bool any_group = false;

    // validate + parse; q = dimension of beta; scan = how many entries of `groups` take part
    // (src/oem_dense.h:421-456; oem_big.h:445 scans nvars only); zero_w0: logistic sets w = 0 for group 0
    void parse(const oemb200_spec *s, int q, int scan, bool zero_w0);
    // per-penalty lambda vectors (src/oem_dense.cpp:179-227; logistic .net fudge oem_logistic_dense.cpp:210-225)
    void build_lambdas(const oemb200_spec *s, double lmax, bool logistic_fudge);
};

// Device-side mirrors of a Setup + the buffers a path launch fills.
struct PathBuffers {
    DBuf<double> lambdas, pen_fact, gw, beta_out, d, beta_final;
    DBuf<int> unique, ptr, idx, cover, niter, lz;
    std::vector<int> lam_off;     // per penalty
    std::vector<double> h_beta;   // nchains x Lmax x q raw iterates
    std::vector<int> h_niter;     // nchains x Lmax
    std::vector<double> h_d;      // ngram
    std::vector<int> h_lz;
};

// Run chains = ngram x P (chain index = g * P + pp) on XX / XY.  pen_fact_q: host, length q.
// lam_scale: lambdas handed to the solver are lam / lam_scale (scaleY for oem_fit_dense, else 1).
void run_paths(Ctx &cx, const Setup &su, const oemb200_opts *o, int q, int ngram, const double *XX, const double *XY,
               const std::vector<double> &pen_fact_q, double lam_scale, double eig_factor, bool accelerate,
               const double *post_scale_dev, PathBuffers &pb);

// ---- shared by the entry drivers (entries.cu) ----
void check_common(const oemb200_spec *s, const oemb200_opts *o, const oemb200_result *r, const char *want_family,
                  bool allow_weights = false);
struct DevMatrix { const double *p = nullptr; int64_t ld = 0; DBuf<double> own; };
struct DevVector { const double *p = nullptr; DBuf<double> own; };
void to_device_matrix(Ctx &cx, const double *x, int64_t n, int p, int64_t ldx, DevMatrix &m);
void to_device_vector(Ctx &cx, const double *v, int64_t n, DevVector &d);
void fill_common_outputs(const Setup &su, oemb200_result *res);

// ---- entry_sparse.cu: a dgCMatrix design on the device (validated CSC slots + CSR copy) and the passes over it ----
struct SparseDesign;
SparseDesign *sparse_design_create(Ctx &cx, const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p);
void sparse_design_destroy(SparseDesign *sd);
int sparse_design_nnz(const SparseDesign *sd);
// stats3p[0*p + j] = sum_i x_ij, [1*p + j] = sum_i x_ij v_i, [2*p + j] = sum_i x_ij^2
void sparse_colstats_launch(Ctx &cx, const SparseDesign *sd, const double *v, double *stats3p);
// G (p x p) = X' diag(roww) X (roww may be NULL); sparse or densified-tile route by cost model
void sparse_gram_launch(Ctx &cx, const SparseDesign *sd, const double *roww, double *G);
// prob / resid = y - prob / w = prob (1 - prob) of eta = X b + *b0_dev (any output may be NULL)
void sparse_xb_logistic_launch(Ctx &cx, const SparseDesign *sd, const double *b, const double *b0_dev, const double *y,
                               double *prob, double *resid, double *w);

// ---- entry_xval.cu: steps 1-3 shared by the gaussian and the binomial xval drivers ----
struct XvalSystems {
    int F = 0, NG = 0;                       // folds, systems (0 = full data, k = without fold k)
    std::vector<int64_t> cnt, off;           // rows per fold; fold k = sorted rows [off[k], off[k] + cnt[k]), padded to off[k + 1]
    int64_t npad = 0;                        // rows of the fold-sorted copy
    DBuf<double> Xs, ys, ws;                 // fold-sorted X (column-major, ld npad), y, weights (zero padding rows)
    DBuf<double> XX, XY, cinv, nout;         // NG assembled systems (assemble_aug_launch)
    std::vector<double> hXY, hcinv, hn;      // host: XY of system 0, cinv of every system, row count of every system
};
// weights may be NULL.  hess_scale scales the Grams, column sums and corners before assembly (the binomial driver's
// upper-bound Hessian X'WX at beta = 0 has W = 1/4; a power of two, so the scaled sums are exact); 1 = no launch.
void xval_build_systems(Ctx &cx, const double *x, int64_t n, int p, int64_t ldx, const double *y, const double *weights,
                        int F, const int *foldid, int icpt, bool stdz, double hess_scale, XvalSystems &xs);

// ---- entry_logistic.cu ----
// tot[0] = get_loss() of prob (src/oem_logistic_dense.h:1057-1088) summed over n rows; partial: 1024 doubles of scratch
void logistic_loss_launch(Ctx &cx, const double *y, const double *prob, int64_t n, double *partial, double *tot2);

// row-slab copy of X kept across logistic fits (owned by an oemb200_matrix handle); `rt` = rows per slab it was built with
struct SlabCache { double *slabs = nullptr; int rt = 0; };
void finish_stats(Ctx &cx, PhaseTimers &tm, size_t total_id, oemb200_result *res);

}  // namespace oemb200
