// host_common.h -- host-side bookkeeping shared by the fit drivers: penalty / group / lambda setup (the part of the
// reference's entry functions that is not arithmetic on X) and its device mirror, the helper that runs a set of chains
// through the path kernel and brings the raw iterates back, the layout of the reported beta, and the parts of the three
// logistic (IRLS) drivers that are not their data passes: the init step and the outer loop with its per-model state.
#pragma once
#include <cmath>
#include <functional>
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
    std::vector<std::vector<double>> lam; // per penalty (filled by build_lambdas), Lmax entries each: parse requires
                                          // equal-length user sequences, the generated grid has nlambda = Lmax
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

// Device mirror of a Setup, uploaded once per fit: the lambdas (P x Lmax, penalty pp at pp * Lmax) divided by lam_scale
// (scaleY for oem_fit_dense, else 1), the penalty factor of length q = p + icpt (0 in the unpenalised intercept slot)
// and the group CSR.  h_lam / h_pf are the host sources of the asynchronous uploads and live as long as the tables.
struct PenaltyTables {
    int q = 0, Lmax = 0, ngroups = 0, ngidx = 0;
    std::vector<double> h_lam, h_pf;
    DBuf<double> lambdas, pen_fact, gw;
    DBuf<int> unique, ptr, idx, cover;
    PenaltyTables(Ctx &cx, const Setup &su, const oemb200_spec *s, int p, int icpt, double lam_scale = 1.0);
};

// The buffers a path launch fills.
struct PathBuffers {
    DBuf<double> beta_out, d;
    DBuf<int> niter, lz;
    std::vector<double> h_beta;   // nchains x Lmax x q raw iterates
    std::vector<int> h_niter;     // nchains x Lmax
    std::vector<double> h_d;      // ngram
    std::vector<int> h_lz;
};

// Run chains = ngram x P (chain index = g * P + pp) on XX / XY.
void run_paths(Ctx &cx, const Setup &su, const PenaltyTables &tb, const oemb200_opts *o, int ngram, const double *XX,
               const double *XY, double eig_factor, bool accelerate, const double *post_scale_dev, PathBuffers &pb);

// res->beta (P x Lmax x (p + 1): intercept row first, zero where no lambda ran) from the raw q-vectors of a fit, iterate
// (pp, i) at raw + (pp * Lmax + i) * q with q = p + icpt; cinv (host, p) undoes the standardisation, NULL if none.
void write_beta(const Setup &su, const double *raw, int p, int icpt, const double *cinv, oemb200_result *res);

// init_oem of the dense and sparse logistic drivers (src/oem_logistic_dense.h:721-793, oem_logistic_sparse.h:727-818):
// colstats(out) enqueues [sum x | X'y | sum x^2] (3p) of this rank's rows into out; the sums and n are all-reduced and
// brought to the host.  Refuses n <= q with `refusal`.  stats keeps the all-reduced sums on the device (then n at 3p).
struct LogisticInit {
    double n_tot = 0.0;
    std::vector<double> cinv;     // host, p: 1 / sd of every column (ones when not standardised)
    double lmax = 0.0;            // compute_lambda_zero: max_j |X'y o cinv| / n
    DBuf<double> stats;
};
LogisticInit logistic_init(Ctx &cx, int64_t n, int p, int q, bool stdz, const std::function<void(double *)> &colstats,
                           const char *refusal);

// The device slots of one model of an IRLS loop: its system XX / XY (q = tb.q) and eigenvalue bound d, the path launch's
// iteration count, Lanczos steps and tables, the convergence flag that predicates the model's work, the running count of
// inner iterations (may be shared by models), and the coefficients of the model's next data pass, b (p = q - icpt) and
// *b0, with the column scaling cinv (device, p; NULL when not standardised).  t_acc (may be NULL): see PathProblem.
struct IrlsModel {
    const double *XX = nullptr;
    double *XY = nullptr, *d = nullptr;
    int *niter = nullptr, *lz = nullptr;
    PathScratch *scratch = nullptr;
    int *conv = nullptr;
    long long *iters_total = nullptr;
    int icpt = 0;
    const double *cinv = nullptr;
    double *b = nullptr, *b0 = nullptr;
    unsigned long long *t_acc = nullptr;
};

// n mapped pinned ints: the IRLS verdict slots a path launch writes (PathProblem::irls_host_flag) and the host reads
struct PinnedFlags {
    int *p = nullptr;
    explicit PinnedFlags(int n) {
        OEM_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&p), sizeof(int) * (size_t)n, cudaHostAllocMapped));
        memset(p, 0, sizeof(int) * (size_t)n);
    }
    ~PinnedFlags() { if (p) cudaFreeHost(p); }
};
// n PathScratch tables, one per chain layout that is launched over and over
struct PathScratches {
    std::vector<PathScratch *> s;
    explicit PathScratches(int n) { for (int i = 0; i < n; ++i) s.push_back(path_scratch_create()); }
    ~PathScratches() { for (auto *x : s) path_scratch_destroy(x); }
};

// The outer IRLS loop (src/oem_logistic_dense.h:1000-1035) of M logistic models in lockstep, and their device state.  Per
// penalty every model starts from beta = 0, so the first data pass multiplies X with b = 0, b0 = 0.  Per lambda, round k
// enqueues iteration k of every model still iterating: the driver's data pass, then one path launch per model
// (path_step), which writes the model's stop-rule verdict to the device flag that predicates the model's later kernels of
// the lambda and to a mapped host slot.  The host's one round trip per round is a wait for the round (an event wait
// with speculation, else a stream sync) and a read of those verdicts.  With `speculate` (M = 1 only) round k + 1 is
// enqueued before round k's verdict is read, so the GPU never waits for the host (the gap was ~100 us per iteration: 5 %
// of a dense fit on one GPU, 25 % row-sharded over eight); a round enqueued after convergence is a few empty launches,
// and its counters are rolled back.  Only a driver whose every kernel of the chain can be predicated may speculate.
class IrlsLoop {
public:
    IrlsLoop(Ctx &cx, const Setup &su, const PenaltyTables &tb, const oemb200_opts *o, int M, int icpt, bool speculate);
    IrlsLoop(const IrlsLoop &) = delete;
    ~IrlsLoop();
    // the device slots of model m that the driver owns (see IrlsModel)
    void set_model(int m, const double *XX, double *XY, double *d, const double *cinv, unsigned long long *t_acc = nullptr);

    DBuf<double> b, b0;          // M x p, M: the coefficients of each model's next data pass
    DBuf<int> conv;              // M: the model has converged in this lambda (the predicate of its kernels)
    DBuf<double> path;           // M x P x Lmax x q raw iterates, model m's penalty pp at chain m * P + pp
    std::vector<char> active;    // host, M: the models still iterating in this lambda

    // Every lambda of every penalty: round(i, k, pass) enqueues round k of lambda i (pass = false on a warm lambda's first
    // iteration, where the reference skips the data pass), ending with path_step for every active model.  When every
    // model has stopped, lambda_end(pp, i) runs, then the final iterates go into `path` and model 0's niter into res.
    void run(oemb200_result *res, const std::function<void(int, int, bool)> &round,
             const std::function<void(int, int)> &lambda_end);
    // model m's path launch of this round.  compute_eig: the Hessian was rebuilt; with grad (device, [sum r, X'r] over
    // n_rows rows) the launch first forms XY = XX beta + grad / n_rows (scaled by cinv), without it keeps the last XY
    void path_step(int m, bool compute_eig, const double *grad, double n_rows);
    double *final_iterate(int m);       // in lambda_end: the iterate of the model's last executed iteration
    // after the loop: model 0's path, d and the count of inner iterations into res (cinv: host, p; NULL if none)
    void write_path(const double *cinv, oemb200_result *res);

private:
    Ctx &cx_;
    const Setup &su_;
    const PenaltyTables &tb_;
    const oemb200_opts *o_;
    const int M_, q_;
    const bool speculate_;
    DBuf<double> iter_;                  // M x 2 x q: the model's iterate ping-pongs between its two slots
    DBuf<int> niter_, lz_;
    DBuf<long long> iters_total_;
    PathScratches scratch_;
    std::vector<IrlsModel> md_;
    PinnedFlags flag_;                   // 4 x M verdict slots: round g writes row g & 3
    cudaEvent_t ev_[2];                  // with speculation, recorded after round g: ev_[g & 1]
    long long gi_ = 0;                   // rounds enqueued so far
    int pp_ = 0, i_ = 0, k_ = 0;         // the round being enqueued
    std::vector<int> par0_, last_, niter_h_;   // per model: slot of iteration 0, last executed iteration, reported niter
    bool wait_round(long long g, int k);
};

// Copy stream of a streamed pass over host row chunks, with ping-pong events: ready[b] = staging buffer b holds its chunk,
// freed[b] = the compute stream is done reading it.  Released on every exit path (a throwing launch included).
struct CopyLane {
    cudaStream_t s = nullptr;
    cudaEvent_t ready[2] = {nullptr, nullptr}, freed[2] = {nullptr, nullptr};
    CopyLane() {
        OEM_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            OEM_CUDA(cudaEventCreateWithFlags(&ready[b], cudaEventDisableTiming));
            OEM_CUDA(cudaEventCreateWithFlags(&freed[b], cudaEventDisableTiming));
        }
    }
    CopyLane(const CopyLane &) = delete;
    ~CopyLane() {
        if (s) cudaStreamSynchronize(s);
        for (int b = 0; b < 2; ++b) { if (ready[b]) cudaEventDestroy(ready[b]); if (freed[b]) cudaEventDestroy(freed[b]); }
        if (s) cudaStreamDestroy(s);
    }
};

// ---- shared by the entry drivers (entries.cu) ----
void check_common(const oemb200_spec *s, const oemb200_opts *o, const oemb200_result *r, const char *want_family,
                  bool allow_weights = false);
struct DevMatrix { const double *p = nullptr; int64_t ld = 0; DBuf<double> own; };
struct DevVector { const double *p = nullptr; DBuf<double> own; };
void to_device_matrix(Ctx &cx, const double *x, int64_t n, int p, int64_t ldx, DevMatrix &m);
void to_device_vector(Ctx &cx, const double *v, int64_t n, DevVector &d);
void fill_common_outputs(const Setup &su, oemb200_result *res);
// rows per chunk of a pass that streams X: opts->gigs GB (1 when unset), a multiple of the fold-segment alignment
// 2 * gram_kt(), at most n rounded up to it
int64_t big_chunk_rows(const oemb200_opts *o, int64_t n, int p);

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
// stable counting sort of the rows by fold on the host (more folds than fold_bucket_max_folds()): cnt / off as in
// XvalSystems, dest / order (n ints each) for fold_gather_launch; refuses ids outside 1..F
void xval_bucket_host(const int *foldid, int64_t n, int F, int64_t align, std::vector<int64_t> &cnt, std::vector<int64_t> &off,
                      int *dest, int *order);

// ---- entry_logistic.cu ----
// get_loss() of prob (src/oem_logistic_dense.h:1057-1088) summed over the n rows and over ranks
double logistic_loss(Ctx &cx, const double *y, const double *prob, int64_t n);

// row-slab copy of X kept across logistic fits (owned by an oemb200_matrix handle); `rt` = rows per slab it was built with
struct SlabCache { double *slabs = nullptr; int rt = 0; };
void finish_stats(Ctx &cx, PhaseTimers &tm, size_t total_id, oemb200_result *res);

}  // namespace oemb200
