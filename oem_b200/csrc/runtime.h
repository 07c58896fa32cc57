// runtime.h -- host-side runtime shared by the entry-point drivers: device context, RAII device
// buffers, phase timers, and the declarations of the kernel launchers (one .cu file each).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstring>
#include <string>
#include <array>
#include <vector>
#include "../../include/oem_b200.h"
#include "common.cuh"

namespace oemb200 {

// CUDA-event phase timer: adds elapsed ms to *acc when stopped (after a stream sync at the end
// of the call: see PhaseTimers::collect()).
// Timing events come from a per-thread, per-device free list (event_acquire / event_release in runtime.cu): the IRLS loop
// of the logistic entries opens ~1000 timed phases per fit, and a cudaEventCreate / cudaEventDestroy pair per phase boundary
// was a measurable part of the host-bound gap between its small kernels.
cudaEvent_t event_acquire();
void event_release(cudaEvent_t e);

struct PhaseTimers {
    struct Rec { cudaEvent_t a, b; double *acc; };
    std::vector<Rec> recs;
    cudaStream_t s;
    explicit PhaseTimers(cudaStream_t s_) : s(s_) {}
    PhaseTimers(const PhaseTimers &) = delete;
    ~PhaseTimers() { for (auto &r : recs) { event_release(r.a); event_release(r.b); } }
    size_t start(double *acc) {
        Rec r; r.acc = acc;
        r.a = event_acquire(); r.b = event_acquire();
        OEM_CUDA(cudaEventRecord(r.a, s));
        recs.push_back(r);
        return recs.size() - 1;
    }
    void stop(size_t i) { OEM_CUDA(cudaEventRecord(recs[i].b, s)); }
    void collect() {   // call after the stream is synchronized
        for (auto &r : recs) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess && r.acc) *r.acc += ms;
        }
    }
};

struct Ctx {
    int device = 0;
    int prev_device = -1;
    int num_sms = 148;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    oemb200_stats st;              // accumulated by the launchers
    oemb200_allreduce_fn allreduce = nullptr;
    void *allreduce_ctx = nullptr;
    oemb200_comm *comm = nullptr;  // in-library communicator (comm.cu); wins over the callback
    int rank = 0, world = 1;
    PhaseTimers *tm = nullptr;     // created with the context, collected by finish()

    explicit Ctx(const oemb200_opts *o);
    ~Ctx();
    void sync() { st.host_syncs += 1; OEM_CUDA(cudaStreamSynchronize(stream)); }
    bool distributed() const { return comm != nullptr || allreduce != nullptr; }
    // in-place sum over ranks, ordered on `stream`; no-op in single-process runs
    void all_reduce(double *dev_buf, int64_t count, const int *skip = nullptr, unsigned long long *t_acc = nullptr);
    bool all_reduce_can_skip(int64_t count) const;   // true in single-process runs and on the peer-memory transport
    void finish();                 // sync the stream, fold the event timings into st
};

// Thread-local caching device allocator: entry calls repeat the same shapes, so after the first call
// no cudaMalloc / cudaFree (and none of their implicit device syncs) happen in steady state.  Blocks are
// handed back while kernels using them may still be queued; that is safe because every block is only
// ever reused by the same host thread on the call's single compute stream (stream order), and each
// entry point synchronizes its stream before returning.
void *pool_alloc(size_t bytes);
void pool_free(void *p);
void pool_release_all();      // cudaFree everything cached by this thread

// RAII device buffer (pooled)
template <typename T>
struct DBuf {
    T *p = nullptr;
    size_t n = 0;
    DBuf() {}
    explicit DBuf(size_t n_) { alloc(n_); }
    DBuf(const DBuf &) = delete;
    DBuf &operator=(const DBuf &) = delete;
    DBuf(DBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DBuf &operator=(DBuf &&o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
        return *this;
    }
    ~DBuf() { release(); }
    void alloc(size_t n_) {
        release();
        n = n_;
        if (n) p = static_cast<T *>(pool_alloc(n * sizeof(T)));
    }
    void release() {
        if (p) pool_free(p);
        p = nullptr;
        n = 0;
    }
    void zero(cudaStream_t s) { if (n) OEM_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
    void upload(const T *h, size_t cnt, cudaStream_t s) {
        OEM_CUDA(cudaMemcpyAsync(p, h, cnt * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void download(T *h, size_t cnt, cudaStream_t s) const {
        OEM_CUDA(cudaMemcpyAsync(h, p, cnt * sizeof(T), cudaMemcpyDeviceToHost, s));
    }
};

bool is_device_ptr(const void *p);

// Rank-local validation in front of a collective: runs f(); in row-sharded runs the ranks then agree (one 1-value
// all-reduce) on whether anybody failed, so that a rank with bad inputs cannot leave its peers waiting in the next
// data all-reduce.  The failing rank rethrows its own error, the others report OEMB200_ECOMM.
template <typename F>
void collective_guard(Ctx &cx, F &&f) {
    int code = 0;
    std::string msg;
    try {
        f();
    } catch (const Error &e) {
        code = e.code;
        msg = e.what();
    }
    if (cx.distributed()) {
        DBuf<double> flag(1);
        double h = code ? 1.0 : 0.0;
        flag.upload(&h, 1, cx.stream);
        cx.sync();
        cx.all_reduce(flag.p, 1);
        flag.download(&h, 1, cx.stream);
        cx.sync();
        if (h > 0.0 && !code) fail(OEMB200_ECOMM, "another rank rejected its inputs; this rank stops before the next collective");
    }
    if (code) throw Error(code, msg);
}

// ---------------- ingest.cu ----------------
bool is_pinned_host(const void *p);
// rows [0, nr) x p columns of a column-major HOST block -> device, ordered on `stream`: in place for pinned sources,
// through the pinned bounce ring + reader threads for pageable / memory-mapped ones.  Adds to cx.st.h2d_bytes.
void h2d_block(Ctx &cx, const double *src, int64_t ldx, int64_t nr, int p, double *dst, int64_t ld_dst, cudaStream_t stream);
void release_host_stager();

// ---------------- comm.cu ----------------
// skip (optional device flag, identical on every rank): the collective is a no-op when *skip != 0; only the peer-memory
// transport can honour it (comm_can_skip), NCCL collectives cannot be predicated from the device
void comm_all_reduce(oemb200_comm *c, double *dev_buf, int64_t count, cudaStream_t stream, const int *skip = nullptr,
                     unsigned long long *t_acc = nullptr);      // t_acc: device ns accumulator of the peer-memory kernel
bool comm_can_skip(const oemb200_comm *c, int64_t count);

// ---------------- gram_syrk.cu ----------------
struct RowSegment { int64_t row0, row1; int out; };   // rows [row0,row1) accumulate into Gram #out
// G[out] (q x q col-major, full symmetric; nout matrices, stride q*q) (+)= X_seg' diag(w) X_seg with
// optional column centring.  Segment boundaries must be multiples of 36 rows except at n.
// stats_out (optional, not with row weights or centring): nout x 3 x q = [sum x, sum x*stats_y, sum x^2] per output, in the
// layout of colstats_launch, accumulated by the diagonal-tile CTAs of the same launch (stats_y may be NULL: sum x*y = 0)
void gram_launch(Ctx &cx, const double *X, int64_t n, int q, int64_t ld, const std::vector<RowSegment> &segs,
                 int nout, const double *mean, const double *roww, double *G, bool accumulate,
                 const double *stats_y = nullptr, double *stats_out = nullptr);
int gram_kt();   // rows per pipeline stage (segment alignment)

// ---------------- colstats.cu ----------------
// with xs = x - shift_j (shift may be NULL):
// out[0*p + j] = sum_i xs_ij v0_i, out[1*p + j] = sum_i xs_ij v1_i, out[2*p + j] = sum_i xs_ij^2 (NULL v = ones)
void colstats_launch(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, const double *v0, const double *v1,
                     const double *shift, double *out3p, bool accumulate);
// out2[0] (+)= sum (v - shift), out2[1] (+)= sum (v - shift)^2
void vecsum_launch(Ctx &cx, const double *v, int64_t n, double shift, double *out2, bool accumulate);
// out = (v - shift) / divisor
void affine_launch(Ctx &cx, const double *v, int64_t n, double shift, double divisor, double *out);
// y += a * x
void axpy_launch(Ctx &cx, int64_t n, double a, const double *x, double *y);
// eta = X b + b0 (+ logistic epilogue: prob, resid = y - prob, w = prob (1 - prob))
// b0_dev (optional): a device scalar added to b0 (the IRLS loop keeps its intercept on the device)
void xb_launch(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, const double *b, double b0, const double *y,
               double *eta, double *prob, double *resid, double *w, bool logistic, const double *b0_dev = nullptr);

// ---------------- path_kernel.cu ----------------
struct ChainDesc {          // one warm-started lambda path: (Gram, penalty)
    int gram;               // index of the Gram / XY this chain runs on
    int penalty;            // OEMB200_PEN_*
    int nlam;               // number of lambdas
    int lam_off;            // offset into the lambda array
    double alpha, gamma, tau;
    int out_off;            // chain slot in beta_out / niter_out (units of chains)
};
// device tables of a generic path launch (chain descriptors, team maps, exchange buffers, barrier words); a caller
// that launches the same chain layout many times (the logistic IRLS loop) keeps one and skips the re-uploads
struct PathScratch;
PathScratch *path_scratch_create();
void path_scratch_destroy(PathScratch *s);

struct PathProblem {
    int q = 0;              // dimension of beta
    int ngram = 0;          // number of Grams (teams)
    const double *XX = nullptr;    // device, ngram x q x q (already scaled, / n)
    const double *XY = nullptr;    // device, ngram x q
    double *d = nullptr;           // device, ngram: in (compute_eig=0) or out (compute_eig=1)
    bool compute_eig = true;
    double eig_factor = 1.005;
    double eig_tol = 1e-10;
    std::vector<ChainDesc> chains;
    const double *lambdas = nullptr;   // device, concatenated
    int Lmax = 0;                      // stride (in lambdas) of a chain's output block
    const double *pen_fact = nullptr;  // device, q
    // group structure (device), CSR over unique groups
    int ngroups = 0;
    int ngidx = 0;          // length of grp_idx
    const int *unique_groups = nullptr, *grp_ptr = nullptr, *grp_idx = nullptr;
    const double *group_weights = nullptr;
    const int *grp_cover = nullptr;       // device, q: 1 if the variable belongs to a listed group
    const double *post_scale = nullptr;   // oem_xtx scale.factor quirk: beta *= post_scale after each lambda
    const double *beta_init = nullptr;    // device, nchains x q warm start (NULL = zeros)
    int maxit = 500;
    double tol = 1e-7;
    bool accelerate = false;
    double *beta_out = nullptr;    // device, nchains x Lmax x q  (raw iterates)
    int *niter_out = nullptr;      // device, nchains x Lmax
    int *lanczos_steps = nullptr;  // device, ngram (may be NULL)
    PathScratch *scratch = nullptr;   // optional, see above
    const int *skip = nullptr;        // optional device flag: the launch does nothing when it is non-zero
    // Outer (IRLS) loop of the logistic entries folded into the launch's last step (one Gram, one chain, one lambda): the
    // stop rule stopRule(beta_new, beta_init, irls_tol) (src/utils.cpp:537-549, called at src/oem_logistic_dense.h:1028),
    // its verdict for the device (*irls_conv = 1: every later launch predicated on it returns at once) and for the host
    // (*irls_host_flag, mapped pinned memory), the running count of inner iterations, and the coefficients the NEXT data
    // pass multiplies X with: b = beta_new[icpt:] o cinv, b0 = beta_new[0] (src/oem_logistic_dense.h:875-890).
    int *irls_conv = nullptr;
    volatile int *irls_host_flag = nullptr;
    long long *irls_iters_total = nullptr;
    double irls_tol = 0.0;
    const double *irls_cinv = nullptr;
    int irls_p = 0, irls_icpt = 0;
    double *irls_b = nullptr, *irls_b0 = nullptr;
    unsigned long long *t_acc = nullptr;   // optional device word: += the kernel's duration in ns (%globaltimer of team 0's first member)
    // Logistic inner loop (src/oem_logistic_dense.h:970-999): with xy_grad set the launch first forms
    //   XY = XX beta_init + [g[0] / n, (g[1 + j] / n) o cinv[j]]
    // into xy_out (which must be the buffer XY points at; one Gram, one chain).  The register-resident global mode does it
    // with the XX slice its members have just loaded; the other modes launch path_xy_kernel in front.
    const double *xy_grad = nullptr, *xy_cinv = nullptr;
    double xy_n = 0.0;
    int xy_icpt = 0;
    double *xy_out = nullptr;
};
void path_launch(Ctx &cx, const PathProblem &pp);
// throws OEMB200_EUNSUPPORTED if a beta of dimension q (chains_per_gram penalties, Lmax lambdas) cannot be held by the path kernel
void path_check_fits(Ctx &cx, int q, int chains_per_gram, int Lmax, int ngroups, int ngidx);

// ---------------- assemble.cu ----------------
// oem_big / logistic / xval convention: explicit intercept border, uncentred scaling (SURVEY A.4-A.6).
// Output o sums all parts except part o-1 (o = 0: all).  XY / colsq_inv / nobs_out may be NULL.
void assemble_aug_launch(Ctx &cx, int p, int intercept, int standardize, int nparts, int nout,
                         const double *G_parts /*nparts x p x p*/, const double *stats_parts /*nparts x 3 x p*/,
                         const double *ysum_parts /*nparts, stride ysum_stride*/, int ysum_stride,
                         const double *corner_parts /*nparts*/,
                         const double *nobs_parts /*nparts*/, double *XX /*nout x q x q*/, double *XY /*nout x q*/,
                         double *colsq_inv /*nout x p*/, double *nobs_out /*nout*/);
// oem_dense convention (SURVEY A.2): G is the Gram of centred (flag 2,3) or raw (flag 0,1) columns
void assemble_dense_launch(Ctx &cx, int p, int flag, double n, const double *G, const double *xy, const double *css,
                           double *XX, double *XY, double *scalex);
// oem_xtx scale.factor (sinv may be NULL = plain copy)
void scale_sym_launch(Ctx &cx, int p, const double *sinv, const double *XXin, const double *XYin, double *XX,
                      double *XY);

// ---------------- logit_slab.cu ----------------
int logit_slab_rows(int p);                       // rows per slab (0: the slab route does not apply to this p; it does for 8 <= p <= 2048)
bool logit_slab_preferred(int64_t n, int p);      // the default route: slab for p >= 128, and for smaller p when n <= 1e5 (launch-bound)
size_t logit_slab_doubles(int64_t n, int p);      // size of the re-laid-out copy
void logit_slab_relayout(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, double *slabs);
// one pass over the slabs: prob, w (may be NULL), grad_out[0] = sum (y - prob), grad_out[1 + j] = sum_i x_ij (y_i - prob_i)
// skip (optional device flag): the pass does nothing and leaves every output untouched when *skip != 0
void logit_slab_launch(Ctx &cx, const double *slabs, int64_t n, int p, const double *b, const double *b0_dev,
                       const double *y, double *prob, double *w, double *grad_out, const int *skip = nullptr,
                       unsigned long long *t_clock = nullptr);   // t_clock (device, 2 words): [0] += ns of the pass, [1] scratch
// Fused pass of M logistic models over one 4-row slab copy (logit_fold_relayout): model g uses the rows whose fold[i] is
// neither 0 nor g; grad (M x (p + 1)): row g = [sum r, X' r] of model g.  B: M x p, b0: M (device).  conv (device, M ints,
// may be NULL) / active (host, may be NULL): converged models are skipped and their grad rows left untouched; a group of
// models with no active member costs no launch.  prob0 (may be NULL): sigma(eta) of model 0 on its rows.  Returns the
// number of sweeps over X (ceil(M / logit_fold_models(p)) when every group is active).
int logit_fold_models(int p);                     // models per sweep (0: 8 <= p <= 2048 does not hold)
size_t logit_fold_doubles(int64_t n, int p);
void logit_fold_relayout(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, double *slabs);
int logit_fold_launch(Ctx &cx, const double *slabs, int64_t n, int p, const double *B, const double *b0, const double *y,
                      const int *fold, int M, const int *conv, const std::vector<char> *active, double *prob0, double *grad);

// ---------------- cvscore.cu ----------------
// order[i]: for every tile of fold_gather_tile_rows() source rows, the tile-local row indices grouped by fold
void fold_gather_launch(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, const int *dest, const int *order,
                        double *Xs, int64_t lds, const double *y, double *ys, const double *w = nullptr,
                        double *ws = nullptr, double *yws = nullptr);
int fold_gather_tile_rows();
// stable counting sort of the rows by fold on the device (nfolds <= 64): dest, order (device), cnt / off (host)
bool fold_bucket_device(Ctx &cx, const int *foldid_dev, int64_t n, int F, int64_t align, int *dest, int *order,
                        std::vector<int64_t> &cnt, std::vector<int64_t> &off);
// its two halves, with no host round trip in between: per-tile prefixes tcount (ceil(n / fold_gather_tile_rows()) x F),
// fold totals (device, F) and *err (set on an id outside 1..F); then dest / order from tcount and each fold's first
// sorted row base (device, F)
void fold_count_launch(Ctx &cx, const int *foldid_dev, int64_t n, int F, int *tcount, int *err, long long *total);
void fold_rank_launch(Ctx &cx, const int *foldid_dev, int64_t n, int F, const int *tcount, const long long *base, int *dest,
                      int *order);
int fold_bucket_max_folds();     // largest nfolds of the device bucketing
int cv_ncld(int nc);     // leading dimension (columns) of the coefficient matrices handed to cvscore_launch
// out3 = 3 x nc: (count, mean, M2) of t = (y - pred)^2 | |y - pred| over all valid rows, per column
// ws: optional observation weights (fold-sorted like ys): t is multiplied by w_i.  accumulate: merge these rows' moments
// into the (count, mean, M2) already in out3 (after them, in a fixed order), for rows scored one chunk at a time
void cvscore_launch(Ctx &cx, const double *Xs, int64_t nrows_total, int p, int64_t lds, const double *ys,
                    const double *ws, int nfolds, const std::vector<std::array<int64_t, 3>> &segs, const double *B,
                    const double *b0, int nc, bool mae, double *out3, bool accumulate = false);
// the same moments of cv.oem's binomial measures (R/cv_oem.R:288-330) on p = 1 / (1 + exp(-(x . b + b0))), unweighted:
// measure 0 = deviance (p clamped to [1e-5, 1 - 1e-5]), 1 = class error (p > 0.5) != y, 2 = 2 (y - p)^2, 3 = 2 |y - p|
void cvscore_binomial_launch(Ctx &cx, const double *Xs, int64_t nrows_total, int p, int64_t lds, const double *ys, int nfolds,
                             const std::vector<std::array<int64_t, 3>> &segs, const double *B, const double *b0, int nc,
                             int measure, double *out3);
// B / b0 operands of cvscore_launch built on the device from the path kernel's raw iterates (chains (k+1) * P + pp)
void cv_build_coef_launch(Ctx &cx, const double *beta_raw, const double *cinv, int nfolds, int P, int L, int p, int q, int icpt,
                          bool standardize, const int *nlam_run_dev, double *B, double *b0);
// pred (n x nc col-major, ld ldo) = X B + b0 (B, b0 in cvscore layout with one "fold"); response: 1/(1+exp(-link))
void predict_launch(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, const double *B, const double *b0, int nc,
                    bool response, double *pred, int64_t ldo);

}  // namespace oemb200
