/*
 * oem_b200.h -- C ABI of the B200-native OEM hot path (liboem_b200.so).
 *
 * Drop-in boundary for the five C++ entry points of jaredhuling/oem 2.0.12 that the R
 * front-ends reach through .Call (paths relative to the reference tree):
 *
 *   oemb200_fit_dense            replaces  oem_fit_dense            src/oem_dense.cpp:30-48
 *   oemb200_xtx                  replaces  oem_xtx                  src/oem_xtx.cpp:29-44
 *   oemb200_xval_dense           replaces  oem_xval_dense           src/oem_xval_dense.cpp:31-52
 *   oemb200_xval_big             oem_xval_dense on an x streamed in row chunks (no reference counterpart)
 *   oemb200_fit_logistic_dense   replaces  oem_fit_logistic_dense   src/oem_logistic_dense.cpp:29-47
 *   oemb200_fit_big              replaces  oem_fit_big / oem_fit_fb_big   src/oem_big.cpp:30-48
 *   oemb200_fit_sparse           replaces  oem_fit_sparse           src/oem_sparse.cpp:30
 *   oemb200_fit_logistic_sparse  replaces  oem_fit_logistic_sparse  src/oem_logistic_sparse.cpp:30
 *
 * Argument ORDER and meaning follow the reference's .Call lists (R/oem.R:556-575,
 * R/oem_xtx.R:389-420, R/oem_xval.R:525-548, R/big_oem.R:449-490); SEXPs become plain
 * pointers + sizes.  Matrices are column-major FP64 exactly like R.  Return layout follows
 * the reference's named list (beta / lambda / niter / loss / d [/ cvm / cvsd]) as flat,
 * caller-allocated buffers (oemb200_result).  No torch / Rcpp / Eigen types cross this ABI.
 *
 * Every function returns 0 on success or an OEMB200_E* code; oemb200_last_error() gives
 * the message (thread-local).  Nothing throws across the ABI.  There is NO CPU fallback:
 * without a CUDA device every compute entry returns OEMB200_ENODEVICE.
 *
 * x / y / xtx / xty may be HOST or DEVICE pointers (detected with
 * cudaPointerGetAttributes).  Host inputs are copied to the device inside the call
 * (oem_fit_big streams row chunks and never needs all of X resident).
 */
#ifndef OEM_B200_H
#define OEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OEMB200_OK          0
#define OEMB200_EINVAL      1   /* bad argument (message says which) */
#define OEMB200_ENODEVICE   2   /* no CUDA device / driver */
#define OEMB200_ECUDA       3   /* a CUDA call or kernel failed */
#define OEMB200_EUNSUPPORTED 4  /* a shape or flag combination the reference itself leaves undefined or incoherent (the message cites where) */
#define OEMB200_ECOMM       5   /* the all-reduce callback failed */

/* Penalty ids, in the order the oracle uses (oracle/oem_oracle.c). Names are the R strings. */
enum {
    OEMB200_PEN_LASSO = 0, OEMB200_PEN_OLS = 1, OEMB200_PEN_ENET = 2, OEMB200_PEN_SCAD = 3,
    OEMB200_PEN_SCAD_NET = 4, OEMB200_PEN_MCP = 5, OEMB200_PEN_MCP_NET = 6,
    OEMB200_PEN_GRP_LASSO = 7, OEMB200_PEN_GRP_LASSO_NET = 8, OEMB200_PEN_GRP_MCP = 9,
    OEMB200_PEN_GRP_SCAD = 10, OEMB200_PEN_GRP_MCP_NET = 11, OEMB200_PEN_GRP_SCAD_NET = 12,
    OEMB200_PEN_SPARSE_GRP_LASSO = 13
};

/*
 * Sum-all-reduce of `count` doubles living in DEVICE memory at `buf`, in place, ordered on
 * CUDA stream `stream` (a cudaStream_t).  Supplied by the host program (NCCL through
 * torch.distributed in the Python host, ncclAllReduce in an R/C++ host).  Must return 0 on
 * success.  NULL = single process.
 */
typedef int (*oemb200_allreduce_fn)(void *buf, int64_t count, void *stream, void *ctx);

/* `options` list of the reference (R/oem.R:438-444, R/big_oem.R:352-357) + runtime knobs. */
typedef struct oemb200_opts {
    int    maxit;          /* opts$maxit        (default 500)  */
    double tol;            /* opts$tol          (default 1e-7) */
    int    irls_maxit;     /* opts$irls_maxit   (default 100)  */
    double irls_tol;       /* opts$irls_tol     (default 1e-3) */
    int    ncores;         /* accepted and ignored: the GPU path has no OpenMP team */
    int    hessian_full;   /* opts$hessian.type: 0 = "upper.bound", 1 = "full" */
    int    accelerate;     /* opts$accelerate (Nesterov), oem_fit_dense only */
    double gigs;           /* big.oem `gigs`: here = host->device streaming chunk size in GB (<=0: 1 GB) */
    /* ---- runtime (not in the reference) ---- */
    int    device;         /* CUDA device ordinal; -1 = current device */
    void  *stream;         /* cudaStream_t to run on; NULL = the legacy default stream */
    oemb200_allreduce_fn allreduce;  /* row-sharded multi-process runs; NULL = single process */
    void  *allreduce_ctx;
    int    rank, world;    /* informational (world<=1: single process) */
    struct oemb200_comm *comm;       /* in-library communicator (oemb200_comm_create); takes precedence over `allreduce` */
} oemb200_opts;

/* Arguments shared by all entries, in the reference's .Call order (family .. compute_loss). */
typedef struct oemb200_spec {
    const char          *family;            /* "gaussian" | "binomial" */
    int                  n_penalty;
    const char  *const  *penalty;           /* R penalty names */
    const double        *weights;  int64_t n_weights;        /* observation weights: xval only (R/oem_xval.R:215); else empty (R/oem.R:244) */
    const int           *groups;   int n_groups;             /* length p, or 0 */
    const int           *unique_groups; int n_unique_groups;
    const double        *group_weights; int n_group_weights; /* 0 => sqrt(|g|) */
    const double *const *lambda;            /* per penalty; may be NULL */
    const int           *n_lambda;          /* per penalty lengths; NULL/0 => generate */
    int                  nlambda;
    double               lambda_min_ratio;
    double               alpha;
    const double        *gamma;    int n_gamma;  /* 1 value (reference) or one per penalty (extension) */
    double               tau;
    const double        *penalty_factor;    /* length p */
    int                  standardize;
    int                  intercept;
    int                  compute_loss;
} oemb200_spec;

/* Phase timings (ms, CUDA events on the library stream) and counters; optional. */
typedef struct oemb200_stats {
    double ms_h2d, ms_colstats, ms_gram, ms_gram_reduce, ms_allreduce, ms_assemble,
           ms_path, ms_cvscore, ms_irls_xb, ms_irls_xtr, ms_total;
    double gram_flops;        /* algorithmic: rows * q * (q+1) summed over launches */
    double gemv_bytes;        /* algorithmic bytes of the logistic GEMV launches */
    int64_t kernel_launches;  /* our kernels launched inside the call */
    int64_t gram_launches, xb_launches, xtr_launches;
    int64_t total_oem_iters;  /* sum of niter over all chains */
    int64_t lanczos_steps;
    int64_t h2d_bytes, d2h_bytes;
    /* appended in 0.2 */
    int64_t allreduce_calls;    /* sum all-reduces issued inside the call (0 in single-process runs) */
    int64_t allreduce_doubles;  /* FP64 values they carried */
    int64_t data_passes;        /* logistic: IRLS data passes over X (fused sigma(X beta) / X'r sweeps) */
    int64_t host_syncs;         /* stream synchronisations the host driver performed inside the call */
    double  ms_relayout;        /* logistic: one-time row-slab re-layout of X */
    double  ms_ingest_wait;     /* host time spent filling the pinned bounce ring from pageable / mmap'd sources */
} oemb200_stats;

/*
 * Result buffers (caller-allocated).  With P = n_penalty, L = oemb200_nlambda_max(spec):
 *   beta   P blocks of (p+1) x L column-major, row 0 = intercept   (oem_xtx: p x L, no intercept row)
 *   lambda P x L      niter P x L (true per-penalty counts; the reference aliases one vector,
 *   loss   P x L      src/oem_dense.cpp:200,292)      nlam_out[P] = columns actually filled (ols: 1)
 *   d      1          cvm / cvsd  P x L (xval only)
 */
typedef struct oemb200_result {
    double *beta; double *lambda; int *niter; double *loss; double *d;
    double *cvm;  double *cvsd;   int *nlam_out;
    oemb200_stats *stats;          /* may be NULL */
} oemb200_result;

/*
 * In-library communicator for row-sharded runs (one process per GPU).  The sum all-reduces of the path -- the packed
 * sufficient statistics once per fit, the (p+1)-vector X'(y - prob) once per IRLS iteration of the logistic entry
 * (src/oem_logistic_dense.h:970-1000 is the single-process sum it replaces) -- are then issued by the library itself on
 * its own CUDA stream: ncclAllReduce from the libnccl.so.2 already loaded in the process (else the system one; the
 * library is dlopen()ed, never linked), or, for vectors up to OEMB200_P2P_MAX_DOUBLES on one NVLink / NVSwitch node, a
 * one-shot peer-memory kernel (every rank stores its vector into every peer's mailbox over NVLink and sums the
 * mailboxes in rank order, so all ranks hold bit-identical results).  No host callback, no host synchronisation.
 *
 *   rank 0:     oemb200_comm_unique_id(id)           -> broadcast the 128 bytes by any host channel
 *   every rank: oemb200_comm_create(id, rank, world, device, &comm);   opts.comm = comm;   ...fits...
 *               oemb200_comm_destroy(comm)
 * An R / C++ host that already owns an ncclComm_t wraps it with oemb200_comm_from_nccl (not owned, not destroyed).
 *
 * Rules: creation and destruction are collective (every rank, same order).  A communicator serves ONE stream of calls at a
 * time -- collectives are matched across ranks by their order on that stream, and the peer-memory transport keeps its epoch
 * counter in device memory in stream order -- so do not issue fits that share a communicator from two host threads at once.
 * If a peer dies, the peer-memory kernel traps after 30 s instead of spinning forever (the CUDA context is then lost, like
 * after any device-side fault).
 */
#define OEMB200_COMM_ID_BYTES 128
#define OEMB200_P2P_MAX_DOUBLES 8192
typedef struct oemb200_comm oemb200_comm;
int  oemb200_comm_unique_id(void *id_out);
int  oemb200_comm_create(const void *id, int rank, int world, int device, oemb200_comm **out);
int  oemb200_comm_from_nccl(void *nccl_comm, int rank, int world, int device, oemb200_comm **out);
int  oemb200_comm_destroy(oemb200_comm *c);
/* in-place sum all-reduce of `count` device doubles on `stream` (what the entries call internally); *us_out (optional)
 * = device time of the collective in microseconds (forces a stream synchronisation: measurement only) */
int  oemb200_comm_allreduce(oemb200_comm *c, double *dev_buf, int64_t count, void *stream, double *us_out);
/* 1 if the one-shot NVLink peer-memory path is active for this communicator (all ranks on one node with P2P access) */
int  oemb200_comm_p2p_enabled(const oemb200_comm *c);

const char *oemb200_last_error(void);
const char *oemb200_version(void);
int  oemb200_device_count(void);
void oemb200_default_opts(oemb200_opts *o);
int  oemb200_penalty_id(const char *name);          /* -1 if unknown */
int  oemb200_nlambda_max(const oemb200_spec *s);    /* L used to size the result buffers */
/* Host-only helpers (no device needed): the lambda grid exp(LinSpaced(nl, log lmax, log(ratio*lmax)))
 * of src/oem_dense.cpp:179-186, and stopRule of src/utils.cpp:537-549. */
int  oemb200_lambda_grid(double lmax, int nlambda, double lambda_min_ratio, double *out);
int  oemb200_stop_rule(const double *cur, const double *prev, int q, double tol);
void oemb200_release_cache(void);                   /* free the calling thread's cached device buffers */

/* src/oem_dense.cpp:30 -- x: n x p column-major (ldx >= n), y: n. */
int oemb200_fit_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y,
                      const oemb200_spec *spec, const oemb200_opts *opts, oemb200_result *res);

/* src/oem_xtx.cpp:29 -- xtx: p x p (already / n), xty: p, scale_factor: p or NULL. */
int oemb200_xtx(const double *xtx, const double *xty, int p,
                const oemb200_spec *spec, const double *scale_factor, int n_scale_factor,
                const oemb200_opts *opts, oemb200_result *res);

/* src/oem_xval_dense.cpp:31 -- foldid: n ints in 1..nfolds; type_measure "mse" | "mae". */
int oemb200_xval_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y,
                       const oemb200_spec *spec, int nfolds, const int *foldid,
                       const char *type_measure, const oemb200_opts *opts, oemb200_result *res);

/* oemb200_xval_dense on an x that is never resident on the device: same arguments, same meaning, same result layout
 * (weights, the standardize x intercept flags, "mse" | "mae" | "deviance" (= mse), compute_loss, foldid on the host or
 * the device, more than 64 folds with a host foldid).  x (and y, weights, foldid) may be pageable or pinned host memory
 * or device memory (e.g. the data of an oemb200_matrix whose fold-sorted copy would not fit beside it); x is read in row
 * chunks of opts->gigs GB, twice: one pass forms the fold Grams, one scores the fold models after the path.  Device
 * memory does not grow with n: two staging chunks (host x only), one fold-sorted chunk, the fold Grams, the nfolds + 1
 * systems, the path and the coefficient matrices.  stats: data_passes = 2, gram_launches = the number of chunks,
 * h2d_bytes = every host-to-device copy (a host x, y and weights once per pass, a host foldid three times: once to count
 * the rows of every (chunk, fold), once per pass), host_syncs independent of the number of chunks.  Results agree with
 * oemb200_xval_dense up to summation order (bit for bit when x is one chunk).  OEMB200_EUNSUPPORTED, before any device
 * work, for the binomial family (each IRLS round would be another pass over the host link) and row-sharded calls
 * (world > 1, comm or allreduce). */
int oemb200_xval_big(const double *x, int64_t n, int p, int64_t ldx, const double *y,
                     const oemb200_spec *spec, int nfolds, const int *foldid,
                     const char *type_measure, const oemb200_opts *opts, oemb200_result *res);

/* Binomial cross-validation (the reference's xval.oem stops on the binomial family, R/oem_xval.R:160-163): the full-data
 * model is oemb200_fit_logistic_dense on all rows, fold model k the same fit on the rows with foldid != k at the full
 * model's lambda sequence; every IRLS data pass serves all nfolds + 1 models in one sweep of x.  Result as for
 * oemb200_xval_dense (beta / lambda / niter / loss / d of the full model).  cvm / cvsd: mean over all n rows of the
 * held-out measure of cv.oem (R/cv_oem.R:288-330) and sqrt(M2 / (n - 1)) / sqrt(n); type_measure "deviance" (default,
 * NULL) | "class" | "mse" | "mae" ("auc" needs per-fold ranks: OEMB200_EINVAL).  OEMB200_EUNSUPPORTED for
 * opts->hessian_full, observation weights, row-sharded calls and p outside 8..2048. */
int oemb200_xval_logistic_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y,
                                const oemb200_spec *spec, int nfolds, const int *foldid,
                                const char *type_measure, const oemb200_opts *opts, oemb200_result *res);

/* src/oem_logistic_dense.cpp:29 -- y in {0,1}. */
int oemb200_fit_logistic_dense(const double *x, int64_t n, int p, int64_t ldx, const double *y,
                               const oemb200_spec *spec, const oemb200_opts *opts,
                               oemb200_result *res);

/* src/oem_big.cpp:30 (and oem_fb_big.cpp) -- x is the big.matrix payload: n x p column-major
 * doubles (the mmap'd region the reference wraps at oem_big.cpp:64). */
int oemb200_fit_big(const double *x, int64_t n, int p, int64_t ldx, const double *y,
                    const oemb200_spec *spec, const oemb200_opts *opts, oemb200_result *res);

/* src/oem_sparse.cpp:30 -- x is a Matrix::dgCMatrix (what R/oem.R:236-240 coerces every sparseMatrix to), passed as its
 * three slots: row_idx = x@i (nnz 0-based row indices), col_ptr = x@p (p + 1 column pointers, col_ptr[p] = nnz),
 * values = x@x; host or device pointers.  Gaussian family; n > p, and n <= p without an intercept (src/oem_sparse.h:609-616,
 * 630-640: the raw-X iteration; with an intercept the reference runs past the end of XY and beta there: OEMB200_EUNSUPPORTED).
 * Same result layout as oemb200_fit_dense (beta (p+1) x L per penalty, row 0 = intercept). */
int oemb200_fit_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p,
                       const double *y, const oemb200_spec *spec, const oemb200_opts *opts,
                       oemb200_result *res);

/* src/oem_logistic_sparse.cpp:30 -- binomial family on a dgCMatrix (slots as in oemb200_fit_sparse), y in {0,1}, n > p, the
 * reference's ncores <= 1 code path.  standardize = TRUE with or without intercept, and standardize = FALSE without
 * intercept, follow the reference; intercept = TRUE with standardize = FALSE returns OEMB200_EUNSUPPORTED (the reference
 * multiplies by a vector it never initialised there, src/oem_logistic_sparse.h:880 vs :737-751). */
int oemb200_fit_logistic_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p,
                                const double *y, const oemb200_spec *spec, const oemb200_opts *opts,
                                oemb200_result *res);

/* predict.oem (R/methods.R:48-119; logistic response R/methods.R:346-366): out (n x nlambda, column-major,
 * ldo >= n, host or device) = newx (n x p) * beta[intercept rows dropped] + beta[0, :].  beta is the host
 * coefficient matrix of one model as the fit entries return it: beta_rows x nlambda column-major with
 * beta_rows = p + 1 (row 0 = intercept) or p (oem_xtx).  type 0 = "link", 1 = "response" of the binomial
 * family, 1 / (1 + exp(-link)).  One FP64 DMMA GEMM launch (the CV-scoring kernel with a store epilogue). */
int oemb200_predict(const double *x, int64_t n, int p, int64_t ldx, const double *beta, int beta_rows,
                    int nlambda, int type, double *out, int64_t ldo, const oemb200_opts *opts,
                    oemb200_stats *stats);

/* predict.oem on a sparse newx (dgCMatrix slots as in oemb200_fit_sparse; `as.matrix(newx %*% nbeta)`, R/methods.R:113-118).
 * Same beta / type / out conventions as oemb200_predict. */
int oemb200_predict_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p,
                           const double *beta, int beta_rows, int nlambda, int type, double *out, int64_t ldo,
                           const oemb200_opts *opts, oemb200_stats *stats);

/* ------------------------------------------------------------------------------------------
 * Device-resident design matrix (SURVEY.md 8b "Ownership").  The reference copies / maps x inside every .Call
 * (src/oem_dense.cpp:61-67; src/oem_big.cpp:52-64 wraps the big.matrix external pointer without copying); an R host
 * cannot hold a device pointer, so without a handle every fit would re-upload x.  oemb200_matrix_create uploads an
 * n x p column-major FP64 matrix ONCE (pageable sources through the pinned bounce ring) -- or streams the raw
 * column-major doubles of a bigmemory backing file (.bk) -- and the *_h entries run the same drivers on it with no
 * host -> device traffic for x.  The handle also keeps the row-slab copy the logistic entry builds on first use, so
 * repeated binomial fits skip the re-layout too.  An Rcpp shim wraps the handle in an XPtr with
 * oemb200_matrix_destroy as its finalizer (INTEGRATION.md), exactly like the reference passes `x@address`.
 * A handle is immutable after creation except for that lazily built slab copy: fits on one handle may run one after the
 * other from any thread, but not concurrently.
 * ------------------------------------------------------------------------------------------ */
typedef struct oemb200_matrix oemb200_matrix;
int oemb200_matrix_create(const double *x, int64_t n, int p, int64_t ldx, const oemb200_opts *opts,
                          oemb200_matrix **out);
int oemb200_matrix_create_from_file(const char *bk_path, int64_t n, int p, const oemb200_opts *opts,
                                    oemb200_matrix **out);
int oemb200_matrix_destroy(oemb200_matrix *m);
/* any output pointer may be NULL; h2d_bytes = bytes uploaded when the handle was created */
int oemb200_matrix_info(const oemb200_matrix *m, int64_t *n, int *p, int64_t *ld, const double **dev_ptr,
                        int64_t *h2d_bytes, double *ms_upload);
int oemb200_fit_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec,
                        const oemb200_opts *opts, oemb200_result *res);
int oemb200_fit_big_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec,
                      const oemb200_opts *opts, oemb200_result *res);
int oemb200_fit_logistic_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec,
                                 const oemb200_opts *opts, oemb200_result *res);
int oemb200_xval_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec, int nfolds,
                         const int *foldid, const char *type_measure, const oemb200_opts *opts,
                         oemb200_result *res);
int oemb200_predict_h(const oemb200_matrix *x, const double *beta, int beta_rows, int nlambda, int type,
                      double *out, int64_t ldo, const oemb200_opts *opts, oemb200_stats *stats);
int oemb200_xval_logistic_dense_h(const oemb200_matrix *x, const double *y, const oemb200_spec *spec, int nfolds,
                                  const int *foldid, const char *type_measure, const oemb200_opts *opts,
                                  oemb200_result *res);

/* ------------------------------------------------------------------------------------------
 * Phase-level entries (device pointers only) used by bench.py for the roofline numbers and by
 * the Gram-level parity tests.  They are the kernels the five entries above are made of.
 * ------------------------------------------------------------------------------------------ */

/* G (q x q col-major, full symmetric) = sum_i w_i (x_i - mean)(x_i - mean)'  over rows of x.
 * mean / row_w may be NULL.  src/oem_dense.h:318-361 (XtX), oem_logistic_dense.h:334-381 (XtWX). */
int oemb200_gram(const double *x_dev, int64_t n, int p, int64_t ldx,
                 const double *mean_dev, const double *row_w_dev, double *g_dev,
                 void *stream, double *ms_out);

/* out[j] = sum_i x_ij v_i for up to two vectors (NULL = ones) and sum_i x_ij^2:
 * out_dev is 3 x p (row 0: v0, row 1: v1, row 2: squares).  src/oem_big.h:743-837. */
int oemb200_colstats(const double *x_dev, int64_t n, int p, int64_t ldx,
                     const double *v0_dev, const double *v1_dev, double *out_dev,
                     void *stream, double *ms_out);

/* eta = x b + b0; prob = 1/(1+exp(-eta)); resid = y - prob; w = prob(1-prob).
 * src/oem_logistic_dense.h:864-949. Any of prob/resid/w may be NULL. */
int oemb200_xb_logistic(const double *x_dev, int64_t n, int p, int64_t ldx, const double *b_dev,
                        double b0, const double *y_dev, double *prob_dev, double *resid_dev,
                        double *w_dev, void *stream, double *ms_out);

/* One fused IRLS data pass of the logistic entry on a row-slab copy of x (csrc/logit_slab.cu): X is read from HBM
 * once, grad_dev[0] = sum_i (y_i - prob_i), grad_dev[1 + j] = sum_i x_ij (y_i - prob_i); prob_dev / w_dev as in
 * oemb200_xb_logistic (either may be NULL).  The slab copy is built inside the call (time reported separately in
 * *ms_relayout_out); the pass is run `reps` times and *ms_out is the CUDA-event average of one pass.  Returns
 * OEMB200_EUNSUPPORTED for p outside the slab kernel's range (8..2048).
 * src/oem_logistic_dense.h:864-949 + 970-992 in one sweep. */
int oemb200_logit_slab_pass(const double *x_dev, int64_t n, int p, int64_t ldx, const double *b_dev, double b0,
                            const double *y_dev, double *prob_dev, double *w_dev, double *grad_dev, int reps,
                            void *stream, double *ms_out, double *ms_relayout_out);

/* The fused data pass of oemb200_xval_logistic_dense for M models: model g uses the rows i with fold_dev[i] not 0 and
 * not g (model 0: every row with a non-zero fold), grad_dev row g (M x (p + 1), row-major) = [sum r, X' r] over its rows
 * with r_i = y_i - 1/(1 + exp(-(b0_dev[g] + x_i . b_dev[g]))); b_dev is M x p row-major, b0_dev M values.  conv_dev (M
 * ints, may be NULL): models with a non-zero flag are skipped and their grad rows left untouched.  A 4-row slab copy of
 * x is built inside the call (*ms_relayout_out); the pass (ceil(M / models-per-sweep) sweeps) runs `reps` times and
 * *ms_out is the average of one pass; *sweeps_out (may be NULL) = sweeps per pass.  OEMB200_EUNSUPPORTED for p
 * outside 8..2048. */
int oemb200_logit_fold_pass(const double *x_dev, int64_t n, int p, int64_t ldx, const double *b_dev,
                            const double *b0_dev, const double *y_dev, const int *fold_dev, int M, const int *conv_dev,
                            double *grad_dev, int reps, void *stream, double *ms_out, double *ms_relayout_out,
                            int *sweeps_out);

/* Largest eigenvalue of the symmetric q x q matrix (device, col-major) by on-device Lanczos.
 * Stands in for Spectra::SymEigsSolver at src/oem_dense.h:485-498. */
int oemb200_top_eig(const double *xx_dev, int q, double *lambda_max_out, int *steps_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* OEM_B200_H */
