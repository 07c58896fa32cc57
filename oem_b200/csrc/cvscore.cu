// cvscore.cu -- the second data pass of xval.oem: out-of-fold prediction errors for every
// (penalty, lambda) column with running mean / M2, without materialising the n x (P*L) predictions.
//
// Replaces the CV-scoring loop of oem_xval_dense (src/oem_xval_dense.cpp:345-464):
//     for each row i:  pred = x_i . B_fold(i)[1:, :] + B_fold(i)[0, :];  t = (y_i - pred)^2  or |y_i - pred|
//     Welford over i:  cvm = mean(t),  cvsd = sqrt(M2 / (n-1)) / sqrt(n)
// As a GEMM:  T(rows x NC) = X_k (rows x p) * B_k (p x NC)  per fold segment k (rows are fold-sorted by
// fold_gather_kernel), on the FP64 tensor pipe (DMMA.8x8x4) with both operands staged by TMA:
//   X box  [68 rows x 20 cols]  (64 used; the 4 extra rows make the k-stride 68 = 4 mod 16: conflict-free)
//   B box  2 x [164 cols x 20 rows] (160 used each, stride 164 = 4 mod 16)
// CTA tile = 64 rows x 320 columns, 8 warps as 2 x 4 with 32 x 80 warp tiles (80 accumulator doubles per
// thread); with at most 160 columns (one penalty's lambda path) 128 rows x 160 columns, 8 warps as 4 x 2.  A CTA walks a contiguous range of row tiles of one fold and keeps (count, mean, M2) per column
// with Chan's pairwise update, so one partial per CTA reaches the fixed-order final merge.
#include <algorithm>
#include <array>
#include "runtime.h"

namespace oemb200 {

constexpr int CV_KC = 20;
constexpr int CV_KSTEPS = CV_KC / 4;
constexpr int CV_COLS = 320;
constexpr int CV_BHALF = 160;
constexpr int CV_BBOX = 164;
constexpr int CV_STAGES = 3;
constexpr int CV_THREADS = 256;
constexpr int CV_B_BYTES = CV_KC * CV_BBOX * 8;                 // 26240
// dynamic shared memory of the NH-half variant: stages + barriers + [2][rows/32][cols] reduction + running mean / M2 + y, w tiles
constexpr int cv_smem_bytes(int nh) {
    return CV_STAGES * (CV_KC * ((nh == 2 ? 64 : 128) + 4) * 8 + nh * CV_B_BYTES) + 128 +
           (2 * ((nh == 2 ? 64 : 128) / 32) * (CV_BHALF * nh) + 2 * (CV_BHALF * nh) + 2 * (nh == 2 ? 64 : 128) + 8) * 8;
}

struct CvItem {
    int fold, colblock, pad0, pad1;
    long long row0;       // first row of the item in the fold-sorted matrix (multiple of 64 from the segment start)
    long long row_end;    // end of the item's rows (exclusive)
    long long valid_end;  // rows >= valid_end are padding
};

// Rows into fold-sorted order: Xs[dest[i], j] = X[i, j].  A CTA stages a tile of 1024 source rows x 4 columns in
// shared memory with coalesced loads, then writes it out in the tile's fold-grouped order (`order`, built on the host
// by a per-tile counting sort): rows of one fold are consecutive in the destination, so the stores are coalesced runs
// of ~1024/nfolds doubles instead of isolated 8-byte writes.
constexpr int FG_ROWS = 1024;
constexpr int FG_COLS = 4;

__global__ void __launch_bounds__(256)
fold_gather_kernel(const double *__restrict__ X, long long n, int p, long long ld, const int *__restrict__ dest,
                   const int *__restrict__ order, double *__restrict__ Xs, long long lds, const double *__restrict__ y,
                   double *__restrict__ ys, const double *__restrict__ w, double *__restrict__ ws,
                   double *__restrict__ yws) {
    __shared__ double tile[FG_COLS][FG_ROWS];
    const long long r0 = (long long)blockIdx.x * FG_ROWS;
    const int j0 = blockIdx.y * FG_COLS;
    const int nr = (int)min((long long)FG_ROWS, n - r0);
    const int nc = min(FG_COLS, p - j0);
    for (int c = 0; c < nc; ++c)
        for (int r = threadIdx.x; r < nr; r += 256) tile[c][r] = X[(size_t)(j0 + c) * ld + r0 + r];
    __syncthreads();
    for (int t = threadIdx.x; t < nr; t += 256) {
        const int rl = order[r0 + t];                 // tile-local source row, fold-grouped
        const long long d = dest[r0 + rl];
        for (int c = 0; c < nc; ++c) Xs[(size_t)(j0 + c) * lds + d] = tile[c][rl];
        if (blockIdx.y == 0 && y) {
            const double yv = y[r0 + rl];
            ys[d] = yv;
            if (w) {                                  // observation weights: w and y*w in fold-sorted order
                const double wv = w[r0 + rl];
                ws[d] = wv;
                yws[d] = yv * wv;
            }
        }
    }
}

void fold_gather_launch(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, const int *dest, const int *order,
                        double *Xs, int64_t lds, const double *y, double *ys, const double *w, double *ws,
                        double *yws) {
    dim3 grid((unsigned)((n + FG_ROWS - 1) / FG_ROWS), (p + FG_COLS - 1) / FG_COLS);
    fold_gather_kernel<<<grid, 256, 0, cx.stream>>>(X, n, p, ld, dest, order, Xs, lds, y, ys, w, ws, yws);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

int fold_gather_tile_rows() { return FG_ROWS; }

// ---- fold bucketing on the device (stable counting sort of the rows by fold, nfolds <= 64) ----
constexpr int FB_MAXF = 64;

// per-tile histogram of foldid (1-based); bad ids raise *err
__global__ void __launch_bounds__(256)
fold_count_kernel(const int *__restrict__ foldid, long long n, int F, int *__restrict__ tcount, int *__restrict__ err) {
    __shared__ int hist[FB_MAXF];
    if (threadIdx.x < FB_MAXF) hist[threadIdx.x] = 0;
    __syncthreads();
    const long long r0 = (long long)blockIdx.x * FG_ROWS;
    for (int r = threadIdx.x; r < FG_ROWS && r0 + r < n; r += 256) {
        const int f = foldid[r0 + r];
        if (f < 1 || f > F) atomicExch(err, 1);
        else atomicAdd(&hist[f - 1], 1);            // integer counts: order-independent, deterministic
    }
    __syncthreads();
    if (threadIdx.x < F) tcount[(size_t)blockIdx.x * F + threadIdx.x] = hist[threadIdx.x];
}

// exclusive scan over tiles, one thread per fold; total[f] = rows of fold f
__global__ void fold_scan_kernel(int *__restrict__ tcount, int ntiles, int F, long long *__restrict__ total) {
    const int f = threadIdx.x;
    if (f >= F) return;
    long long run = 0;
    for (int t = 0; t < ntiles; ++t) {
        const int c = tcount[(size_t)t * F + f];
        tcount[(size_t)t * F + f] = (int)run;
        run += c;
    }
    total[f] = run;
}

// dest[i] = foldbase[f] + (rows of fold f before i); order = tile-local rows grouped by fold (stable)
__global__ void __launch_bounds__(256)
fold_rank_kernel(const int *__restrict__ foldid, long long n, int F, const int *__restrict__ tprefix,
                 const long long *__restrict__ foldbase, int *__restrict__ dest, int *__restrict__ order) {
    __shared__ int seg[32][FB_MAXF];      // rows of fold f in 32-row segment s, then exclusive prefix over s
    __shared__ int fstart[FB_MAXF];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long r0 = (long long)blockIdx.x * FG_ROWS;
    int myf[4], lrank[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r = k * 256 + threadIdx.x;
        const int f = (r0 + r < n) ? foldid[r0 + r] - 1 : -1;
        myf[k] = f;
        lrank[k] = 0;
        for (int ff = 0; ff < F; ++ff) {
            const unsigned m = __ballot_sync(0xffffffffu, f == ff);
            if (f == ff) lrank[k] = __popc(m & ((1u << lane) - 1u));
            if (lane == 0) seg[k * 8 + warp][ff] = __popc(m);
        }
    }
    __syncthreads();
    if (threadIdx.x < F) {
        int run = 0;
        for (int sgi = 0; sgi < 32; ++sgi) { const int c = seg[sgi][threadIdx.x]; seg[sgi][threadIdx.x] = run; run += c; }
        fstart[threadIdx.x] = run;        // tile count of this fold
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int ff = 0; ff < F; ++ff) { const int c = fstart[ff]; fstart[ff] = run; run += c; }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r = k * 256 + threadIdx.x, f = myf[k];
        if (f < 0) continue;
        const int within = seg[k * 8 + warp][f] + lrank[k];
        dest[r0 + r] = (int)(foldbase[f] + tprefix[(size_t)blockIdx.x * F + f] + within);
        order[r0 + fstart[f] + within] = r;
    }
}

// Per-fold row counts of foldid[0, n): fold_count_kernel's per-tile histogram, turned by fold_scan_kernel into each tile's
// exclusive prefix (tcount, what fold_rank_launch reads) and the fold totals (device, F).  Bad ids set *err.
void fold_count_launch(Ctx &cx, const int *foldid_dev, int64_t n, int F, int *tcount, int *err, long long *total) {
    const int ntiles = (int)((n + FG_ROWS - 1) / FG_ROWS);
    fold_count_kernel<<<ntiles, 256, 0, cx.stream>>>(foldid_dev, n, F, tcount, err);
    fold_scan_kernel<<<1, FB_MAXF, 0, cx.stream>>>(tcount, ntiles, F, total);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 2;
}

// dest / order of foldid[0, n) from fold_count_launch's tile prefixes and the first sorted row of every fold (base, device)
void fold_rank_launch(Ctx &cx, const int *foldid_dev, int64_t n, int F, const int *tcount, const long long *base, int *dest,
                      int *order) {
    const int ntiles = (int)((n + FG_ROWS - 1) / FG_ROWS);
    fold_rank_kernel<<<ntiles, 256, 0, cx.stream>>>(foldid_dev, n, F, tcount, base, dest, order);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

int fold_bucket_max_folds() { return FB_MAXF; }

// Device-side bucketing: fills dest / order (device) and counts (host).  Returns false if nfolds is too large for
// this path (the caller then buckets on the host).
bool fold_bucket_device(Ctx &cx, const int *foldid_dev, int64_t n, int F, int64_t align, int *dest, int *order,
                        std::vector<int64_t> &cnt, std::vector<int64_t> &off) {
    if (F > FB_MAXF) return false;
    const int ntiles = (int)((n + FG_ROWS - 1) / FG_ROWS);
    DBuf<int> tcount((size_t)ntiles * F), err(1);
    DBuf<long long> total(F), base(F);
    err.zero(cx.stream);
    fold_count_launch(cx, foldid_dev, n, F, tcount.p, err.p, total.p);
    std::vector<long long> ht(F);
    int herr = 0;
    total.download(ht.data(), F, cx.stream);
    err.download(&herr, 1, cx.stream);
    cx.sync();
    if (herr) fail(OEMB200_EINVAL, "foldid has entries outside 1..%d", F);
    cnt.assign(F, 0);
    off.assign(F + 1, 0);
    std::vector<long long> hb(F);
    for (int k = 0; k < F; ++k) {
        cnt[k] = ht[k];
        off[k + 1] = off[k] + (cnt[k] + align - 1) / align * align;
        hb[k] = off[k];
    }
    base.upload(hb.data(), F, cx.stream);
    fold_rank_launch(cx, foldid_dev, n, F, tcount.p, base.p, dest, order);
    cx.sync();      // tcount / base go back to the pool
    return true;
}

// Coefficient operand of the CV-scoring GEMM straight from the path kernel's output (no host round trip):
//   B[k][j][c] = beta_raw[chain (k+1, pp)][lambda i][icpt + j] * (standardize ? colsq_inv[k+1][j] : 1),  c = pp * L + i
//   b0[k][c]   = intercept entry; columns beyond a penalty's lambda count (ols) and the padding up to ncld are zero
// (get_beta() un-scaling of the fold fits, src/oem_xval_dense.h:1102-1120).
__global__ void cv_build_coef_kernel(const double *__restrict__ beta_raw, const double *__restrict__ cinv, int P, int L, int p,
                                     int q, int icpt, int standardize, const int *__restrict__ nlam_run, int ncld,
                                     double *__restrict__ B, double *__restrict__ b0) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;             // 0..p-1: coefficient row, p: intercept row
    const int k = blockIdx.z;             // fold
    if (c >= ncld) return;
    const int pp = c / L, i = c - pp * L;
    const bool live = pp < P && i < nlam_run[pp];
    const double *raw = beta_raw + (((size_t)(k + 1) * P + (live ? pp : 0)) * L + (live ? i : 0)) * q;
    if (j == p) {
        b0[(size_t)k * ncld + c] = (live && icpt) ? raw[0] : 0.0;
    } else {
        double v = live ? raw[icpt + j] : 0.0;
        if (standardize) v *= cinv[(size_t)(k + 1) * p + j];
        B[((size_t)k * p + j) * ncld + c] = v;
    }
}

void cv_build_coef_launch(Ctx &cx, const double *beta_raw, const double *cinv, int nfolds, int P, int L, int p, int q, int icpt,
                          bool standardize, const int *nlam_run_dev, double *B, double *b0) {
    const int ncld = cv_ncld(P * L);
    dim3 grid((ncld + 127) / 128, p + 1, nfolds);
    cv_build_coef_kernel<<<grid, 128, 0, cx.stream>>>(beta_raw, cinv, P, L, p, q, icpt, standardize ? 1 : 0, nlam_run_dev, ncld, B, b0);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

// EPI: 0 = squared error moments, 1 = absolute error moments (the CV score), 2..5 = the binomial measures of cv.oem
// (R/cv_oem.R:288-330) on p = 1 / (1 + exp(-link)): deviance -2 [y log p~ + (1 - y) log(1 - p~)] with p~ = p clamped to
// [1e-5, 1 - 1e-5], class error (p > 0.5) != y, 2 (y - p)^2, 2 |y - p|;  6 = store the linear predictor x_i . b + b0
// (predict.oem type = "link", R/methods.R:113-118), 7 = store 1 / (1 + exp(-link)) (type = "response" of
// predict.oemfit_binomial, R/methods.R:355-358).  The store modes write pred[c * ldo + row] for c < nc.
constexpr int EPI_MSE = 0, EPI_MAE = 1, EPI_BDEV = 2, EPI_BCLASS = 3, EPI_BMSE = 4, EPI_BMAE = 5, EPI_LINK = 6, EPI_RESPONSE = 7;

template <int EPI>
__device__ __forceinline__ double cv_measure(double yv, double link) {
    if (EPI == EPI_MSE) { const double r = yv - link; return r * r; }
    if (EPI == EPI_MAE) return fabs(yv - link);
    const double pr = 1.0 / (1.0 + exp(-link));
    if (EPI == EPI_BDEV) {
        const double pm = fmin(fmax(pr, 1e-5), 1.0 - 1e-5);
        return -2.0 * ((1.0 - yv) * log(1.0 - pm) + yv * log(pm));
    }
    if (EPI == EPI_BCLASS) return (pr > 0.5) != (yv == 1.0) ? 1.0 : 0.0;
    if (EPI == EPI_BMSE) return 2.0 * (yv - pr) * (yv - pr);
    return 2.0 * fabs(yv - pr);
}

// one k-tile (CV_KC rows of the contraction) of a warp's 32 x (8 NAT) tile: NAT column atoms, compile-time
template <int NAT>
__device__ __forceinline__ void cv_ktile(double (&acc)[4][10][2], const double *__restrict__ xs, const double *__restrict__ bs,
                                         int xbox, int offA, int offB, int t) {
#pragma unroll
    for (int ks = 0; ks < CV_KSTEPS; ++ks) {
        double a[4], b[NAT];
        const int k = ks * 4 + t;
#pragma unroll
        for (int ma = 0; ma < 4; ++ma) a[ma] = xs[k * xbox + offA + ma * 8];
#pragma unroll
        for (int na = 0; na < NAT; ++na) b[na] = bs[k * CV_BBOX + offB + na * 8];
#pragma unroll
        for (int ma = 0; ma < 4; ++ma)
#pragma unroll
            for (int na = 0; na < NAT; ++na) dmma884(acc[ma][na][0], acc[ma][na][1], a[ma], b[na]);
    }
}

template <int EPI, int NH>
__global__ void __launch_bounds__(CV_THREADS, 1)
cvscore_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmB, int p, int ncld,
               const CvItem *__restrict__ items, const double *__restrict__ ys, const double *__restrict__ ws,
               const double *__restrict__ b0, double *__restrict__ partial, int part_stride,
               double *__restrict__ pred, long long ldo, int nc) {
    // NH = 2: CTA tile 64 rows x 320 columns (8 warps as 2 x 4);  NH = 1: 128 rows x 160 columns (4 x 2) for
    // nc <= 160 (one penalty's lambda path), which halves the padded columns.  Warp tile 32 x 80 in both.
    constexpr int ROWS = NH == 2 ? 64 : 128, XBOX = ROWS + 4, COLS = CV_BHALF * NH, NWM = ROWS / 32;
    constexpr int X_BYTES = CV_KC * XBOX * 8, STAGE_BYTES = X_BYTES + NH * CV_B_BYTES;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + CV_STAGES * STAGE_BYTES);
    uint64_t *empty = full + CV_STAGES;
    double *red = reinterpret_cast<double *>(smem_raw + CV_STAGES * STAGE_BYTES + 128);   // [2][NWM][COLS]
    double *run_mean = red + 2 * NWM * COLS;     // [COLS]
    double *run_m2 = run_mean + COLS;          // [COLS]
    double *ytile = run_m2 + COLS;             // [ROWS]
    double *wtile = ytile + ROWS;              // [ROWS] observation weights (1 when none)

    const CvItem it = items[blockIdx.x];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    // Warp columns.  Warps w and w + 4 share an SM sub-partition (and its FP64 tensor pipe); rotating the column index of the
    // upper warp rows pairs a wide warp column with a narrow one on every sub-partition (see `nat` below).
    const int wm = NH == 2 ? warp >> 2 : warp >> 1;
    const int wn = NH == 2 ? ((warp & 3) + 2 * wm) & 3 : ((warp & 1) ^ (wm >> 1));
    const int nkt = (p + CV_KC - 1) / CV_KC;
    const int ntiles = (int)((it.row_end - it.row0 + ROWS - 1) / ROWS);
    const long long total = (long long)ntiles * nkt;
    const int col0 = it.colblock * COLS;

    if (threadIdx.x == 0) {
        for (int s = 0; s < CV_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CV_THREADS / 32); }
        mbar_fence_init();
        tma_prefetch_desc(&tmX);
        tma_prefetch_desc(&tmB);
    }
    for (int c = threadIdx.x; c < COLS; c += CV_THREADS) { run_mean[c] = 0.0; run_m2[c] = 0.0; }
    __syncthreads();

    auto issue = [&](long long idx) {      // thread 0 only
        const int s = (int)(idx % CV_STAGES);
        const int tile = (int)(idx / nkt), kt = (int)(idx - (long long)tile * nkt);
        unsigned char *base = smem_raw + (size_t)s * STAGE_BYTES;
        mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
        tma_load_2d(base, &tmX, &full[s], (int)(it.row0 + (long long)tile * ROWS), kt * CV_KC);
        tma_load_2d(base + X_BYTES, &tmB, &full[s], col0, it.fold * p + kt * CV_KC);
        if (NH == 2) tma_load_2d(base + X_BYTES + CV_B_BYTES, &tmB, &full[s], col0 + CV_BHALF, it.fold * p + kt * CV_KC);
    };
    if (threadIdx.x == 0)
        for (long long i = 0; i < CV_STAGES && i < total; ++i) issue(i);

    // Column atoms (8 columns each) this warp owns.  A column block holds `a` live atoms (<= 20 per 160-column box); each box
    // splits its atoms over its two warp columns (first gets the odd one), so the 300 columns of three penalties x 100 lambdas
    // cost 10 / 10 / 9 / 9 atoms = 19 per sub-partition instead of the 20 of a padded 320-column tile, and a narrow last block
    // costs what it holds.  Atoms beyond `nat` are skipped in the main loop and in every epilogue.
    const int a_live = max(0, min(COLS / 8, (nc - col0 + 7) / 8));
    const int box = wn >> 1;
    const int a_box = max(0, min(20, a_live - 20 * box));
    const int nat = (wn & 1) ? a_box / 2 : (a_box + 1) / 2;
    const int colw = (wn & 1) ? ((a_box + 1) / 2) * 8 : 0;          // first column of this warp inside its box
    const int offA = wm * 32 + g;                         // + ma*8 + (k)*XBOX
    const int offB = colw + g;                            // + na*8 + (k)*CV_BBOX, box = wn >> 1
    double run_cnt = 0.0;
    for (int c = threadIdx.x; c < 2 * NWM * COLS; c += CV_THREADS) red[c] = 0.0;     // columns no warp owns stay finite
    __syncthreads();

    long long idx = 0;
    for (int tile = 0; tile < ntiles; ++tile) {
        double acc[4][10][2];
#pragma unroll
        for (int ma = 0; ma < 4; ++ma)
#pragma unroll
            for (int na = 0; na < 10; ++na) acc[ma][na][0] = acc[ma][na][1] = 0.0;
        const long long trow0 = it.row0 + (long long)tile * ROWS;
        if (EPI < EPI_LINK && threadIdx.x < ROWS) {
            const long long r = trow0 + threadIdx.x;
            ytile[threadIdx.x] = r < it.valid_end ? ys[r] : 0.0;
            wtile[threadIdx.x] = (ws && r < it.valid_end) ? ws[r] : 1.0;
        }
        for (int kt = 0; kt < nkt; ++kt, ++idx) {
            const int s = (int)(idx % CV_STAGES);
            const uint32_t ph = (uint32_t)((idx / CV_STAGES) & 1);
            mbar_wait(&full[s], ph);
            const double *xs = reinterpret_cast<const double *>(smem_raw + (size_t)s * STAGE_BYTES);
            const double *bs = xs + CV_KC * XBOX + (wn >> 1) * (CV_KC * CV_BBOX);
            // the atom count is warp-uniform: dispatch ONCE per k-tile to a straight-line loop with a compile-time count (a
            // per-atom runtime test inside the unrolled loop cost more issue slots than the trimmed atoms saved)
            switch (nat) {
                case 10: cv_ktile<10>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 9:  cv_ktile<9>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 8:  cv_ktile<8>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 7:  cv_ktile<7>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 6:  cv_ktile<6>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 5:  cv_ktile<5>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 4:  cv_ktile<4>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 3:  cv_ktile<3>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 2:  cv_ktile<2>(acc, xs, bs, XBOX, offA, offB, t); break;
                case 1:  cv_ktile<1>(acc, xs, bs, XBOX, offA, offB, t); break;
                default: break;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (threadIdx.x == 0 && idx + CV_STAGES < total) {
                mbar_wait(&empty[s], ph);
                issue(idx + CV_STAGES);
            }
        }
        const int cbase = box * CV_BHALF + colw + 2 * t;                     // + na*8 + {0,1}
        if (EPI >= EPI_LINK) {
            // ---------------- epilogue (predict): store link / response, rows of one atom are 64 contiguous bytes ----------------
#pragma unroll
            for (int ma = 0; ma < 4; ++ma) {
                const long long row = trow0 + wm * 32 + ma * 8 + g;
                if (row >= it.valid_end) continue;
#pragma unroll
                for (int na = 0; na < 10; ++na)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int c = col0 + cbase + na * 8 + h;
                        if (na >= nat || c >= nc) continue;
                        double v = acc[ma][na][h] + __ldg(b0 + (size_t)it.fold * ncld + c);
                        if (EPI == EPI_RESPONSE) v = 1.0 / (1.0 + exp(-v));
                        pred[(size_t)c * ldo + row] = v;
                    }
            }
            continue;
        }
        // ---------------- epilogue: t = measure(y - b0 - pred), tile (count, mean, M2) per column ----------------
        __syncthreads();     // ytile visible
        double s1[20];
#pragma unroll
        for (int c = 0; c < 20; ++c) s1[c] = 0.0;
#pragma unroll
        for (int ma = 0; ma < 4; ++ma) {
            const int rl = wm * 32 + ma * 8 + g;
            const bool valid = (trow0 + rl) < it.valid_end;
            const double yv = ytile[rl], wv = wtile[rl];
#pragma unroll
            for (int na = 0; na < 10; ++na)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (na >= nat) continue;
                    const int c = cbase + na * 8 + h;
                    const double link = acc[ma][na][h] + __ldg(b0 + (size_t)it.fold * ncld + col0 + c);
                    const double tv = valid ? cv_measure<EPI>(yv, link) * wv : 0.0;   // oem_xval_dense.cpp:389-401
                    acc[ma][na][h] = tv;
                    s1[na * 2 + h] += tv;
                }
        }
#pragma unroll
        for (int c = 0; c < 20; ++c) {
            double v = s1[c];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            s1[c] = v;
        }
        if (g == 0) {
#pragma unroll
            for (int na = 0; na < 10; ++na)
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (na < nat) red[(0 * NWM + wm) * COLS + cbase + na * 8 + h] = s1[na * 2 + h];
        }
        __syncthreads();
        const double cnt = (double)max(0ll, min((long long)ROWS, it.valid_end - trow0));
        double m2[20];
#pragma unroll
        for (int c = 0; c < 20; ++c) m2[c] = 0.0;
        if (cnt > 0.0) {
#pragma unroll
            for (int na = 0; na < 10; ++na)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (na >= nat) continue;
                    const int c = cbase + na * 8 + h;
                    double ssum = red[c];
#pragma unroll
                    for (int w2 = 1; w2 < NWM; ++w2) ssum += red[w2 * COLS + c];
                    const double mean = ssum / cnt;
#pragma unroll
                    for (int ma = 0; ma < 4; ++ma) {
                        const bool valid = (trow0 + wm * 32 + ma * 8 + g) < it.valid_end;
                        const double dlt = acc[ma][na][h] - mean;
                        m2[na * 2 + h] += valid ? dlt * dlt : 0.0;
                    }
                }
        }
#pragma unroll
        for (int c = 0; c < 20; ++c) {
            double v = m2[c];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            m2[c] = v;
        }
        if (g == 0) {
#pragma unroll
            for (int na = 0; na < 10; ++na)
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (na < nat) red[(1 * NWM + wm) * COLS + cbase + na * 8 + h] = m2[na * 2 + h];
        }
        __syncthreads();
        // Chan merge of the tile into the running state, one thread per column
        if (cnt > 0.0) {
            for (int c = threadIdx.x; c < COLS; c += CV_THREADS) {
                double ssum = red[c], tm2 = red[NWM * COLS + c];
#pragma unroll
                for (int w2 = 1; w2 < NWM; ++w2) { ssum += red[w2 * COLS + c]; tm2 += red[(NWM + w2) * COLS + c]; }
                const double tmean = ssum / cnt;
                const double ntot = run_cnt + cnt;
                const double dlt = tmean - run_mean[c];
                run_mean[c] += dlt * (cnt / ntot);
                run_m2[c] += tm2 + dlt * dlt * (run_cnt * cnt / ntot);
            }
        }
        run_cnt += cnt;
        __syncthreads();
    }
    if (EPI >= EPI_LINK) return;
    double *out = partial + (size_t)blockIdx.x * part_stride;
    if (threadIdx.x == 0) out[0] = run_cnt;
    for (int c = threadIdx.x; c < COLS; c += CV_THREADS) {
        out[1 + 2 * c] = run_mean[c];
        out[2 + 2 * c] = run_m2[c];
    }
}

// out[c] = (count, mean, M2) merged over this column block's items in item order.  accumulate: the merge starts from the
// (count, mean, M2) already in out3 instead of the empty state, so that row chunks scored one launch at a time merge in
// chunk order (Chan's update; from the empty state the first merge reproduces its operand exactly).
__global__ void cv_merge_kernel(const double *__restrict__ partial, int part_stride, const CvItem *__restrict__ items,
                                int nitems, int nc, int cols, double *__restrict__ out3, int accumulate) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nc) return;
    const int cb = c / cols, cl = c - cb * cols;
    double n = 0.0, mean = 0.0, m2 = 0.0;
    if (accumulate) { n = out3[c]; mean = out3[nc + c]; m2 = out3[2 * nc + c]; }
    for (int i = 0; i < nitems; ++i) {
        if (items[i].colblock != cb) continue;
        const double *pp = partial + (size_t)i * part_stride;
        const double nb = pp[0];
        if (nb <= 0.0) continue;
        const double mb = pp[1 + 2 * cl], qb = pp[2 + 2 * cl];
        const double nt = n + nb, dlt = mb - mean;
        mean += dlt * (nb / nt);
        m2 += qb + dlt * dlt * (n * nb / nt);
        n = nt;
    }
    out3[c] = n;
    out3[nc + c] = mean;
    out3[2 * nc + c] = m2;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        fail(OEMB200_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
    return reinterpret_cast<EncodeTiledFn>(p);
}

int cv_ncld(int nc) { return (nc + CV_COLS - 1) / CV_COLS * CV_COLS + 8; }

// Xs: fold-sorted, column-major, leading dimension lds (even), nrows_total rows.  B: nfolds x p x ncld (column index
// contiguous), b0: nfolds x ncld.  segs[k] = {row0, padded end, valid end}.  ws: optional observation weights in
// fold-sorted order.  epi < EPI_LINK: out = 3 x nc (count, mean, M2); else out = predictions, column-major, ld ldo.
static void cv_gemm_launch(Ctx &cx, const double *Xs, int64_t nrows_total, int p, int64_t lds, const double *ys,
                           const double *ws, int nfolds, const std::vector<std::array<int64_t, 3>> &segs,
                           const double *B, const double *b0, int nc, int epi, double *out, int64_t ldo,
                           bool accumulate = false) {
    const int ncld = cv_ncld(nc);
    const int nh = nc <= CV_BHALF ? 1 : 2;                  // narrow problems: 128 x 160 tiles
    const int cols = CV_BHALF * nh, rows = nh == 2 ? 64 : 128;
    const int ncb = (nc + cols - 1) / cols;
    if ((lds & 1) || (reinterpret_cast<uintptr_t>(Xs) & 15))
        fail(OEMB200_EINVAL, "cvscore: X must have an even leading dimension and a 16-byte aligned base");
    // items: contiguous ranges of 64-row tiles, a few waves of CTAs
    int64_t tiles_total = 0;
    for (auto &s : segs) tiles_total += (s[2] - s[0] + rows - 1) / rows;
    const int64_t target = std::max<int64_t>(1, (int64_t)cx.num_sms * 4 / ncb);
    const int64_t tiles_per_item = std::max<int64_t>(1, (tiles_total + target - 1) / target);
    std::vector<CvItem> items;
    for (int cb = 0; cb < ncb; ++cb)
        for (int k = 0; k < nfolds; ++k) {
            const int64_t nt = (segs[k][2] - segs[k][0] + rows - 1) / rows;
            for (int64_t t0 = 0; t0 < nt; t0 += tiles_per_item) {
                CvItem it;
                it.fold = k; it.colblock = cb; it.pad0 = it.pad1 = 0;
                it.row0 = segs[k][0] + t0 * rows;
                it.row_end = segs[k][0] + std::min(nt, t0 + tiles_per_item) * rows;
                it.valid_end = segs[k][2];
                items.push_back(it);
            }
        }
    if (items.empty()) fail(OEMB200_EINVAL, "cvscore: no rows");
    const int part_stride = 1 + 2 * cols;
    const bool store = epi >= EPI_LINK;
    DBuf<CvItem> d_items(items.size());
    DBuf<double> partial(store ? 1 : items.size() * (size_t)part_stride);
    d_items.upload(items.data(), items.size(), cx.stream);

    CUtensorMap tmX, tmB;
    EncodeTiledFn enc = encode_fn();
    {
        cuuint64_t dims[2] = {(cuuint64_t)nrows_total, (cuuint64_t)p};
        cuuint64_t strides[1] = {(cuuint64_t)lds * 8};
        cuuint32_t box[2] = {(cuuint32_t)rows + 4, CV_KC};
        cuuint32_t es[2] = {1, 1};
        if (enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(Xs), dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            fail(OEMB200_ECUDA, "cvscore: tensor map for X failed");
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)ncld, (cuuint64_t)nfolds * p};
        cuuint64_t strides[1] = {(cuuint64_t)ncld * 8};
        cuuint32_t box[2] = {CV_BBOX, CV_KC};
        cuuint32_t es[2] = {1, 1};
        if (enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(B), dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            fail(OEMB200_ECUDA, "cvscore: tensor map for B failed");
    }
    const size_t t0 = cx.tm->start(&cx.st.ms_cvscore);
#define CV_LAUNCH(E, H)                                                                                               \
    do {                                                                                                              \
        OEM_CUDA(cudaFuncSetAttribute(cvscore_kernel<E, H>, cudaFuncAttributeMaxDynamicSharedMemorySize,              \
                                      cv_smem_bytes(H)));                                                             \
        cvscore_kernel<E, H><<<(unsigned)items.size(), CV_THREADS, cv_smem_bytes(H), cx.stream>>>(                    \
            tmX, tmB, p, ncld, d_items.p, ys, ws, b0, partial.p, part_stride, store ? out : nullptr, (long long)ldo,  \
            nc);                                                                                                      \
    } while (0)
#define CV_LAUNCH_NH(E) do { if (nh == 1) CV_LAUNCH(E, 1); else CV_LAUNCH(E, 2); } while (0)
    switch (epi) {
        case EPI_MSE: CV_LAUNCH_NH(EPI_MSE); break;
        case EPI_MAE: CV_LAUNCH_NH(EPI_MAE); break;
        case EPI_BDEV: CV_LAUNCH_NH(EPI_BDEV); break;
        case EPI_BCLASS: CV_LAUNCH_NH(EPI_BCLASS); break;
        case EPI_BMSE: CV_LAUNCH_NH(EPI_BMSE); break;
        case EPI_BMAE: CV_LAUNCH_NH(EPI_BMAE); break;
        case EPI_LINK: CV_LAUNCH_NH(EPI_LINK); break;
        default: CV_LAUNCH_NH(EPI_RESPONSE); break;
    }
#undef CV_LAUNCH_NH
#undef CV_LAUNCH
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
    if (!store) {
        cv_merge_kernel<<<(nc + 127) / 128, 128, 0, cx.stream>>>(partial.p, part_stride, d_items.p, (int)items.size(), nc, cols, out,
                                                                 accumulate ? 1 : 0);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 1;
    }
    cx.tm->stop(t0);
}

void cvscore_launch(Ctx &cx, const double *Xs, int64_t nrows_total, int p, int64_t lds, const double *ys,
                    const double *ws, int nfolds, const std::vector<std::array<int64_t, 3>> &segs, const double *B,
                    const double *b0, int nc, bool mae, double *out3, bool accumulate) {
    cv_gemm_launch(cx, Xs, nrows_total, p, lds, ys, ws, nfolds, segs, B, b0, nc, mae ? EPI_MAE : EPI_MSE, out3, 0, accumulate);
}

void cvscore_binomial_launch(Ctx &cx, const double *Xs, int64_t nrows_total, int p, int64_t lds, const double *ys, int nfolds,
                             const std::vector<std::array<int64_t, 3>> &segs, const double *B, const double *b0, int nc,
                             int measure, double *out3) {
    if (measure < 0 || measure > 3) fail(OEMB200_EINVAL, "cvscore: binomial measure %d", measure);
    cv_gemm_launch(cx, Xs, nrows_total, p, lds, ys, nullptr, nfolds, segs, B, b0, nc, EPI_BDEV + measure, out3, 0);
}

// pred (n x nc, column-major, ld ldo) = X (n x p) * B (p x ncld layout of cvscore) + b0, optionally through the logistic
// link: the GEMM of predict.oem (R/methods.R:113-118, 355-358) on the CV-scoring kernel with a store epilogue.
void predict_launch(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, const double *B, const double *b0, int nc,
                    bool response, double *pred, int64_t ldo) {
    std::vector<std::array<int64_t, 3>> segs{{0, n, n}};
    cv_gemm_launch(cx, X, n, p, ld, nullptr, nullptr, 1, segs, B, b0, nc, response ? EPI_RESPONSE : EPI_LINK, pred, ldo);
}

}  // namespace oemb200
