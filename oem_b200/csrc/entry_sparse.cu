// entry_sparse.cu -- oemb200_fit_sparse <- oem_fit_sparse  src/oem_sparse.cpp:30-264 (+ oem_sparse.h), SURVEY.md 8f row 4.
//
// X arrives as the three slots of a Matrix::dgCMatrix (compressed sparse column: i = 0-based row indices, p = column
// pointers, x = values; R/oem.R:236-240 coerces every sparseMatrix to it).  What the reference computes from it
// (oem_sparse.h:490-636, 791-862) are the same sufficient statistics as oem_big -- X'X (dense p x p), column sums,
// X'y, column sums of squares -- so the sparse entry only replaces the data pass; assembly, top eigenvalue and the whole
// lambda path are the kernels every other entry uses.
//
// Data pass, all deterministic (no floating-point atomics):
//   csc_colstats_kernel   one CTA per column: sum x, sum x*y, sum x^2                       (oem_sparse.h:495-507, 580, 829)
//   csr_count / scan / fill / sort_rows   CSC -> CSR on the device (integer atomics only; rows are then put into
//                         ascending column order by ranking, so every later sum has a fixed order)
//   sparse_gram_kernel    CTA (j, split): for every stored x_ij of column j (32 at a time per warp, chunks dealt round-robin
//                         to the warps) add x_ij * row_i into the warp's private p-vector in shared memory; fixed-order
//                         reduce over warps, then over splits -> column j of X'X.  Work = sum_i nnz(row i)^2 multiply-adds, the
//                         same count as the row-wise outer-product form Eigen's rankUpdate performs (oem_sparse.h:341-344)
//   sparse_loss_kernel    compute.loss: one warp per row, lanes over the (penalty, lambda) columns       (oem_sparse.h:918-943)
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>
#include "host_common.h"

namespace oemb200 {

// ------------------------------------------------------------------------------------------------ column statistics
__global__ void __launch_bounds__(256) csc_colstats_kernel(const int *__restrict__ col_ptr, const int *__restrict__ row_idx,
                                                           const double *__restrict__ val, const double *__restrict__ y,
                                                           int p, double *__restrict__ stats) {
    const int j = blockIdx.x;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    for (int e = col_ptr[j] + threadIdx.x; e < col_ptr[j + 1]; e += 256) {
        const double v = val[e];
        s0 += v;
        s1 = fma(v, y[row_idx[e]], s1);
        s2 = fma(v, v, s2);
    }
    __shared__ double sh[3][8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_down_sync(0xffffffffu, s0, o);
        s1 += __shfl_down_sync(0xffffffffu, s1, o);
        s2 += __shfl_down_sync(0xffffffffu, s2, o);
    }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s0; sh[1][threadIdx.x >> 5] = s1; sh[2][threadIdx.x >> 5] = s2; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sh[threadIdx.x][w];
        stats[(size_t)threadIdx.x * p + j] = t;
    }
}

// ------------------------------------------------------------------------------------------------ CSC -> CSR
__global__ void csr_count_kernel(const int *__restrict__ row_idx, int nnz, int *__restrict__ cnt) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nnz) atomicAdd(&cnt[row_idx[e]], 1);
}

constexpr int SCAN_ITEMS = 4, SCAN_THREADS = 1024, SCAN_TILE = SCAN_ITEMS * SCAN_THREADS;

// exclusive scan of one tile in place; the tile total goes to totals[blockIdx.x]
__device__ __forceinline__ int block_exclusive_scan(int v, int *total) {
    __shared__ int wsum[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
        int s = wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        wsum[lane] = s;
    }
    __syncthreads();
    const int base = w ? wsum[w - 1] : 0;
    *total = wsum[31];
    __syncthreads();
    return base + inc - v;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_tiles_kernel(int *__restrict__ a, int n, int *__restrict__ totals) {
    const int i0 = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS], s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) { v[k] = (i0 + k < n) ? a[i0 + k] : 0; s += v[k]; }
    int total;
    int ex = block_exclusive_scan(s, &total);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        if (i0 + k < n) a[i0 + k] = ex;
        ex += v[k];
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = total;
}

// one CTA: exclusive scan of the tile totals (any count, chunk by chunk with a running carry)
__global__ void __launch_bounds__(SCAN_THREADS) scan_totals_kernel(int *__restrict__ totals, int nt) {
    int carry = 0;
    for (int c0 = 0; c0 < nt; c0 += SCAN_THREADS) {
        const int i = c0 + threadIdx.x;
        const int v = i < nt ? totals[i] : 0;
        int total;
        const int ex = block_exclusive_scan(v, &total);
        if (i < nt) totals[i] = carry + ex;
        carry += total;
    }
}

// row_ptr[i] = tile-local scan + tile offset; row_ptr[n] = nnz; cursor = row_ptr copy for the fill
__global__ void scan_finish_kernel(int *__restrict__ row_ptr, int n, const int *__restrict__ totals, int nnz,
                                   int *__restrict__ cursor) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int v = row_ptr[i] + totals[i / SCAN_TILE];
        row_ptr[i] = v;
        cursor[i] = v;
    } else if (i == n) row_ptr[n] = nnz;
}

__global__ void __launch_bounds__(256) csr_fill_kernel(const int *__restrict__ col_ptr, const int *__restrict__ row_idx,
                                                       const double *__restrict__ val, int *__restrict__ cursor,
                                                       int *__restrict__ csr_col, double *__restrict__ csr_val) {
    const int j = blockIdx.x;
    for (int e = col_ptr[j] + threadIdx.x; e < col_ptr[j + 1]; e += 256) {
        const int pos = atomicAdd(&cursor[row_idx[e]], 1);
        csr_col[pos] = j;
        csr_val[pos] = val[e];
    }
}

// The fill's atomics leave a row's entries in arbitrary order.  The Gram does not care (distinct slots), but the loss sums
// along a row, so rows are put into ascending column order: one warp per row, every entry's position is its rank (the
// number of smaller column indices) -- m^2 / 32 comparisons per lane for a row of m entries, never more than the Gram's
// own m^2 multiply-adds for that row.
__global__ void __launch_bounds__(256) csr_sort_rows_kernel(const int *__restrict__ row_ptr, int n, const int *__restrict__ col_in,
                                                            const double *__restrict__ val_in, int *__restrict__ col_out,
                                                            double *__restrict__ val_out) {
    const int lane = threadIdx.x & 31;
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    const int s = row_ptr[i], m = row_ptr[i + 1] - s;
    for (int base = 0; base < m; base += 32) {
        const int k = base + lane;
        const int mycol = k < m ? col_in[s + k] : 0x7fffffff;
        const double myval = k < m ? val_in[s + k] : 0.0;
        int rank = 0;
        for (int b0 = 0; b0 < m; b0 += 32) {
            const int oc = b0 + lane < m ? col_in[s + b0 + lane] : 0x7fffffff;
#pragma unroll
            for (int t = 0; t < 32; ++t) rank += __shfl_sync(0xffffffffu, oc, t) < mycol;
        }
        if (k < m) { col_out[s + rank] = mycol; val_out[s + rank] = myval; }
    }
}

// ------------------------------------------------------------------------------------------------ sparse Gram
// grid (p, nsplit); dynamic smem = nwarps * p doubles.  Split s of column j owns the contiguous part
// [e0 + s * len, e0 + (s + 1) * len) of the column's stored entries.
__global__ void __launch_bounds__(256) sparse_gram_kernel(const int *__restrict__ col_ptr, const int *__restrict__ row_idx,
                                                          const double *__restrict__ val, const int *__restrict__ row_ptr,
                                                          const int *__restrict__ csr_col, const double *__restrict__ csr_val,
                                                          const double *__restrict__ roww, int p, int nwarps,
                                                          double *__restrict__ Gpart) {
    extern __shared__ double acc[];
    const int j = blockIdx.x, s = blockIdx.y, ns = gridDim.y;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int c = threadIdx.x; c < nwarps * p; c += blockDim.x) acc[c] = 0.0;
    __syncthreads();
    const int e0 = col_ptr[j], e1 = col_ptr[j + 1];
    const int len = (e1 - e0 + ns - 1) / ns;
    const int b = e0 + s * len, e = min(b + len, e1);
    if (w < nwarps) {
        double *a = acc + (size_t)w * p;
        const unsigned lt = (1u << lane) - 1u;
        // A warp takes 32 stored entries of column j at a time: lane l owns entry t = chunk + l (row i_l, value x_l, the
        // row's CSR extent).  The rows' entries are then walked as ONE flat list, 32 per step, so every step has 32
        // independent loads in flight instead of one short row's worth (the first version: long_scoreboard 20.7 warps per
        // issue, profiles/r01_sparse_gram_ncu_summary.md).  Two lanes of a step can hit the same slot (different rows,
        // same column): they are applied in lane order = flat order, so each slot still sees a fixed sequence of adds.
        for (int chunk = b + w * 32; chunk < e; chunk += nwarps * 32) {
            const int t = chunk + lane;
            const bool own = t < e;
            const int i = own ? row_idx[t] : 0;
            const double xv = own ? (roww ? val[t] * roww[i] : val[t]) : 0.0;     // X'WX: the row weight rides on x_ij
            const int rs = own ? row_ptr[i] : 0;
            const int m = own ? row_ptr[i + 1] - rs : 0;
            int inc = m;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += v;
            }
            const int pre = inc - m;                                   // exclusive prefix of the row lengths
            const int T = __shfl_sync(0xffffffffu, inc, 31);
            for (int f0 = 0; f0 < T; f0 += 32) {
                const int f = f0 + lane;
                const bool act = f < T;
                int u = 0;                                             // last lane whose prefix is <= f: the owning row
#pragma unroll
                for (int step = 16; step > 0; step >>= 1) {
                    const int cand = u + step;
                    const int pc = __shfl_sync(0xffffffffu, pre, cand & 31);
                    if (cand < 32 && pc <= f) u = cand;
                }
                const int k = __shfl_sync(0xffffffffu, rs, u) + (f - __shfl_sync(0xffffffffu, pre, u));
                const double x = __shfl_sync(0xffffffffu, xv, u);
                const int c = act ? csr_col[k] : -1 - lane;            // inactive lanes get unique dummies
                const double v = act ? csr_val[k] : 0.0;
                const unsigned same = __match_any_sync(0xffffffffu, c);
                const unsigned r = __popc(same & lt);                  // my position among the lanes hitting slot c
                const unsigned rmax = __reduce_max_sync(0xffffffffu, act ? r : 0u);
                for (unsigned rr = 0; rr <= rmax; ++rr) {
                    if (act && r == rr) a[c] = fma(x, v, a[c]);
                    __syncwarp();
                }
            }
        }
    }
    __syncthreads();
    double *out = Gpart + ((size_t)s * p + j) * p;
    for (int c = threadIdx.x; c < p; c += blockDim.x) {
        double t = 0.0;
        for (int ww = 0; ww < nwarps; ++ww) t += acc[(size_t)ww * p + c];
        out[c] = t;
    }
}

// ---- dense route for not-so-sparse designs: rows [r0, r1) of the CSC matrix scattered into a zeroed column-major tile ----
__global__ void __launch_bounds__(256) csc_densify_kernel(const int *__restrict__ col_ptr, const int *__restrict__ row_idx,
                                                          const double *__restrict__ val, int r0, int r1, long long ld,
                                                          double *__restrict__ dense) {
    const int j = blockIdx.x;
    for (int e = col_ptr[j] + threadIdx.x; e < col_ptr[j + 1]; e += 256) {
        const int i = row_idx[e];
        if (i >= r0 && i < r1) dense[(size_t)j * ld + (i - r0)] = val[e];
    }
}

// sum_i nnz(row i)^2 = multiply-adds of the sparse route (one partial per CTA, summed on the host)
__global__ void __launch_bounds__(256) row_pairs_kernel(const int *__restrict__ row_ptr, int n, double *__restrict__ partial) {
    double s = 0.0;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        const double m = (double)(row_ptr[i + 1] - row_ptr[i]);
        s = fma(m, m, s);
    }
    __shared__ double sh[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sh[w];
        partial[blockIdx.x] = t;
    }
}

__global__ void sum_splits_kernel(const double *__restrict__ Gpart, int ns, size_t pp, double *__restrict__ G) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= pp) return;
    double t = 0.0;
    for (int s = 0; s < ns; ++s) t += Gpart[(size_t)s * pp + e];
    G[e] = t;
}

// ------------------------------------------------------------------------------------------------ loss
// Bt: p x C row-major (row = variable, C = all (penalty, lambda) columns), b0: C.  One warp per row, lanes over columns in
// chunks of 32 * LOSS_CPL; per-warp partial sums, summed in fixed order by sum_partials below.
constexpr int LOSS_CPL = 4;
__global__ void __launch_bounds__(256) sparse_loss_kernel(const int *__restrict__ row_ptr, const int *__restrict__ csr_col,
                                                          const double *__restrict__ csr_val, const double *__restrict__ y,
                                                          int n, const double *__restrict__ Bt, const double *__restrict__ b0,
                                                          int C, double *__restrict__ partial) {
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (int c0 = 0; c0 < C; c0 += 32 * LOSS_CPL) {
        double sum[LOSS_CPL], bb[LOSS_CPL];
#pragma unroll
        for (int u = 0; u < LOSS_CPL; ++u) {
            const int c = c0 + u * 32 + lane;
            sum[u] = 0.0;
            bb[u] = c < C ? b0[c] : 0.0;
        }
        for (int i = gw; i < n; i += nw) {
            double pr[LOSS_CPL];
#pragma unroll
            for (int u = 0; u < LOSS_CPL; ++u) pr[u] = 0.0;
            for (int k = row_ptr[i]; k < row_ptr[i + 1]; ++k) {
                const double v = csr_val[k];
                const double *brow = Bt + (size_t)csr_col[k] * C;
#pragma unroll
                for (int u = 0; u < LOSS_CPL; ++u) {
                    const int c = c0 + u * 32 + lane;
                    if (c < C) pr[u] = fma(v, brow[c], pr[u]);
                }
            }
            const double yi = y[i];
#pragma unroll
            for (int u = 0; u < LOSS_CPL; ++u) {
                const double r = (yi - pr[u]) - bb[u];          // (Y - X b).array() - beta(0)   oem_sparse.h:925
                sum[u] = fma(r, r, sum[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < LOSS_CPL; ++u) {
            const int c = c0 + u * 32 + lane;
            if (c < C) partial[(size_t)gw * C + c] = sum[u];
        }
    }
}

__global__ void sum_rows_kernel(const double *__restrict__ partial, int rows, int C, double *__restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double t = 0.0;
    for (int r = 0; r < rows; ++r) t += partial[(size_t)r * C + c];
    out[c] = t;
}

// ------------------------------------------------------------------------------------------------ logistic SpMV
// eta_i = sum_k x_ik b[col_k] + *b0; prob = 1 / (1 + exp(-eta)); resid = y - prob; w = prob (1 - prob)
// (src/oem_logistic_sparse.h:864-946).  8 lanes per row, fixed-order 3-step butterfly.
__global__ void __launch_bounds__(256) sparse_xb_logistic_kernel(const int *__restrict__ row_ptr, const int *__restrict__ csr_col,
                                                                 const double *__restrict__ csr_val, int n,
                                                                 const double *__restrict__ b, const double *__restrict__ b0,
                                                                 const double *__restrict__ y, double *__restrict__ prob,
                                                                 double *__restrict__ resid, double *__restrict__ w) {
    const int sub = threadIdx.x & 7;
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    double e = 0.0;
    if (i < n)
        for (int k = row_ptr[i] + sub; k < row_ptr[i + 1]; k += 8) e = fma(csr_val[k], b[csr_col[k]], e);
    e += __shfl_xor_sync(0xffffffffu, e, 4);
    e += __shfl_xor_sync(0xffffffffu, e, 2);
    e += __shfl_xor_sync(0xffffffffu, e, 1);
    if (i < n && sub == 0) {
        e += b0 ? *b0 : 0.0;
        const double pr = 1.0 / (1.0 + exp(-e));
        if (prob) prob[i] = pr;
        if (resid) resid[i] = y[i] - pr;
        if (w) w[i] = pr * (1.0 - pr);
    }
}

// ------------------------------------------------------------------------------------------------ driver
// CSC slots -> CSR copy on the device, rows in ascending column order (count / scan / fill / rank-sort above)
struct DeviceCsr {
    DBuf<int> row_ptr, col;
    DBuf<double> val;
    void build(Ctx &cx, const int *d_cp, const int *d_ri, const double *d_v, int64_t n, int p, int nnz) {
        const int ntile = (int)((n + SCAN_TILE - 1) / SCAN_TILE);
        DBuf<int> cursor((size_t)n), totals((size_t)ntile), col_u((size_t)std::max(nnz, 1));
        DBuf<double> val_u((size_t)std::max(nnz, 1));
        row_ptr.alloc((size_t)n + 1);
        col.alloc((size_t)std::max(nnz, 1));
        val.alloc((size_t)std::max(nnz, 1));
        row_ptr.zero(cx.stream);
        if (nnz > 0) csr_count_kernel<<<(nnz + 255) / 256, 256, 0, cx.stream>>>(d_ri, nnz, row_ptr.p);
        scan_tiles_kernel<<<ntile, SCAN_THREADS, 0, cx.stream>>>(row_ptr.p, (int)n, totals.p);
        scan_totals_kernel<<<1, SCAN_THREADS, 0, cx.stream>>>(totals.p, ntile);
        scan_finish_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, cx.stream>>>(row_ptr.p, (int)n, totals.p, nnz, cursor.p);
        csr_fill_kernel<<<p, 256, 0, cx.stream>>>(d_cp, d_ri, d_v, cursor.p, col_u.p, val_u.p);
        csr_sort_rows_kernel<<<(unsigned)((n + 7) / 8), 256, 0, cx.stream>>>(row_ptr.p, (int)n, col_u.p, val_u.p, col.p, val.p);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 5 + (nnz > 0 ? 1 : 0);
    }
};

template <typename T>
static const T *to_device_array(Ctx &cx, const T *h, size_t cnt, DBuf<T> &own) {
    if (cnt == 0) return nullptr;
    if (is_device_ptr(h)) return h;
    own.alloc(cnt);
    own.upload(h, cnt, cx.stream);
    cx.st.h2d_bytes += (int64_t)(cnt * sizeof(T));
    return own.p;
}

// dgCMatrix invariants: 0 <= i < n, strictly increasing inside every column (no duplicates).  flag: bit 0 = range, bit 1 = order
__global__ void __launch_bounds__(256) csc_validate_kernel(const int *__restrict__ col_ptr, const int *__restrict__ row_idx, int n,
                                                           int *__restrict__ flag) {
    const int j = blockIdx.x;
    int bad = 0;
    for (int e = col_ptr[j] + threadIdx.x; e < col_ptr[j + 1]; e += 256) {
        const int i = row_idx[e];
        if (i < 0 || i >= n) bad |= 1;
        if (e > col_ptr[j] && row_idx[e - 1] >= i) bad |= 2;
    }
    if (bad) atomicOr(flag, bad);
}

// validated CSC slots on the device
struct CscInput {
    DBuf<int> o_cp, o_ri;
    DBuf<double> o_v;
    const int *cp = nullptr, *ri = nullptr;
    const double *v = nullptr;
    int nnz = 0;
    void load(Ctx &cx, const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p) {
        std::vector<int> h_cp(p + 1);
        if (is_device_ptr(col_ptr)) {
            OEM_CUDA(cudaMemcpyAsync(h_cp.data(), col_ptr, sizeof(int) * (p + 1), cudaMemcpyDeviceToHost, cx.stream));
            cx.sync();
        } else memcpy(h_cp.data(), col_ptr, sizeof(int) * (p + 1));
        if (h_cp[0] != 0) fail(OEMB200_EINVAL, "sparse: col_ptr[0] must be 0");
        for (int j = 0; j < p; ++j)
            if (h_cp[j + 1] < h_cp[j]) fail(OEMB200_EINVAL, "sparse: col_ptr must be non-decreasing");
        nnz = h_cp[p];
        if (nnz > 0 && (!row_idx || !values)) fail(OEMB200_EINVAL, "sparse: row_idx / values missing");
        cp = to_device_array(cx, col_ptr, (size_t)p + 1, o_cp);
        ri = to_device_array(cx, row_idx, (size_t)nnz, o_ri);
        v = to_device_array(cx, values, (size_t)nnz, o_v);
        if (nnz > 0) {
            DBuf<int> flag(1);
            flag.zero(cx.stream);
            csc_validate_kernel<<<p, 256, 0, cx.stream>>>(cp, ri, (int)n, flag.p);
            OEM_CUDA(cudaGetLastError());
            cx.st.kernel_launches += 1;
            int h = 0;
            flag.download(&h, 1, cx.stream);
            cx.sync();
            if (h & 1) fail(OEMB200_EINVAL, "sparse: a row index is outside [0, n)");
            if (h & 2) fail(OEMB200_EINVAL, "sparse: row indices must be strictly increasing inside every column (dgCMatrix invariant)");
        }
    }
};

// The design as the kernels need it: validated CSC slots, the CSR copy, sum_i nnz(row i)^2 (route cost model)
struct SparseDesign {
    CscInput in;
    DeviceCsr csr;
    int64_t n = 0;
    int p = 0;
    double row_pairs = 0.0;
};

SparseDesign *sparse_design_create(Ctx &cx, const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p) {
    std::unique_ptr<SparseDesign> sd(new SparseDesign());
    sd->n = n; sd->p = p;
    sd->in.load(cx, row_idx, col_ptr, values, n, p);
    sd->csr.build(cx, sd->in.cp, sd->in.ri, sd->in.v, n, p, sd->in.nnz);
    const int npart = 4 * cx.num_sms;
    DBuf<double> pairs_part((size_t)npart);
    row_pairs_kernel<<<npart, 256, 0, cx.stream>>>(sd->csr.row_ptr.p, (int)n, pairs_part.p);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
    std::vector<double> h_pairs(npart);
    pairs_part.download(h_pairs.data(), npart, cx.stream);
    cx.sync();
    for (double v : h_pairs) sd->row_pairs += v;
    return sd.release();
}
void sparse_design_destroy(SparseDesign *sd) { delete sd; }
int sparse_design_nnz(const SparseDesign *sd) { return sd->in.nnz; }

// stats3p[0*p + j] = sum_i x_ij, [1*p + j] = sum_i x_ij v_i, [2*p + j] = sum_i x_ij^2
void sparse_colstats_launch(Ctx &cx, const SparseDesign *sd, const double *v, double *stats3p) {
    csc_colstats_kernel<<<sd->p, 256, 0, cx.stream>>>(sd->in.cp, sd->in.ri, sd->in.v, v, sd->p, stats3p);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

void sparse_xb_logistic_launch(Ctx &cx, const SparseDesign *sd, const double *b, const double *b0_dev, const double *y,
                               double *prob, double *resid, double *w) {
    const unsigned grid = (unsigned)((sd->n * 8 + 255) / 256);
    sparse_xb_logistic_kernel<<<grid, 256, 0, cx.stream>>>(sd->csr.row_ptr.p, sd->csr.col.p, sd->csr.val.p, (int)sd->n, b, b0_dev, y,
                                                          prob, resid, w);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
    cx.st.xb_launches += 1;
}

// G (p x p, column-major, full) = X' diag(roww) X; roww may be NULL.
// Route: the sparse kernel costs sum_i nnz(row i)^2 shared-memory multiply-adds at ~8e10 / s (measured: n = 1e6,
// p = 1000: 1.8 ms at 1 % density, 31 ms at 5 %), the dense route (scatter 2 GB row blocks into a zeroed tile, TMA / DMMA
// Gram on each) a flat 43 ms at that shape, i.e. n p (p + 1) flops at ~2.4e13 / s all in.  From about 6 % density on the
// dense route is cheaper (same deterministic result, different rounding).
void sparse_gram_launch(Ctx &cx, const SparseDesign *sd, const double *roww, double *G) {
    const int p = sd->p;
    const int64_t n = sd->n;
    const size_t pp2 = (size_t)p * p;
    const char *route_env = getenv("OEMB200_SPARSE_ROUTE");       // "dense" / "sparse" force a route (tests, A/B)
    bool dense_route = 300.0 * sd->row_pairs > (double)n * p * (p + 1.0) && p >= 64;
    if (route_env && !strcmp(route_env, "dense")) dense_route = true;
    if (route_env && !strcmp(route_env, "sparse")) dense_route = false;
    if (dense_route) {
        const int64_t align = 2 * gram_kt();
        int64_t rows = (int64_t)((double)(1ll << 31) / (8.0 * p));
        rows = std::max<int64_t>(align, rows / align * align);
        rows = std::min<int64_t>(rows, (n + align - 1) / align * align);
        DBuf<double> tile((size_t)rows * p);
        for (int64_t r0 = 0, c = 0; r0 < n; r0 += rows, ++c) {
            const int64_t nr = std::min(rows, n - r0);
            tile.zero(cx.stream);
            csc_densify_kernel<<<p, 256, 0, cx.stream>>>(sd->in.cp, sd->in.ri, sd->in.v, (int)r0, (int)(r0 + nr), (long long)rows, tile.p);
            OEM_CUDA(cudaGetLastError());
            cx.st.kernel_launches += 1;
            gram_launch(cx, tile.p, nr, p, rows, {RowSegment{0, nr, 0}}, 1, nullptr, roww ? roww + r0 : nullptr, G, c > 0);
        }
        return;
    }
    int nwarps = 8;
    while (nwarps > 1 && (size_t)nwarps * p * 8 > cx.smem_optin) nwarps >>= 1;
    if ((size_t)nwarps * p * 8 > cx.smem_optin) fail(OEMB200_EUNSUPPORTED, "sparse: p = %d exceeds the shared-memory accumulator", p);
    const int nsplit = std::max(1, std::min(16, (4 * cx.num_sms + p - 1) / p));
    PhaseTimers &tm = *cx.tm;
    const size_t t_k = tm.start(&cx.st.ms_gram);
    DBuf<double> Gpart;
    double *gout = G;
    if (nsplit > 1) { Gpart.alloc((size_t)nsplit * pp2); gout = Gpart.p; }
    const size_t smem = (size_t)nwarps * p * 8;
    OEM_CUDA(cudaFuncSetAttribute(sparse_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sparse_gram_kernel<<<dim3(p, nsplit), 256, smem, cx.stream>>>(sd->in.cp, sd->in.ri, sd->in.v, sd->csr.row_ptr.p, sd->csr.col.p,
                                                                 sd->csr.val.p, roww, p, nwarps, gout);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
    if (nsplit > 1) {
        sum_splits_kernel<<<(unsigned)((pp2 + 255) / 256), 256, 0, cx.stream>>>(Gpart.p, nsplit, pp2, G);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 1;
    }
    cx.st.gram_launches += 1;
    tm.stop(t_k);
}

// out[i + c * ldo] = b0[c] + sum_k x_ik Bt[col_k, c] (+ logistic response): one warp per row, lanes over the columns
__global__ void __launch_bounds__(256) sparse_predict_kernel(const int *__restrict__ row_ptr, const int *__restrict__ csr_col,
                                                             const double *__restrict__ csr_val, int n,
                                                             const double *__restrict__ Bt, const double *__restrict__ b0,
                                                             int C, int response, double *__restrict__ out, long long ldo) {
    const int lane = threadIdx.x & 31;
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = gw; i < n; i += nw) {
        const int k0 = row_ptr[i], k1 = row_ptr[i + 1];
        for (int c = lane; c < C; c += 32) {
            double pr = 0.0;
            for (int k = k0; k < k1; ++k) pr = fma(csr_val[k], Bt[(size_t)csr_col[k] * C + c], pr);
            pr += b0[c];
            out[i + (size_t)c * ldo] = response ? 1.0 / (1.0 + exp(-pr)) : pr;
        }
    }
}

void predict_sparse_entry(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *beta,
                          int nrows, int L, int type, double *out, int64_t ldo, const oemb200_opts *o, oemb200_stats *stats) {
    if (!col_ptr || !beta || !out || !o) fail(OEMB200_EINVAL, "col_ptr / beta / out / opts must not be NULL");
    if (n < 1 || p < 1 || L < 1 || ldo < n || n >= (1ll << 31))
        fail(OEMB200_EINVAL, "bad dimensions n=%lld p=%d L=%d ldo=%lld", (long long)n, p, L, (long long)ldo);
    if (nrows != p && nrows != p + 1)
        fail(OEMB200_EINVAL, "beta has %d rows; newx has %d columns (expected %d or %d)", nrows, p, p, p + 1);   // R/methods.R:115-116
    if (type != 0 && type != 1) fail(OEMB200_EINVAL, "type must be 0 (link) or 1 (response)");
    if (is_device_ptr(beta)) fail(OEMB200_EINVAL, "beta must be a host pointer");
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    CscInput in;
    in.load(cx, row_idx, col_ptr, values, n, p);
    DeviceCsr csr;
    csr.build(cx, in.cp, in.ri, in.v, n, p, in.nnz);
    const int icpt = nrows - p;
    std::vector<double> hBt((size_t)p * L), hb0(L, 0.0);
    for (int c = 0; c < L; ++c) {
        const double *col = beta + (size_t)c * nrows;
        if (icpt) hb0[c] = col[0];
        for (int j = 0; j < p; ++j) hBt[(size_t)j * L + c] = col[icpt + j];
    }
    DBuf<double> dBt(hBt.size()), db0(L), dout;
    dBt.upload(hBt.data(), hBt.size(), cx.stream);
    db0.upload(hb0.data(), L, cx.stream);
    const bool out_dev = is_device_ptr(out);
    double *po = out;
    int64_t ldp = ldo;
    if (!out_dev) { dout.alloc((size_t)n * L); po = dout.p; ldp = n; }
    const size_t t_k = tm.start(&cx.st.ms_cvscore);
    sparse_predict_kernel<<<4 * cx.num_sms, 256, 0, cx.stream>>>(csr.row_ptr.p, csr.col.p, csr.val.p, (int)n, dBt.p, db0.p, L,
                                                               type, po, (long long)ldp);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
    tm.stop(t_k);
    if (!out_dev) {
        OEM_CUDA(cudaMemcpy2DAsync(out, (size_t)ldo * 8, po, (size_t)n * 8, (size_t)n * 8, L, cudaMemcpyDeviceToHost, cx.stream));
        cx.st.d2h_bytes += (int64_t)n * L * 8;
    }
    tm.stop(t_total);
    cx.finish();
    if (stats) *stats = cx.st;
}

void fit_sparse(const int *row_idx, const int *col_ptr, const double *values, int64_t n, int p, const double *y,
                const oemb200_spec *s, const oemb200_opts *o, oemb200_result *res) {
    check_common(s, o, res, "gaussian");
    if (n < 1 || p < 1 || !col_ptr || !y) fail(OEMB200_EINVAL, "bad sparse input: n=%lld p=%d", (long long)n, p);
    if (n >= (1ll << 31)) fail(OEMB200_EINVAL, "sparse: more than 2^31-1 rows per call; shard the rows");
    const int icpt = s->intercept ? 1 : 0, q = p + icpt;
    Ctx cx(o);
    PhaseTimers &tm = *cx.tm;
    const size_t t_total = tm.start(&cx.st.ms_total);
    Setup su;
    su.parse(s, q, /*scan=*/q, /*zero_w0=*/false);      // scans all of `groups` (src/oem_sparse.h:466)

    // ---- inputs to the device, CSC -> CSR ----
    const size_t t_h = tm.start(&cx.st.ms_h2d);
    std::unique_ptr<SparseDesign, void (*)(SparseDesign *)> sd(nullptr, sparse_design_destroy);
    collective_guard(cx, [&] { sd.reset(sparse_design_create(cx, row_idx, col_ptr, values, n, p)); });   // dgCMatrix checks are per rank
    DBuf<int> &row_ptr = sd->csr.row_ptr, &csr_col = sd->csr.col;
    DBuf<double> &csr_val = sd->csr.val;
    DevVector yv;
    to_device_vector(cx, y, n, yv);
    tm.stop(t_h);

    // bundle = [G p*p | stats 3p | sum y, sum y^2 | n]  -> one all-reduce (row-sharded runs)
    const size_t pp2 = (size_t)p * p;
    const size_t nb = pp2 + 3 * (size_t)p + 3;
    DBuf<double> bundle(nb);
    bundle.zero(cx.stream);
    double *G = bundle.p, *stats = G + pp2, *ysum = stats + 3 * (size_t)p, *nobs = ysum + 2;

    const size_t t_c = tm.start(&cx.st.ms_colstats);
    vecsum_launch(cx, yv.p, n, 0.0, ysum, false);
    sparse_colstats_launch(cx, sd.get(), yv.p, stats);
    tm.stop(t_c);

    // ---- X'X ----
    sparse_gram_launch(cx, sd.get(), nullptr, G);

    const double nd = (double)n;
    OEM_CUDA(cudaMemcpyAsync(nobs, &nd, 8, cudaMemcpyHostToDevice, cx.stream));
    const size_t t_ar = tm.start(&cx.st.ms_allreduce);
    cx.all_reduce(bundle.p, (int64_t)nb);
    tm.stop(t_ar);
    double n_tot = 0.0;
    OEM_CUDA(cudaMemcpyAsync(&n_tot, nobs, 8, cudaMemcpyDeviceToHost, cx.stream));
    cx.sync();
    // n <= p (src/oem_sparse.h:609-616, 630-640): d = 1.005 lambda_max(XX'/n) and u = X'(Y - X beta)/n + d beta on the RAW X --
    // term by term (dI - X'X/n) beta + X'y/n with the same non-zero spectrum, so the p x p route serves it.  `standardize`
    // only reaches lambda_max (XY is scaled in init_oem, :829-846, but next_u never uses XY) and get_beta() (:901-911).
    // With an intercept the reference indexes XY(n) and beta(p + 1) past their ends (XXdim = min(n, p), :782-784): rejected.
    const bool wide = !(n_tot > p);
    if (wide && icpt)
        fail(OEMB200_EUNSUPPORTED, "oem_fit_sparse with n <= p and intercept = TRUE is dimensionally inconsistent in the reference "
             "(src/oem_sparse.h:782-784, 829-841)");

    // ---- assembly: the oem_big layout, then row / column 0 times intval (src/oem_sparse.h:566-594, 829-846) ----
    const size_t t_as = tm.start(&cx.st.ms_assemble);
    DBuf<double> XX0((size_t)q * q), XY0(q), XX((size_t)q * q), XY(q), cinv(p), dscale;
    assemble_aug_launch(cx, p, icpt, s->standardize ? 1 : 0, 1, 1, G, stats, ysum, 1, nobs, nobs, XX0.p, XY0.p, cinv.p, nullptr);
    std::vector<double> hcinv(p), hsq(p), hXY(q), hXYlam;
    if (wide && s->standardize) {
        // lambda_max from the scaled XY (kept from the call above), the iteration from the raw statistics
        hXYlam.resize(q);
        XY0.download(hXYlam.data(), q, cx.stream);
        cx.sync();
        assemble_aug_launch(cx, p, 0, 0, 1, 1, G, stats, ysum, 1, nobs, nobs, XX0.p, XY0.p, nullptr, nullptr);
    }
    cinv.download(hcinv.data(), p, cx.stream);
    OEM_CUDA(cudaMemcpyAsync(hsq.data(), stats + 2 * (size_t)p, sizeof(double) * p, cudaMemcpyDeviceToHost, cx.stream));
    cx.sync();
    double intval = 1.0;
    const double *pXX = XX0.p, *pXY = XY0.p;
    if (icpt) {
        double tr = 0.0;       // xxdiag = XX.diagonal().tail(nvars).mean() of the (scaled) X block before the division by n
        for (int j = 0; j < p; ++j) tr += s->standardize ? (hcinv[j] * hsq[j]) * hcinv[j] : hsq[j];
        const double xxdiag = tr / p;
        intval = std::sqrt(xxdiag / n_tot);
        std::vector<double> hd(q, 1.0);
        hd[0] = intval;
        dscale.alloc(q);
        dscale.upload(hd.data(), q, cx.stream);
        scale_sym_launch(cx, q, dscale.p, XX0.p, XY0.p, XX.p, XY.p);
        pXX = XX.p; pXY = XY.p;
    }
    OEM_CUDA(cudaMemcpyAsync(hXY.data(), pXY, sizeof(double) * q, cudaMemcpyDeviceToHost, cx.stream));
    tm.stop(t_as);
    cx.sync();

    double lmax = 0.0;   // compute_lambda_zero: the X entries only (src/oem_sparse.h:851-862)
    for (int j = icpt; j < q; ++j) lmax = std::max(lmax, std::fabs(hXYlam.empty() ? hXY[j] : hXYlam[j]));
    su.build_lambdas(s, lmax, false);

    PenaltyTables tb(cx, su, s, p, icpt);
    PathBuffers pb;
    const size_t t_p = tm.start(&cx.st.ms_path);
    // get_beta() multiplies the member beta(0) by intval in place (src/oem_sparse.h:895-900): the path kernel's post-scale
    run_paths(cx, su, tb, o, 1, pXX, pXY, 1.005, false, icpt ? dscale.p : nullptr, pb);
    tm.stop(t_p);

    const int L = su.Lmax;
    fill_common_outputs(su, res);
    write_beta(su, pb.h_beta.data(), p, icpt, s->standardize ? hcinv.data() : nullptr, res);
    for (int pp = 0; pp < su.P; ++pp)
        for (int i = 0; i < su.nlam_run[pp]; ++i) res->niter[(size_t)pp * L + i] = pb.h_niter[(size_t)pp * L + i];
    *res->d = pb.h_d[0];

    // ---- compute.loss: all (penalty, lambda) columns in one pass over the CSR copy ----
    if (s->compute_loss && res->loss) {
        std::vector<std::pair<int, int>> cols;
        for (int pp = 0; pp < su.P; ++pp)
            for (int i = 0; i < su.nlam_run[pp]; ++i) cols.push_back({pp, i});
        const int C = (int)cols.size();
        std::vector<double> hBt((size_t)p * C), hb0(C);
        for (int c = 0; c < C; ++c) {
            const double *b = res->beta + ((size_t)cols[c].first * L + cols[c].second) * (p + 1);
            hb0[c] = b[0];
            for (int j = 0; j < p; ++j) hBt[(size_t)j * C + c] = b[1 + j];
        }
        const int nblk = 2 * cx.num_sms, nw = nblk * 8;
        DBuf<double> dBt(hBt.size()), db0(C), partial((size_t)nw * C), dloss(C);
        dBt.upload(hBt.data(), hBt.size(), cx.stream);
        db0.upload(hb0.data(), C, cx.stream);
        const size_t t_l = tm.start(&cx.st.ms_cvscore);
        sparse_loss_kernel<<<nblk, 256, 0, cx.stream>>>(row_ptr.p, csr_col.p, csr_val.p, yv.p, (int)n, dBt.p, db0.p, C, partial.p);
        sum_rows_kernel<<<(C + 127) / 128, 128, 0, cx.stream>>>(partial.p, nw, C, dloss.p);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 2;
        tm.stop(t_l);
        cx.all_reduce(dloss.p, C);
        std::vector<double> hl(C);
        dloss.download(hl.data(), C, cx.stream);
        cx.sync();
        for (int c = 0; c < C; ++c) res->loss[(size_t)cols[c].first * L + cols[c].second] = hl[c];
    }
    finish_stats(cx, tm, t_total, res);
}

}  // namespace oemb200
