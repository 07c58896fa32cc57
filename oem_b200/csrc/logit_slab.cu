// logit_slab.cu -- one IRLS data pass of the logistic path with X read from HBM ONCE and kept in SHARED MEMORY
// between the two products:
//     eta = X b + b0;  prob = 1 / (1 + exp(-eta));  W = prob (1 - prob);  r = y - prob      (phase 1)
//     grad_0 = sum_i r_i,   grad_j = sum_i x_ij r_i                                          (phase 2)
// replacing the two sweeps of oemLogisticDense::solve (src/oem_logistic_dense.h:864-949 and :970-992).
//
// A fit re-reads the same X a few hundred times (237 passes at BASELINE configs[3]), so X is re-laid out ONCE per
// fit into row slabs (slab_relayout_kernel): a slab is RT consecutive rows x all p columns, stored contiguously as
// [RT/2 row pairs][p columns][2 rows], 64 KB at p = 1000 / RT = 8.  Contiguous slabs keep HBM at streaming speed
// (a slab of the column-major original is p separate 64-byte segments ld*8 bytes apart, which measured 2.3 TB/s in
// round 1) and the pair-major order makes every shared-memory access a conflict-free 128-bit load.
//
// logit_slab_kernel: persistent CTAs (one or two per SM).  A CTA's slabs stream through a 3-stage ring filled with
// cp.async.bulk (TMA bulk copy, mbarrier transaction counts); every thread owns the columns j = t, t + THREADS, ...
// for the whole pass:
//     loads its columns of the slab into registers (LDS.128) and releases the stage at once (the refill is issued
//     as soon as all warps hold their share, so the ring stays full while the arithmetic runs),
//     forms its share of eta for the RT rows, multi-value butterfly over the warp, one partial per warp and row
//     through shared memory in fixed order, RT threads apply the link and publish r,
//     and accumulates grad_j += sum_i x_ij r_i from the SAME registers -- X crosses the L2 -> SM fabric once.
// Every CTA consumes every slab of its ring in order, so no waiter is ever more than one mbarrier phase behind
// (a first version let two thread groups take alternate slabs of one ring: a group could then wait on a stage two
// phases ahead, which the parity test cannot tell from "done").
// Only the per-CTA column sums leave the SM; ls_sum_partials adds them in fixed order, so the pass is
// bit-reproducible for a given grid.
#include <algorithm>
#include "runtime.h"

namespace oemb200 {

constexpr int LS_STAGES = 3;

__device__ __forceinline__ void bulk_load(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

template <int RT, int NC, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 2 : 1)
logit_slab_kernel(const double *__restrict__ slabs, long long n, int p, size_t stage_stride /* doubles */,
                  const double *__restrict__ b, const double *__restrict__ b0_ptr, const double *__restrict__ y,
                  double *__restrict__ prob, double *__restrict__ wout, double *__restrict__ partial,
                  const int *__restrict__ skip, unsigned long long *__restrict__ t_clock) {
    static_assert(RT == 4 || RT == 8 || RT == 16, "rows per slab");
    if (skip && *skip) return;               // speculatively enqueued pass of an IRLS loop that has already converged
    if (t_clock && blockIdx.x == 0 && threadIdx.x == 0) t_clock[1] = global_timer_ns();    // start mark of the pass
    constexpr int LOG_RT = RT == 4 ? 2 : (RT == 8 ? 3 : 4);
    constexpr int WARPS = THREADS / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *stages = reinterpret_cast<double *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + LS_STAGES * stage_stride * 8);
    uint64_t *empty = full + LS_STAGES;
    double *wsum = reinterpret_cast<double *>(empty + LS_STAGES + 2);      // [warps][RT]
    double *rsm = wsum + WARPS * RT;                                       // [RT]

    const long long ntiles = (n + RT - 1) / RT;
    const long long mine = ntiles > blockIdx.x ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, t = threadIdx.x;
    const uint32_t tile_bytes = (uint32_t)RT * (uint32_t)p * 8u;

    if (t == 0) {
        for (int s = 0; s < LS_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], WARPS); }
        mbar_fence_init();
    }
    __syncthreads();

    // refills are issued by thread 0, right after every warp has released the stage
    uint64_t pol = 0;
    const uint32_t pair_bytes = (uint32_t)p * 16u;
    auto issue = [&](long long k) {
        const int s = (int)(k % LS_STAGES);
        const double *src = slabs + (size_t)(blockIdx.x + k * gridDim.x) * RT * p;
        double *dst = stages + (size_t)s * stage_stride;
        mbar_arrive_expect_tx(&full[s], tile_bytes);
#pragma unroll
        for (int kk = 0; kk < RT / 2; ++kk)
            bulk_load(dst + (size_t)kk * 2 * p, src + (size_t)kk * 2 * p, pair_bytes, &full[s], pol);
    };
    if (t == 0) {
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
        for (long long k = 0; k < LS_STAGES && k < mine; ++k) issue(k);
    }

    double bj[NC], gacc[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        const int j = t + c * THREADS;
        bj[c] = j < p ? b[j] : 0.0;
        gacc[c] = 0.0;
    }
    const double b0 = b0_ptr ? *b0_ptr : 0.0;
    double rsum = 0.0;

    for (long long k = 0; k < mine; ++k) {
        const int s = (int)(k % LS_STAGES);
        const uint32_t ph = (uint32_t)((k / LS_STAGES) & 1);
        mbar_wait(&full[s], ph);
        const double2 *tile = reinterpret_cast<const double2 *>(stages + (size_t)s * stage_stride);
        double x[NC][RT], acc[RT];
#pragma unroll
        for (int i = 0; i < RT; ++i) acc[i] = 0.0;
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const int j = t + c * THREADS;
            if (j < p) {
#pragma unroll
                for (int kk = 0; kk < RT / 2; ++kk) {
                    const double2 v = tile[(size_t)kk * p + j];
                    x[c][2 * kk] = v.x; x[c][2 * kk + 1] = v.y;
                }
            } else {
#pragma unroll
                for (int i = 0; i < RT; ++i) x[c][i] = 0.0;
            }
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = fma(x[c][i], bj[c], acc[i]);
        }
        // the slab now lives in registers: hand the stage back and refill it
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (t == 0 && k + LS_STAGES < mine) {
            mbar_wait(&empty[s], ph);
            issue(k + LS_STAGES);
        }

        // multi-value butterfly: RT row sums over the 32 lanes; lane l ends with row l >> (5 - LOG_RT)
        {
            int nval = RT, off = 16;
#pragma unroll
            for (int st = 0; st < LOG_RT; ++st) {
                const int half = nval >> 1;
                const bool upper = (lane & off) != 0;
#pragma unroll
                for (int i = 0; i < half; ++i) {
                    const double send = upper ? acc[i] : acc[i + half];
                    const double keep = upper ? acc[i + half] : acc[i];
                    acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                }
                nval = half; off >>= 1;
            }
#pragma unroll
            for (int st = LOG_RT; st < 5; ++st) { acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], off); off >>= 1; }
        }
        if ((lane & ((32 >> LOG_RT) - 1)) == 0) wsum[warp * RT + (lane >> (5 - LOG_RT))] = acc[0];
        __syncthreads();
        const long long row0 = (blockIdx.x + k * gridDim.x) * RT;
        if (t < RT) {
            double e = b0;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) e += wsum[w * RT + t];
            const long long i = row0 + t;
            double r = 0.0;
            if (i < n) {
                const double pr = 1.0 / (1.0 + exp(-e));
                r = y[i] - pr;
                if (prob) prob[i] = pr;
                if (wout) wout[i] = pr * (1.0 - pr);
            }
            rsm[t] = r;
        }
        __syncthreads();
        double r[RT];
#pragma unroll
        for (int i = 0; i < RT; i += 2) {
            const double2 v = reinterpret_cast<const double2 *>(rsm)[i >> 1];
            r[i] = v.x; r[i + 1] = v.y;
        }
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            double tt = x[c][0] * r[0];
#pragma unroll
            for (int i = 1; i < RT; ++i) tt = fma(x[c][i], r[i], tt);
            gacc[c] += tt;
        }
        if (t == 0) {
            double tt = r[0];
#pragma unroll
            for (int i = 1; i < RT; ++i) tt += r[i];
            rsum += tt;
        }
    }
    double *out = partial + (size_t)blockIdx.x * (p + 1);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        const int j = t + c * THREADS;
        if (j < p) out[1 + j] = gacc[c];
    }
    if (t == 0) out[0] = rsum;
}

// out[k] = sum over the CTAs' rows of partial[c][k], in row order.  32 columns per block, 8 row lanes each summing every
// 8th row, then a fixed-order sum of the 8 lanes: same result for a given grid on every run, ~5 us instead of the 32 us a
// one-thread-per-column loop over ~300 rows took.
__global__ void __launch_bounds__(256) ls_sum_partials_kernel(const double *__restrict__ partial, int nparts, int width,
                                                              double *__restrict__ out, const int *__restrict__ skip,
                                                              unsigned long long *__restrict__ t_clock) {
    __shared__ double sm[8][33];
    if (skip && *skip) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int k = blockIdx.x * 32 + tx;
    double s = 0.0;
    if (k < width)
        for (int c = ty; c < nparts; c += 8) s += partial[(size_t)c * width + k];
    sm[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && k < width) {
        double t = sm[0][tx];
#pragma unroll
        for (int r = 1; r < 8; ++r) t += sm[r][tx];
        out[k] = t;
    }
    // device-side phase clock: slab kernel start -> (about) the end of this reduction
    if (t_clock && blockIdx.x == 0 && threadIdx.x == 0) t_clock[0] += global_timer_ns() - t_clock[1];
}

// ---------------------------------------------------------------------------------------------
// one-time re-layout: column-major X (n x p, ld) -> row slabs [tile][RT/2][p][2], zero rows beyond n
// ---------------------------------------------------------------------------------------------
constexpr int RL_ROWS = 64, RL_COLS = 32;

__global__ void __launch_bounds__(256)
slab_relayout_kernel(const double *__restrict__ X, long long n, int p, long long ld, int rt, double *__restrict__ slabs) {
    __shared__ __align__(16) double sm[RL_COLS][RL_ROWS + 2];       // 33 16-byte units per column: conflict-free 128-bit reads
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const long long r0 = (long long)blockIdx.x * RL_ROWS;
    const int c0 = blockIdx.y * RL_COLS;
    for (int cc = ty; cc < RL_COLS; cc += 8) {
        const int col = c0 + cc;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const long long row = r0 + tx + 32 * h;
            sm[cc][tx + 32 * h] = (col < p && row < n) ? X[(size_t)col * ld + row] : 0.0;
        }
    }
    __syncthreads();
    const int col = c0 + tx;
    if (col >= p) return;
    const long long nrows_pad = (n + rt - 1) / rt * rt;
    for (int pr = ty; pr < RL_ROWS / 2; pr += 8) {
        const long long row = r0 + 2 * pr;
        if (row >= nrows_pad) break;
        const long long tile = row / rt;
        const int kk = (int)(row - tile * rt) >> 1;
        const double2 v = *reinterpret_cast<const double2 *>(&sm[tx][2 * pr]);
        reinterpret_cast<double2 *>(slabs)[((size_t)tile * (rt / 2) + kk) * p + col] = v;
    }
}

// Shape of the pass for a given p: rows per slab, columns per thread, threads per CTA, CTAs per SM.  Up to p = 1024: two
// CTAs of 256 threads per SM, each with its own ring of three <= 32 KB slabs -- two independent pipelines per SM hide the
// per-slab reduction latency (measured on a B200, 16 GB: 2.36 ms against 2.43 ms with one 512-thread CTA and 64 KB slabs
// at p = 1000; 1.20 against 1.45 ms at p = 500).  For 1024 < p <= 2048, one CTA of 512 threads per SM.
struct SlabShape { int rt, nc, threads, ctas; };
static SlabShape slab_shape(int p) {
    SlabShape z{0, 0, 0, 0};
    if (p < 8 || p > 2048) return z;
    if (p <= 512) return SlabShape{8, (p + 255) / 256, 256, 2};
    if (p <= 1024) return SlabShape{4, (p + 255) / 256, 256, 2};
    return SlabShape{4, (p + 511) / 512, 512, 1};
}

int logit_slab_rows(int p) { return slab_shape(p).rt; }      // rows per slab; 0 = the slab route does not apply

// Which data-pass route a logistic fit takes by default.  From p = 128 on the slab kernel runs at the HBM copy rate.  Below,
// most of its 256 threads own no column and a pass costs ~1 us per 8-row slab and CTA, whatever p is -- but it is 2 launches
// against the 5 of the two column sweeps, which decides problems small enough to be launch-bound.  Measured on a B200
// (40 lambdas, ms per fit, slab / sweeps): n = 5e4: p = 8 14.1 / 16.0, p = 16 12.9 / 16.1, p = 64 16.3 / 17.5, p = 100 (the
// vignette's example) 26.6 / 34.1;  n = 1e6: p = 16 48.5 / 18.4, p = 64 57.6 / 34.5 (tools/bench_logit_route_small_p.py).
bool logit_slab_preferred(int64_t n, int p) {
    if (!slab_shape(p).rt) return false;
    return p >= 128 || n <= 100000;
}

size_t logit_slab_doubles(int64_t n, int p) {
    const int rt = logit_slab_rows(p);
    if (!rt) return 0;
    return (size_t)((n + rt - 1) / rt) * rt * p;
}

void logit_slab_relayout(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, double *slabs) {
    const int rt = logit_slab_rows(p);
    if (!rt) fail(OEMB200_EINVAL, "slab route does not apply to p = %d", p);
    if (n >= (1ll << 31) * RL_ROWS) fail(OEMB200_EUNSUPPORTED, "slab re-layout: too many rows");
    dim3 grid((unsigned)((n + RL_ROWS - 1) / RL_ROWS), (unsigned)((p + RL_COLS - 1) / RL_COLS));
    slab_relayout_kernel<<<grid, 256, 0, cx.stream>>>(X, n, p, ld, rt, slabs);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

// grad_out[0] = sum r, grad_out[1 + j] = sum_i x_ij r_i (device, p + 1 doubles); b0 is read from device memory
void logit_slab_launch(Ctx &cx, const double *slabs, int64_t n, int p, const double *b, const double *b0_dev,
                       const double *y, double *prob, double *w, double *grad_out, const int *skip, unsigned long long *t_clock) {
    const SlabShape sh = slab_shape(p);
    if (!sh.rt) fail(OEMB200_EINVAL, "slab route does not apply to p = %d", p);
    const int rt = sh.rt;
    void *kern = nullptr;
#define LS_PICK(R, N, T) if (rt == R && sh.nc == N && sh.threads == T) kern = (void *)logit_slab_kernel<R, N, T>
    LS_PICK(4, 3, 512); LS_PICK(4, 4, 512);
    LS_PICK(8, 1, 256); LS_PICK(8, 2, 256); LS_PICK(4, 3, 256); LS_PICK(4, 4, 256);
#undef LS_PICK
    if (!kern) fail(OEMB200_EINVAL, "slab route: no kernel for p = %d", p);
    const int warps = sh.threads / 32;
    const size_t stage_stride = ((size_t)rt * p + 15) / 16 * 16;                 // doubles; keeps stages 128-byte aligned
    const size_t smem = LS_STAGES * stage_stride * 8 + (2 * LS_STAGES + 2) * 8 + ((size_t)warps * rt + rt) * 8;
    if (smem > cx.smem_optin) fail(OEMB200_EUNSUPPORTED, "slab route: %zu bytes of shared memory for p = %d", smem, p);
    OEM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t ntiles = (n + rt - 1) / rt;
    const int grid = (int)std::min<int64_t>(ntiles, (int64_t)cx.num_sms * sh.ctas);
    DBuf<double> partial((size_t)grid * (p + 1));       // every CTA writes its whole row
    long long nn = n;
    void *args[] = {(void *)&slabs, &nn, &p, (void *)&stage_stride, (void *)&b, (void *)&b0_dev, (void *)&y, &prob, &w, &partial.p,
                    (void *)&skip, (void *)&t_clock};
    OEM_CUDA(cudaLaunchKernel(kern, dim3(grid), dim3(sh.threads), args, smem, cx.stream));
    ls_sum_partials_kernel<<<(p + 1 + 31) / 32, 256, 0, cx.stream>>>(partial.p, grid, p + 1, grad_out, skip, t_clock);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 2;
    cx.st.xb_launches += 1;
    cx.st.data_passes += 1;
}

// ---------------------------------------------------------------------------------------------
// Fused multi-model pass of binomial cross-validation: ONE sweep of the slabs serves up to MK logistic models that share X
// but not their rows.  Model g (g = m0 + m) uses the rows whose fold is neither 0 (padding) nor g, so model 0 is the
// full-data fit and model k leaves fold k out; for each one the pass forms grad_g = [sum r, X' r] with
// r_i = y_i - sigma(b0_g + x_i . b_g) on its rows and 0 elsewhere.
//
// Layout: one 512-thread CTA per SM, 4-row slabs in a 2-stage ring.  Thread t owns the columns j = t, t + 512, ... (NC of
// them) for the whole pass, as in logit_slab_kernel, but the per-model state no longer fits in registers next to the slab:
//   the MK coefficient vectors live in shared memory (MK x p, read conflict-free by consecutive columns),
//   the MK x NC gradient accumulators stay in registers (at most 64 doubles per thread),
//   eta of every (row, model) is a per-model multi-value butterfly + a fixed-order sum over the warps, as in the single pass.
// Per slab and model the work is 2 NC RT FMAs per thread against one RT-value butterfly, so at p = 1000 and 11 models the
// pass is bound by the FP64 pipe and the shuffles, not by HBM.  A model whose `conv` flag is set (its IRLS loop has
// converged for this lambda) takes no part: no arithmetic, and its gradient row is left untouched.
// ---------------------------------------------------------------------------------------------
constexpr int LF_THREADS = 512, LF_RT = 4, LF_STAGES = 2;

template <int NC, int MK>
__global__ void __launch_bounds__(LF_THREADS, 1)
logit_fold_kernel(const double *__restrict__ slabs, long long n, int p, size_t stage_stride, const double *__restrict__ B,
                  const double *__restrict__ b0, int m0, int nm, const double *__restrict__ y, const int *__restrict__ fold,
                  const int *__restrict__ conv, double *__restrict__ prob0, double *__restrict__ partial) {
    constexpr int RT = LF_RT, WARPS = LF_THREADS / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *stages = reinterpret_cast<double *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + LF_STAGES * stage_stride * 8);
    uint64_t *empty = full + LF_STAGES;
    double *bsm = reinterpret_cast<double *>(empty + LF_STAGES);          // [MK][p]
    double *wsum = bsm + (size_t)MK * p;                                  // [WARPS][MK][RT]
    double *rsm = wsum + WARPS * MK * RT;                                 // [MK][RT]
    double *b0s = rsm + MK * RT;                                          // [MK]
    __shared__ int act[MK];
    __shared__ int nact;

    const long long ntiles = (n + RT - 1) / RT;
    const long long mine = ntiles > blockIdx.x ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, t = threadIdx.x;
    const uint32_t tile_bytes = (uint32_t)RT * (uint32_t)p * 8u;

    if (t == 0) {
        int c = 0;
        for (int m = 0; m < MK; ++m) {
            act[m] = m < nm && !(conv && conv[m0 + m]);
            c += act[m];
        }
        nact = c;
        for (int s = 0; s < LF_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], WARPS); }
        mbar_fence_init();
    }
    for (int e = t; e < nm * p; e += LF_THREADS) bsm[e] = B[(size_t)m0 * p + e];
    if (t < nm) b0s[t] = b0[m0 + t];
    __syncthreads();
    if (nact == 0) return;

    uint64_t pol = 0;
    const uint32_t pair_bytes = (uint32_t)p * 16u;
    auto issue = [&](long long k) {
        const int s = (int)(k % LF_STAGES);
        const double *src = slabs + (size_t)(blockIdx.x + k * gridDim.x) * RT * p;
        double *dst = stages + (size_t)s * stage_stride;
        mbar_arrive_expect_tx(&full[s], tile_bytes);
#pragma unroll
        for (int kk = 0; kk < RT / 2; ++kk)
            bulk_load(dst + (size_t)kk * 2 * p, src + (size_t)kk * 2 * p, pair_bytes, &full[s], pol);
    };
    if (t == 0) {
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
        for (long long k = 0; k < LF_STAGES && k < mine; ++k) issue(k);
    }

    double gacc[MK][NC];
#pragma unroll
    for (int m = 0; m < MK; ++m)
#pragma unroll
        for (int c = 0; c < NC; ++c) gacc[m][c] = 0.0;
    double rsum = 0.0;                       // threads t < MK: sum r of model t

    for (long long k = 0; k < mine; ++k) {
        const int s = (int)(k % LF_STAGES);
        const uint32_t ph = (uint32_t)((k / LF_STAGES) & 1);
        mbar_wait(&full[s], ph);
        const double2 *tile = reinterpret_cast<const double2 *>(stages + (size_t)s * stage_stride);
        double x[NC][RT];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const int j = t + c * LF_THREADS;
#pragma unroll
            for (int kk = 0; kk < RT / 2; ++kk) {
                const double2 v = j < p ? tile[(size_t)kk * p + j] : make_double2(0.0, 0.0);
                x[c][2 * kk] = v.x; x[c][2 * kk + 1] = v.y;
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (t == 0 && k + LF_STAGES < mine) {
            mbar_wait(&empty[s], ph);
            issue(k + LF_STAGES);
        }

#pragma unroll
        for (int m = 0; m < MK; ++m) {
            if (!act[m]) continue;
            double acc[RT];
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = 0.0;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const int j = t + c * LF_THREADS;
                const double bj = j < p ? bsm[(size_t)m * p + j] : 0.0;
#pragma unroll
                for (int i = 0; i < RT; ++i) acc[i] = fma(x[c][i], bj, acc[i]);
            }
            // RT = 4 row sums over the 32 lanes: two halving steps, then three full steps; lane l ends with row l >> 3
            {
                const bool up16 = (lane & 16) != 0;
                acc[0] = (up16 ? acc[2] : acc[0]) + __shfl_xor_sync(0xffffffffu, up16 ? acc[0] : acc[2], 16);
                acc[1] = (up16 ? acc[3] : acc[1]) + __shfl_xor_sync(0xffffffffu, up16 ? acc[1] : acc[3], 16);
                const bool up8 = (lane & 8) != 0;
                acc[0] = (up8 ? acc[1] : acc[0]) + __shfl_xor_sync(0xffffffffu, up8 ? acc[0] : acc[1], 8);
                acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 4);
                acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 2);
                acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 1);
            }
            if ((lane & 7) == 0) wsum[(warp * MK + m) * RT + (lane >> 3)] = acc[0];
        }
        __syncthreads();
        const long long row0 = (blockIdx.x + k * gridDim.x) * RT;
        if (t < MK * RT) {
            const int m = t / RT, i = t - m * RT;
            if (act[m]) {
                double e = b0s[m];
#pragma unroll
                for (int w = 0; w < WARPS; ++w) e += wsum[(w * MK + m) * RT + i];
                const long long row = row0 + i;
                double r = 0.0;
                if (row < n) {
                    const int f = fold[row];
                    if (f != 0 && f != m0 + m) {
                        const double pr = 1.0 / (1.0 + exp(-e));
                        r = y[row] - pr;
                        if (prob0 && m0 + m == 0) prob0[row] = pr;
                    }
                }
                rsm[m * RT + i] = r;
            }
        }
        __syncthreads();
#pragma unroll
        for (int m = 0; m < MK; ++m) {
            if (!act[m]) continue;
            double r[RT];
#pragma unroll
            for (int i = 0; i < RT; ++i) r[i] = rsm[m * RT + i];
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                double tt = x[c][0] * r[0];
#pragma unroll
                for (int i = 1; i < RT; ++i) tt = fma(x[c][i], r[i], tt);
                gacc[m][c] += tt;
            }
        }
        if (t < MK && act[t]) {
            double tt = rsm[t * RT];
#pragma unroll
            for (int i = 1; i < RT; ++i) tt += rsm[t * RT + i];
            rsum += tt;
        }
    }
    double *out = partial + (size_t)blockIdx.x * MK * (p + 1);
#pragma unroll
    for (int m = 0; m < MK; ++m) {
        if (!act[m]) continue;
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const int j = t + c * LF_THREADS;
            if (j < p) out[(size_t)m * (p + 1) + 1 + j] = gacc[m][c];
        }
    }
    if (t < MK && act[t]) out[(size_t)t * (p + 1)] = rsum;
}

// out[(m0 + m) (p + 1) + e] = sum over the CTAs of partial[c][m][e], in CTA order (same order as ls_sum_partials_kernel);
// rows of converged models are left untouched
__global__ void __launch_bounds__(256) lf_sum_partials_kernel(const double *__restrict__ partial, int nparts, int mk, int p,
                                                              int m0, int nm, const int *__restrict__ conv, double *__restrict__ out) {
    __shared__ double sm[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int width = nm * (p + 1);
    const int k = blockIdx.x * 32 + tx;
    const int m = k / (p + 1);
    const bool live = k < width && !(conv && conv[m0 + m]);
    double s = 0.0;
    if (live)
        for (int c = ty; c < nparts; c += 8) s += partial[(size_t)c * mk * (p + 1) + k];
    sm[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && live) {
        double t = sm[0][tx];
#pragma unroll
        for (int r = 1; r < 8; ++r) t += sm[r][tx];
        out[(size_t)m0 * (p + 1) + k] = t;
    }
}

// Models per sweep for a given p: the MK x NC accumulators must stay within 64 doubles per thread (128 registers is the
// ceiling of a 512-thread CTA) and MK coefficient vectors must fit next to the 2-stage ring in shared memory.
static int logit_fold_nc(int p) { return (p + LF_THREADS - 1) / LF_THREADS; }
int logit_fold_models(int p) {
    if (p < 8 || p > 2048) return 0;
    static const int mk[4] = {16, 16, 8, 4};
    return mk[logit_fold_nc(p) - 1];
}

size_t logit_fold_doubles(int64_t n, int p) { return (size_t)((n + LF_RT - 1) / LF_RT) * LF_RT * p; }

void logit_fold_relayout(Ctx &cx, const double *X, int64_t n, int p, int64_t ld, double *slabs) {
    if (!logit_fold_models(p)) fail(OEMB200_EINVAL, "fused fold pass does not apply to p = %d", p);
    if (n >= (1ll << 31) * RL_ROWS) fail(OEMB200_EUNSUPPORTED, "slab re-layout: too many rows");
    dim3 grid((unsigned)((n + RL_ROWS - 1) / RL_ROWS), (unsigned)((p + RL_COLS - 1) / RL_COLS));
    slab_relayout_kernel<<<grid, 256, 0, cx.stream>>>(X, n, p, ld, LF_RT, slabs);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

int logit_fold_launch(Ctx &cx, const double *slabs, int64_t n, int p, const double *B, const double *b0, const double *y,
                      const int *fold, int M, const int *conv, const std::vector<char> *active, double *prob0, double *grad) {
    const int MK = logit_fold_models(p), NC = logit_fold_nc(p);
    if (!MK) fail(OEMB200_EINVAL, "fused fold pass does not apply to p = %d", p);
    void *kern = nullptr;
    if (NC == 1) kern = (void *)logit_fold_kernel<1, 16>;
    else if (NC == 2) kern = (void *)logit_fold_kernel<2, 16>;
    else if (NC == 3) kern = (void *)logit_fold_kernel<3, 8>;
    else kern = (void *)logit_fold_kernel<4, 4>;
    const size_t stage_stride = ((size_t)LF_RT * p + 15) / 16 * 16;
    const size_t smem = LF_STAGES * stage_stride * 8 + 2 * LF_STAGES * 8 +
                        ((size_t)MK * p + (size_t)(LF_THREADS / 32) * MK * LF_RT + (size_t)MK * LF_RT + MK) * 8;
    if (smem > cx.smem_optin) fail(OEMB200_EUNSUPPORTED, "fused fold pass: %zu bytes of shared memory for p = %d", smem, p);
    OEM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t ntiles = (n + LF_RT - 1) / LF_RT;
    const int grid = (int)std::min<int64_t>(ntiles, (int64_t)cx.num_sms);
    DBuf<double> partial((size_t)grid * MK * (p + 1));
    long long nn = n;
    int sweeps = 0;
    for (int m0 = 0; m0 < M; m0 += MK) {
        int nm = std::min(MK, M - m0);
        if (active) {
            bool any = false;
            for (int m = m0; m < m0 + nm; ++m) any = any || (*active)[m];
            if (!any) continue;
        }
        void *args[] = {(void *)&slabs, &nn, &p, (void *)&stage_stride, (void *)&B, (void *)&b0, &m0, &nm, (void *)&y,
                        (void *)&fold, (void *)&conv, &prob0, &partial.p};
        OEM_CUDA(cudaLaunchKernel(kern, dim3(grid), dim3(LF_THREADS), args, smem, cx.stream));
        lf_sum_partials_kernel<<<(nm * (p + 1) + 31) / 32, 256, 0, cx.stream>>>(partial.p, grid, MK, p, m0, nm, conv, grad);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 2;
        cx.st.xb_launches += 1;
        cx.st.data_passes += 1;
        ++sweeps;
    }
    return sweeps;
}

}  // namespace oemb200
