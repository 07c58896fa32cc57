// path_kernel.cu -- everything after the Gram, in ONE persistent kernel:
//   * top eigenvalue of XX by Lanczos  -> d = factor * lambda_max      (stands in for the
//     Spectra::SymEigsSolver call sites: src/oem_dense.h:485-498, oem_xtx.h:357-369,
//     oem_xval_dense.h:770-782,837-843, oem_logistic_dense.h:501-514, oem_big.h:546-559)
//   * A = d I - XX                                                     (src/oem_dense.h:501-505)
//   * for every chain (Gram x penalty), the warm-started lambda path of
//       beta <- prox_penalty(A beta + XY)            oemBase::solve  src/oem_base.h:90-110
//       next_u                                       src/oem_dense.h:508-513
//       next_beta + thresholding family              src/oem_dense.h:76-315, 527-629
//       Nesterov option                              src/oem_dense.h:633-651
//       stopRule                                     src/utils.cpp:537-549
//
// Design.  The CTAs are split into one TEAM per Gram (1 team for oem / oem.xtx / big.oem / the
// logistic inner loop, nfolds+1 teams for xval.oem).  A team member owns a slice of columns of A
// (A is symmetric, so a column slice is a row slice) which it keeps in SHARED MEMORY for the whole
// path whenever it fits (148 x ~200 KB covers q = 1001 with room to spare); otherwise the slice
// is streamed from L2.  Each OEM iteration is
//     u[slice] = A[:,slice]' beta + XY[slice]   for all of the team's chains at once: a skinny GEMM
//                                               (columns x chains x q) on the FP64 TENSOR pipe
//                                               (DMMA.8x8x4, A fragments from shared memory)
//     coordinate-wise penalties: the member that owns coordinate j applies the prox and the stop rule in the
//     mat-vec epilogue and publishes the NEXT BETA; group penalties / Nesterov publish u and every member
//     applies the prox redundantly to the full vector
//     ONE exchange + ONE team barrier
// All members execute bit-identical arithmetic on identical inputs, so they take the same
// convergence decisions without any further communication.  Reductions use fixed orders.
// Small problems (q <= 256, coordinate-wise penalties) take the register-resident variant further down
// (oem_path_reg_kernel): there a DMMA would waste 4/8..7/8 of its B operand on 1..4 chains, and the FP64
// CUDA-core pipe (measured: same rate as DMMA on B200) runs the product from registers.  The same holds at the other
// end: in the global mode with one 8-column atom per member and <= 4 chains (q ~ 450..1184: oem / big.oem / the sparse
// entry / the logistic inner loop at p = 1000) the members keep their XX slice in registers and run matvec_reg
// (oem_path_kernel<MODE_GLOBAL, RPT>); the DMMA mat-vec serves everything else.
// Three exchange modes, chosen on the host from q:
//     MODE_SINGLE   the whole A fits one CTA: u goes straight into shared memory, __syncthreads only
//     MODE_CLUSTER  A fits the shared memory of a thread-block cluster (<= 8 CTAs): every member stores
//                   its u slice into all members' shared memory (DSMEM, st.shared::cluster) and the
//                   barrier is the hardware cluster barrier
//     MODE_GLOBAL   larger q: u goes through an L2-resident buffer, barrier = one atomic counter per team, then ONE batch of
//                   loads fetches every chain's published vector and the members' violation masks
// Everything an iteration needs besides u (chain descriptors, lambdas, penalty factors, XY, group
// tables) is copied to shared memory once: the gpu-scope synchronisation of the barrier invalidates
// L1, so any per-iteration global read would be an L2 round trip on the critical path.  The prox
// and the stop rule avoid FP64-pipe work for the (many) coordinates that are and stay zero.
#include <algorithm>
#include <cstdlib>
#include <vector>
#include "runtime.h"

namespace oemb200 {

constexpr int PK_THREADS = 256;
constexpr int PK_WARPS = PK_THREADS / 32;
constexpr int LZ_MAX = 512;       // Lanczos step cap
constexpr int PK_MAXCT = 32;      // chains per team cap
constexpr int PK_PART = 8;        // partial 8x8 tiles kept in shared memory for the split-K mat-vec (<= 1 per warp)

struct ChainDev {
    int gram, penalty, nlam, lam_off;
    double alpha, gamma, tau;
    int out_off, pad;
};

enum { MODE_SINGLE = 0, MODE_CLUSTER = 1, MODE_GLOBAL = 2 };

struct PathScratch {
    std::vector<unsigned char> key;      // what the tables below were built from
    DBuf<ChainDev> chains;
    DBuf<int> tptr, tidx;
    DBuf<double> ubuf, A;
    DBuf<unsigned> bar;                  // [ngram barrier words | ngram x 2 x team violation flags]
    size_t nflags = 0;
};
PathScratch *path_scratch_create() { return new PathScratch(); }
void path_scratch_destroy(PathScratch *s) { delete s; }

struct PathArgs {
    int q, qs, ngram, team_size, cpc, cpc_pad, max_ct, Lmax, maxit, accelerate, compute_eig, a_in_smem, ngroups, mode;
    int ngidx, pad1;
    double tol, eig_factor, eig_tol;
    const double *XX, *XY;
    double *d, *Abuf;
    const ChainDev *chains;
    const int *team_ptr, *team_idx;   // CSR: chains of each team
    const double *lambdas, *pen_fact;
    const int *unique_groups, *grp_ptr, *grp_idx, *grp_cover;
    const double *group_weights, *post_scale, *beta_init;
    double *beta_out;
    int *niter_out, *lanczos_steps;
    double *ubuf;            // ngram x 2 x max_ct x q
    unsigned *barriers;      // ngram counters, zero-initialised
    int *gflags;             // ngram x 2 x team_size violation masks (global mode)
    long long *prof;         // optional (debug): cycle counters of CTA 0 / thread 0
    const int *skip;         // optional: the whole launch is a no-op when *skip != 0 (speculatively enqueued IRLS iterations)
    // register mode only: form XY = XX beta_init + grad in the prologue (PathProblem::xy_grad)
    const double *xy_grad, *xy_cinv;
    double xy_n;
    int xy_icpt, pad2;
    double *xy_out;
    unsigned long long *t_acc;   // optional: += duration of the launch in ns (CTA 0, device-side phase clock)
    // IRLS epilogue (PathProblem::irls_*)
    int *irls_conv;
    volatile int *irls_host_flag;
    long long *irls_iters_total;
    double irls_tol;
    const double *irls_cinv;
    int irls_p, irls_icpt;
    double *irls_b, *irls_b0;
};

__device__ __forceinline__ double pk_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// deterministic block-wide sum, result returned to every thread
__device__ __forceinline__ double block_sum(double v, double *red) {
    v = pk_warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < PK_WARPS; ++w) s += red[w];
    __syncthreads();
    return s;
}

// |x| > thr for thr >= 0, on the integer pipe (IEEE-754 ordering of non-negative doubles)
__device__ __forceinline__ bool abs_gt(double x, double thr) {
    return (__double_as_longlong(x) & 0x7fffffffffffffffLL) > __double_as_longlong(thr);
}

// x / d given r = 1/d (correctly rounded): q0 = x r, residual by FMA, one correction (Markstein).  Gives the
// IEEE quotient with 3 dependent FP64 operations instead of the ~30 of a full division -- on this part the
// FP64 CUDA-core pipe is slow enough that the divisions of the few non-zero coefficients were the critical
// path of every iteration.
__device__ __forceinline__ double div_r(double x, double d, double r) {
    const double q0 = x * r;
    const double e = fma(-d, q0, x);
    return fma(e, r, q0);
}
// ---- thresholding family (coordinate-wise), operation order as in src/oem_dense.h:76-149 ----
__device__ __forceinline__ double st_lasso(double v, double pen, double d) {
    if (v > pen) return (v - pen) / d;
    if (v < -pen) return (v + pen) / d;
    return 0.0;
}
__device__ __forceinline__ double st_mcp(double v, double pen, double d, double gamma) {
    const double gammad = gamma * d, dmg = d - 1.0 / gamma;
    if (fabs(v) > gammad * pen) return v / d;
    if (v > pen) return (v - pen) / dmg;
    if (v < -pen) return (v + pen) / dmg;
    return 0.0;
}
__device__ __forceinline__ double st_scad(double v, double pen, double d, double gamma) {
    const double gammad = gamma * d, gm1d = (gamma - 1.0) * d;
    if (fabs(v) > gammad * pen) return v / d;
    if (fabs(v) > (d + 1.0) * pen) {
        const double gp = (gamma - 1.0) * v, gpen = gamma * pen;
        if (gp > gpen) return (gp - gpen) / (gm1d - 1.0);
        if (gp < -gpen) return (gp + gpen) / (gm1d - 1.0);
        return 0.0;
    }
    if (v > pen) return (v - pen) / d;
    if (v < -pen) return (v + pen) / d;
    return 0.0;
}
// group factors: src/oem_dense.h:151-191
__device__ __forceinline__ double scad_norm(double b, double pen, double d, double gamma) {
    const double gammad = gamma * d, gm1d = (gamma - 1.0) * d;
    if (fabs(b) > gammad * pen) return 1.0;
    if (fabs(b) > (d + 1.0) * pen) {
        const double gp = gamma - 1.0, gpen = gamma * pen / b;
        if (gp > gpen) return d * (gp - gpen) / (gm1d - 1.0);
        if (gp < -gpen) return d * (gp + gpen) / (gm1d - 1.0);
        return 0.0;
    }
    if (b > pen) return 1.0 - pen / b;
    if (b < -pen) return 1.0 + pen / b;
    return 0.0;
}
__device__ __forceinline__ double mcp_norm(double b, double pen, double d, double gamma) {
    const double gammad = gamma * d, dmg = d - 1.0 / gamma;
    if (fabs(b) > gammad * pen) return 1.0;
    if (b > pen) return d * (1.0 - pen / b) / dmg;
    if (b < -pen) return d * (1.0 + pen / b) / dmg;
    return 0.0;
}

// shared-memory copies of the per-call tables
struct SmemTabs {
    const double *pf, *gw;
    const int *grp_ptr, *grp_unique, *grp_idx, *cover;
    int ngroups;
};

// prox of one chain, in place on v[0..q): on entry v = u, on exit v = next beta.
// Dispatch: src/oem_dense.h:527-629.
__device__ __noinline__ void prox_inplace(int q, const SmemTabs &tb, int pen, double alpha, double gamma, double tau, double lambda,
                             double d, double *v) {
    double denom = d + (1.0 - alpha) * lambda;
    double lam = lambda * alpha;
    if (pen == OEMB200_PEN_SCAD_NET && alpha == 0.0) { lam = 0.0; denom = d + lambda; }
    const bool net = (pen == OEMB200_PEN_ENET || pen == OEMB200_PEN_SCAD_NET || pen == OEMB200_PEN_MCP_NET ||
                      pen == OEMB200_PEN_GRP_LASSO_NET || pen == OEMB200_PEN_GRP_MCP_NET ||
                      pen == OEMB200_PEN_GRP_SCAD_NET);
    const double lp = net ? lam : lambda, dp = net ? denom : d;
    if (pen < OEMB200_PEN_GRP_LASSO) {
        if (pen == OEMB200_PEN_OLS) {
            for (int j = threadIdx.x; j < q; j += PK_THREADS) v[j] = v[j] / d;
        } else {
            // every rule returns 0 when |u| <= pen * min(1, gamma d) (lasso / elastic.net: |u| <= pen); that
            // test runs on the integer pipe, so coordinates that stay zero cost no FP64 work beyond one multiply
            const bool ncv = (pen == OEMB200_PEN_SCAD || pen == OEMB200_PEN_SCAD_NET || pen == OEMB200_PEN_MCP ||
                              pen == OEMB200_PEN_MCP_NET);
            const double zf = ncv ? fmin(1.0, gamma * dp) : 1.0;
            const bool is_scad = (pen == OEMB200_PEN_SCAD || pen == OEMB200_PEN_SCAD_NET);
            for (int j = threadIdx.x; j < q; j += PK_THREADS) {
                const double u = v[j];
                const double tp = tb.pf[j] * lp;
                double r = 0.0;
                if (abs_gt(u, tp * zf)) {
                    if (!ncv) r = st_lasso(u, tp, dp);
                    else if (is_scad) r = st_scad(u, tp, dp, gamma);
                    else r = st_mcp(u, tp, dp, gamma);
                }
                v[j] = r;
            }
        }
        __syncthreads();
        return;
    }
    double glam = lp, gd = dp;
    int kind = 0;
    if (pen == OEMB200_PEN_GRP_MCP || pen == OEMB200_PEN_GRP_MCP_NET) kind = 1;
    if (pen == OEMB200_PEN_GRP_SCAD || pen == OEMB200_PEN_GRP_SCAD_NET) kind = 2;
    if (pen == OEMB200_PEN_SPARSE_GRP_LASSO) {
        const double lam_l1 = tau * lambda;
        glam = (1.0 - tau) * lambda;
        gd = d;
        for (int j = threadIdx.x; j < q; j += PK_THREADS) v[j] = st_lasso(v[j], tb.pf[j] * lam_l1, 1.0);
        __syncthreads();
    }
    // one thread per group: sequential norm in member order like block_soft_threshold (src/oem_dense.h:193-315)
    for (int g = threadIdx.x; g < tb.ngroups; g += PK_THREADS) {
        const int b0 = tb.grp_ptr[g], b1 = tb.grp_ptr[g + 1];
        double tf;
        if (tb.grp_unique[g] == 0) tf = 1.0;
        else {
            double nrm = 0.0;
            for (int k = b0; k < b1; ++k) { const double x = v[tb.grp_idx[k]]; nrm += x * x; }
            nrm = sqrt(nrm);
            const double gw = tb.gw[g];
            if (kind == 0) { const double t = 1.0 - glam * gw / nrm; tf = (0.0 < t) ? t : 0.0; }
            else if (kind == 1) tf = mcp_norm(nrm, glam * gw, gd, gamma);
            else tf = scad_norm(nrm, glam * gw, gd, gamma);
        }
        for (int k = b0; k < b1; ++k) {
            const int c = tb.grp_idx[k];
            v[c] = (tf != 0.0) ? v[c] * tf / gd : 0.0;
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < q; j += PK_THREADS)
        if (!tb.cover[j]) v[j] = 0.0;      // variables in no listed group stay 0 (res.setZero())
    __syncthreads();
}

// Largest eigenvalue of the k x k symmetric tridiagonal (al, be) by 256-way multisection (one trial point
// per thread of the CTA) on the Sturm sign pattern (division-free scaled determinant recurrence), then the
// backward eigenvector recurrence for the residual bound be[k-1] * |s_k| / ||s||.
// out[0] = theta, out[1] = |s_k| / ||s||, out[2] = lower bracket;  ibe[i] = 1 / be[i].  Called by all threads.
// `rounds` multisection rounds (each narrows the bracket 257-fold): 9 reach the last bit from any Gershgorin bracket, 3 are
// enough for the convergence checks on the way.
__device__ __noinline__ void tridiag_top(const double *al, const double *be, const double *ibe, int k, double lo_hint, double *out,
                            double *red, int *ibuf, int rounds) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double lo = -1e300, hi = -1e300;
    for (int i = threadIdx.x; i < k; i += PK_THREADS) {
        const double r = (i > 0 ? fabs(be[i - 1]) : 0.0) + (i + 1 < k ? fabs(be[i]) : 0.0);
        lo = fmax(lo, al[i]);
        hi = fmax(hi, al[i] + r);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmax(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) { red[warp] = lo; red[8 + warp] = hi; }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < PK_WARPS; ++w) { lo = fmax(lo, red[w]); hi = fmax(hi, red[8 + w]); }
    lo = fmax(lo, lo_hint);           // Ritz values grow with k (interlacing)
    hi += 1e-14 * fabs(hi) + 1e-300;
    for (int round = 0; round < rounds; ++round) {
        const double w = hi - lo;
        if (!(w > 2e-16 * fmax(fabs(hi), fabs(lo)))) break;      // uniform: lo / hi are identical in all threads
        const double x = lo + w * (double)(threadIdx.x + 1) / (double)(PK_THREADS + 1);
        // all eigenvalues < x  <=>  the leading principal minors p_i of (T - x I) alternate in sign, p_1 < 0
        bool all_below = true;
        double pm = 1.0, pc = al[0] - x;
        if (!(pc < 0.0)) all_below = false;
        for (int i = 1; i < k && all_below; ++i) {
            const double b = be[i - 1];
            const double pn = (al[i] - x) * pc - (b * b) * pm;
            if (!(pn * pc < 0.0)) all_below = false;
            pm = pc; pc = pn;
            if (abs_gt(pc, 1e150)) { pc *= 1e-150; pm *= 1e-150; }
            else if (!abs_gt(pc, 1e-150)) { pc *= 1e150; pm *= 1e150; }
        }
        const unsigned m = __ballot_sync(0xffffffffu, all_below);
        if (lane == 0) ibuf[warp] = m ? warp * 32 + __ffs(m) - 1 : PK_THREADS;
        __syncthreads();
        int f = PK_THREADS;
#pragma unroll
        for (int ww = 0; ww < PK_WARPS; ++ww) f = min(f, ibuf[ww]);
        __syncthreads();
        // trial point of thread i is lo + w (i+1)/(T+1): the eigenvalue lies in (x_{f-1}, x_f]
        const double nlo = f > 0 ? lo + w * (double)f / (double)(PK_THREADS + 1) : lo;
        if (f < PK_THREADS) hi = lo + w * (double)(f + 1) / (double)(PK_THREADS + 1);
        lo = nlo;
    }
    if (threadIdx.x == 0) {
        const double theta = 0.5 * (lo + hi);
        // backward recurrence from s_k = 1 (the growing, hence stable, direction)
        double s_next = 0.0, s_cur = 1.0, nrm2 = 1.0, s_last = 1.0;   // s_last = s_k in current units
        for (int i = k - 1; i >= 1; --i) {
            // row i: be[i-1] s_{i-1} + (al[i]-theta) s_i + be[i] s_{i+1} = 0
            const double bi = (i + 1 < k) ? be[i] : 0.0;
            const double s_prev = -((al[i] - theta) * s_cur + bi * s_next) * ibe[i - 1];
            s_next = s_cur;
            s_cur = s_prev;
            nrm2 += s_cur * s_cur;
            if (abs_gt(s_cur, 1e120)) { s_cur *= 1e-120; s_next *= 1e-120; nrm2 *= 1e-240; s_last *= 1e-120; }
        }
        out[0] = theta;
        out[1] = s_last / sqrt(nrm2);   // |last eigenvector component| of the unit Ritz vector
        out[2] = lo;
    }
}

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_cluster_f64(double *local_smem_ptr, unsigned cta_rank, double v) {
    unsigned remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local_smem_ptr)), "r"(cta_rank));
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(remote), "d"(v) : "memory");
}
// asynchronous DSMEM stores that complete a transaction count on the DESTINATION CTA's mbarrier: the receiver waits on its
// own barrier for the expected bytes, so the sender needs neither a fence nor a cluster-wide barrier round trip
__device__ __forceinline__ unsigned map_cluster(const void *local_smem_ptr, unsigned cta_rank) {
    unsigned remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local_smem_ptr)), "r"(cta_rank));
    return remote;
}
__device__ __forceinline__ void st_async_f64(unsigned remote_addr, double v, unsigned remote_mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                 ::"r"(remote_addr), "l"(__double_as_longlong(v)), "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ void st_async_u32(unsigned remote_addr, unsigned v, unsigned remote_mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                 ::"r"(remote_addr), "r"(v), "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    const uint32_t a = smem_u32(bar);
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(a), "r"(parity)
            : "memory");
    } while (!ok);
}


// sums acc[c][*] over the 32 lanes for NCT chains at once (stage-major so the chains' shuffles overlap):
// on return tot[c] in lane l is the total of column l / (32 / CPW)
template <int NCT, int CPW>
__device__ __forceinline__ void reduce_cols(double (&acc)[NCT][CPW], double (&tot)[NCT], int lane) {
#pragma unroll
    for (int n = CPW, off = 16; n > 1; n >>= 1, off >>= 1) {
        const bool hi = (lane & off) != 0;
#pragma unroll
        for (int c = 0; c < NCT; ++c)
#pragma unroll
            for (int v = 0; v < n / 2; ++v) {
                const double keep = hi ? acc[c][v + n / 2] : acc[c][v];
                const double send = hi ? acc[c][v] : acc[c][v + n / 2];
                acc[c][v] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
    }
#pragma unroll
    for (int c = 0; c < NCT; ++c) tot[c] = acc[c][0];
#pragma unroll
    for (int off = 16 / CPW; off >= 1; off >>= 1)
#pragma unroll
        for (int c = 0; c < NCT; ++c) tot[c] += __shfl_xor_sync(0xffffffffu, tot[c], off);
}

// Coordinate-wise prox without divergent branches (the lanes of the finishing warp serve different penalties).  Everything
// that does not depend on u -- the thresholds of the region tests -- is computed BEFORE the sums arrive; afterwards the
// region tests run on the integer pipe (abs_gt), select ONE numerator / denominator pair, and a single Markstein division
// follows.  Same operations on the same operands as st_lasso / st_mcp / st_scad above with x / d taken as div_r(x, d, 1 / d)
// (v - copysign(pen, v) is v - pen
// for v > 0 and v + pen for v < 0; |x| > t for t >= 0 is the integer comparison of the bit patterns).
struct ProxPre {
    double tp, thr_big, thr_mid, gpen, gm1, dp, rdp, den2, rden2, tolpv, pv;
    int kind;
};
__device__ __forceinline__ double prox_select(const ProxPre &k, double u) {
    double num = u - copysign(k.tp, u), den = k.dp, rden = k.rdp;
    bool nz = abs_gt(u, k.tp);
    if (k.kind == 1) { den = k.den2; rden = k.rden2; }
    if (k.kind == 2 && abs_gt(u, k.thr_mid)) {
        const double gp = k.gm1 * u;
        num = gp - copysign(k.gpen, gp); den = k.den2; rden = k.rden2;
        nz = abs_gt(gp, k.gpen);
    }
    if (k.kind == 3 || ((k.kind == 1 || k.kind == 2) && abs_gt(u, k.thr_big))) { num = u; den = k.dp; rden = k.rdp; nz = true; }
    return nz ? div_r(num, den, rden) : 0.0;
}

// ---- mat-vec on the FP64 tensor pipe with the prox / stop rule fused into its epilogue ----
struct MvCtx {
    const double *Amine, *xy, *pf, *cpar, *gam;
    const int *kind;          // per chain: 0 lasso-type, 1 mcp, 2 scad, 3 ols
    double *part, *ub;
    int *violw;               // shared word: bit c set when chain c's stop rule is violated somewhere in my slice
    int q, qs, c0, c1, natm, max_ct, team_size;
    double tol;
    long long *prof;          // debug: cycle counters (CTA 0 only)
};

template <int MODE>
__device__ __forceinline__ void mv_publish(const MvCtx &m, double *dst_local, int par, int c, int j, double val) {
    double *dst = dst_local + (size_t)c * m.qs + j;
    if (MODE == MODE_SINGLE) *dst = val;
    else if (MODE == MODE_CLUSTER) {
        for (int r = 0; r < m.team_size; ++r) st_cluster_f64(dst, (unsigned)r, val);
    } else m.ub[((size_t)par * m.max_ct + c) * m.q + j] = val;
}

// Chains in `fastmask` get their coordinate-wise prox (src/oem_dense.h:527-629) and stop rule (src/utils.cpp:537-549)
// right here, on the one member that owns column j: the published value is then the NEXT BETA, not u.
__device__ __forceinline__ double mv_finish(const MvCtx &m, unsigned fastmask, const double *prev, int c, int j, double u, bool &viol) {
    if (!((fastmask >> c) & 1u)) return u;
    const double *cp = m.cpar + c * 8;
    const double gamma = m.gam[c];
    ProxPre k;                                   // everything but the last line is independent of u
    k.kind = m.kind[c];
    k.tp = m.pf[j] * cp[0]; k.dp = cp[1]; k.rdp = cp[4]; k.den2 = cp[6]; k.rden2 = cp[7];
    k.thr_big = cp[5] * k.tp; k.thr_mid = (k.dp + 1.0) * k.tp; k.gpen = gamma * k.tp; k.gm1 = gamma - 1.0;
    const double pv = prev[(size_t)c * m.qs + j];
    const double r = prox_select(k, u);
    if (__double_as_longlong(r) != __double_as_longlong(pv)) {      // identical bit patterns (0 -> 0) need no arithmetic
        const bool bc = abs_gt(r, 1e-13), bp = abs_gt(pv, 1e-13);
        if (bc != bp || (bc && abs_gt(r - pv, m.tol * fabs(pv)))) viol = true;                 // |(cur-prev)/prev| > tol
    }
    return r;
}

// out[c][j] = finish( sum_i S[i][j] vec_c[i] (+ xy[j]) ) for my columns j and nv vectors (vec = prev for the stop rule).
// D(8 columns x 8 vectors) += A(8 columns x 4 rows) * B(4 rows x 8 vectors) per DMMA; a work unit is one
// 8-column x 8-vector tile; with fewer than 8 units the K range is split across warps and the partial
// tiles are summed in fixed order through shared memory.
template <int MODE>
__device__ __noinline__ void matvec_dmma(const MvCtx &m, const double *vec, double *dst_local, int nv, const int *inactive,
                                         int add_xy, unsigned fastmask, int par) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int qs = m.qs;
    const int natn = (nv + 7) >> 3;
    const int units = m.natm * natn;
    const int ksplit = units >= PK_WARPS ? 1 : PK_WARPS / units;
    const int ktot = qs >> 2;                                   // k4 steps (zero padded)
    const int kper = (ktot + ksplit - 1) / ksplit;
    const int tasks = units * ksplit;
    const long long tm0 = m.prof ? clock64() : 0;
    for (int task = warp; task < tasks; task += PK_WARPS) {
        const int unit = task / ksplit, kp = task - unit * ksplit;
        const int am = unit % m.natm, an = unit / m.natm;
        const double *ap = m.Amine + (size_t)(am * 8 + g) * qs + t;
        const int cidx = an * 8 + g;
        const bool bvalid = cidx < nv;
        const double *bp = vec + (size_t)(bvalid ? cidx : 0) * qs + t;
        const int k0 = kp * kper, k1 = min(ktot, k0 + kper);
        double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0, c20 = 0.0, c21 = 0.0, c30 = 0.0, c31 = 0.0;
        int ks = k0;
#pragma unroll 1
        for (; ks + 4 <= k1; ks += 4) {
            const double a0 = ap[ks * 4], a1 = ap[ks * 4 + 4], a2 = ap[ks * 4 + 8], a3 = ap[ks * 4 + 12];
            const double b0 = bvalid ? bp[ks * 4] : 0.0, b1 = bvalid ? bp[ks * 4 + 4] : 0.0;
            const double b2 = bvalid ? bp[ks * 4 + 8] : 0.0, b3 = bvalid ? bp[ks * 4 + 12] : 0.0;
            dmma884(c00, c01, a0, b0);
            dmma884(c10, c11, a1, b1);
            dmma884(c20, c21, a2, b2);
            dmma884(c30, c31, a3, b3);
        }
#pragma unroll 1
        for (; ks < k1; ++ks) {
            const double a0 = ap[ks * 4];
            const double b0 = bvalid ? bp[ks * 4] : 0.0;
            dmma884(c00, c01, a0, b0);
        }
        const double r0 = (c00 + c10) + (c20 + c30), r1 = (c01 + c11) + (c21 + c31);
        // this lane holds column (am*8 + g) for vectors an*8 + 2t, 2t+1
        if (ksplit == 1) {
            const int j = m.c0 + am * 8 + g;
            const int cv = an * 8 + 2 * t;
            if (j < m.c1) {
                const double add = add_xy ? m.xy[j] : 0.0;
                if (cv < nv && !(inactive && inactive[cv])) {
                    bool viol = false;
                    mv_publish<MODE>(m, dst_local, par, cv, j, mv_finish(m, fastmask, vec, cv, j, r0 + add, viol));
                    if (viol) atomicOr(m.violw, 1 << cv);
                }
                if (cv + 1 < nv && !(inactive && inactive[cv + 1])) {
                    bool viol = false;
                    mv_publish<MODE>(m, dst_local, par, cv + 1, j, mv_finish(m, fastmask, vec, cv + 1, j, r1 + add, viol));
                    if (viol) atomicOr(m.violw, 1 << (cv + 1));
                }
            }
        } else {
            m.part[task * 64 + lane * 2] = r0;
            m.part[task * 64 + lane * 2 + 1] = r1;
        }
    }
    if (ksplit > 1) {
        const long long tm1 = m.prof ? clock64() : 0;
        __syncthreads();
        const long long tm2 = m.prof ? clock64() : 0;
        for (int e = threadIdx.x; e < units * 64; e += PK_THREADS) {
            const int unit = e >> 6, w = e & 63;
            const int ln = w >> 1, h = w & 1;
            double sacc = 0.0;
            for (int kp = 0; kp < ksplit; ++kp) sacc += m.part[(unit * ksplit + kp) * 64 + w];
            const int am = unit % m.natm, an = unit / m.natm;
            const int j = m.c0 + am * 8 + (ln >> 2);
            const int cv = an * 8 + 2 * (ln & 3) + h;
            if (j < m.c1 && cv < nv && !(inactive && inactive[cv])) {
                bool viol = false;
                mv_publish<MODE>(m, dst_local, par, cv, j, mv_finish(m, fastmask, vec, cv, j, sacc + (add_xy ? m.xy[j] : 0.0), viol));
                if (viol) atomicOr(m.violw, 1 << cv);
            }
        }
        if (m.prof && threadIdx.x == 0 && add_xy) {
            const long long tm3 = clock64();
            m.prof[13] += tm1 - tm0; m.prof[14] += tm2 - tm1; m.prof[15] += tm3 - tm2;
        }
    }
}

// ---- register-resident mat-vec of the global mode (8-column members, <= 4 chains, q <= 256 * RPT) ----
// At q ~ 1000 a member owns ONE 8-column atom and the team runs 1..3 chains: a DMMA would spend 5/8..7/8 of every
// instruction on padding vectors, its split-K partial tiles go through shared memory, and the measured mat-vec was
// 4.2 k cycles of an 11 k-cycle iteration (K loop 2.0 k: two warps per sub-partition queueing on the DMMA pipe with a
// dependent accumulator chain; reduce + prox + publish 2.2 k).  Here thread t keeps rows t, t + 256, ... of the 8 columns
// in registers for the whole launch (8 * RPT doubles), an iteration reads only the iterate from shared memory
// (conflict-free, NV * RPT loads), runs 8 * NV independent DFMA chains, reduces the 8 * NV sums with the multi-value
// butterfly (fixed order), and ONE warp finishes: fixed-order sum over the 8 warps, + XY, coordinate-wise prox, stop
// rule, publication of the next beta and of the member's violation mask.
template <int RPT, int NV>
__device__ __forceinline__ void matvec_reg(const double (&areg)[8][RPT], const MvCtx &m, const double *vec, int *inactive,
                                           int add_xy, unsigned fastmask, int par, int *gflag_slot) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long tm0 = m.prof ? clock64() : 0;
    double acc[NV][8];
#pragma unroll
    for (int c = 0; c < NV; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[c][j] = 0.0;
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
        const int i = threadIdx.x + r * PK_THREADS;
        if (i < m.qs) {
            double b[NV];
#pragma unroll
            for (int c = 0; c < NV; ++c) b[c] = vec[(size_t)c * m.qs + i];
#pragma unroll
            for (int c = 0; c < NV; ++c)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[c][j] = fma(areg[j][r], b[c], acc[c][j]);
        }
    }
    double tot[NV];
    const long long tm1 = m.prof ? clock64() : 0;
    reduce_cols<NV, 8>(acc, tot, lane);          // tot[c] = this warp's sum for column lane / 4, in all 4 lanes of the group
    {
        const int c = lane & 3;
        double v = tot[0];
#pragma unroll
        for (int cc = 1; cc < NV; ++cc) v = (c == cc) ? tot[cc] : v;
        if (c < NV) m.part[warp * 32 + lane] = v;
    }
    const long long tm2 = m.prof ? clock64() : 0;
    // the finishing warp fetches everything its epilogue needs besides the sums BEFORE the barrier
    const int fc = lane & 3, fj = m.c0 + (lane >> 2);
    const bool fin_lane = warp == 0 && fc < NV && fj < m.c1 && !(inactive && inactive[fc]);
    const bool fast = (fastmask >> fc) & 1u;
    ProxPre pk;
    double xyj = 0.0;
    double *pub = nullptr;                 // where this lane publishes (address arithmetic off the critical path)
    if (fin_lane) {
        pub = m.ub + ((size_t)par * m.max_ct + fc) * m.q + fj;
        if (fast) {
            const double *cp = m.cpar + fc * 8;
            const double gamma = m.gam[fc];
            pk.kind = m.kind[fc];
            pk.tp = m.pf[fj] * cp[0]; pk.dp = cp[1]; pk.rdp = cp[4]; pk.den2 = cp[6]; pk.rden2 = cp[7];
            pk.thr_big = cp[5] * pk.tp;               // gamma d t
            pk.thr_mid = (pk.dp + 1.0) * pk.tp;
            pk.gpen = gamma * pk.tp; pk.gm1 = gamma - 1.0;
            pk.pv = vec[(size_t)fc * m.qs + fj];
            pk.tolpv = m.tol * fabs(pk.pv);
        }
        if (add_xy) xyj = m.xy[fj];
    }
    __syncthreads();
    const long long tm3 = m.prof ? clock64() : 0;
    if (warp == 0) {
        const int c = fc;
        bool viol = false;
        if (fin_lane) {
            double pw[PK_WARPS];
#pragma unroll
            for (int w = 0; w < PK_WARPS; ++w) pw[w] = m.part[w * 32 + lane];
            double r = (((pw[0] + pw[1]) + (pw[2] + pw[3])) + ((pw[4] + pw[5]) + (pw[6] + pw[7]))) + xyj;   // fixed order
            if (fast) {
                r = prox_select(pk, r);
                if (__double_as_longlong(r) != __double_as_longlong(pk.pv)) {      // stop rule, src/utils.cpp:537-549
                    const bool bc = abs_gt(r, 1e-13), bp = abs_gt(pk.pv, 1e-13);
                    viol = bc != bp || (bc && abs_gt(r - pk.pv, pk.tolpv));
                }
            }
            *pub = r;
        }
        if (gflag_slot) {
            const unsigned vm = __reduce_or_sync(0xffffffffu, viol ? (1u << c) : 0u);
            if (lane == 0) *gflag_slot = (int)vm;
        }
        if (m.prof && threadIdx.x == 0 && add_xy) {
            const long long tm4 = clock64();
            m.prof[13] += tm1 - tm0; m.prof[14] += tm2 - tm1; m.prof[15] += tm4 - tm3; m.prof[7] += tm3 - tm2;
        }
    }
}

template <int MODE, int RPT>
__global__ void __launch_bounds__(PK_THREADS, 1) oem_path_kernel(const PathArgs a) {
    static_assert(PK_WARPS == 8, "matvec_reg sums eight warp partials");
    static_assert(RPT == 0 || MODE == MODE_GLOBAL, "the register mat-vec belongs to the global mode");
    extern __shared__ __align__(16) double sm[];
    if (a.skip && *a.skip) return;           // uniform over the grid: nobody reaches a barrier
    const unsigned long long t_in = (a.t_acc && blockIdx.x == 0 && threadIdx.x == 0) ? global_timer_ns() : 0ull;
    const int q = a.q, qs = a.qs;            // qs = padded vector / slice stride, = 4 (mod 16), >= roundup(q, 4)
    const int team = blockIdx.x / a.team_size, rank = blockIdx.x - team * a.team_size;
    const int c0 = min(q, rank * a.cpc), c1 = min(q, c0 + a.cpc);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ct0 = a.team_ptr[team], nct = a.team_ptr[team + 1] - ct0;
    const int nvec = max(a.max_ct, 2);

    // ---- shared-memory carve-up (doubles, then ints) ----
    double *Asl = sm;                                      // cpc_pad x qs (slice of XX, then of A)
    double *B0 = sm + (a.a_in_smem ? (size_t)a.cpc_pad * qs : 0);   // ping-pong iterate buffers, nvec x qs each,
    double *B1 = B0 + (size_t)nvec * qs;                   //   zero padded: beta lives in one, the other receives the next
    double *xy = B1 + (size_t)nvec * qs;                   // q
    double *pf = xy + q;                                   // q
    double *lam_sm = pf + q;                               // max_ct * Lmax
    double *gw = lam_sm + (size_t)a.max_ct * a.Lmax;       // ngroups
    double *part = gw + a.ngroups;                         // PK_PART x 64
    double *red = part + PK_PART * 64;                     // 16
    double *lz_al = red + 16;                              // LZ_MAX
    double *lz_be = lz_al + LZ_MAX;                        // LZ_MAX
    double *lz_ib = lz_be + LZ_MAX;                        // LZ_MAX
    double *ak = lz_ib + LZ_MAX;                           // PK_MAXCT
    double *chd = ak + PK_MAXCT;                           // 3 * PK_MAXCT: alpha, gamma, tau
    double *misc = chd + 3 * PK_MAXCT;                     // 8
    double *cpar = misc + 8;                               // 8 * PK_MAXCT: per-lambda derived constants
    double *psm = cpar + 8 * PK_MAXCT;                     // q, only with post_scale (oem.xtx scale.factor / sparse intercept)
    int *lam_idx = reinterpret_cast<int *>(psm + (a.post_scale ? q : 0));   // PK_MAXCT each
    int *iter = lam_idx + PK_MAXCT;
    int *done = iter + PK_MAXCT;
    int *chi = done + PK_MAXCT;                            // 3 * PK_MAXCT: penalty, nlam, out_off
    int *kind = chi + 3 * PK_MAXCT;                        // PK_MAXCT: 0 lasso-type, 1 mcp, 2 scad, 3 ols, 4 replicated (group)
    int *cflag = kind + PK_MAXCT;                          // 2 x 8: violation masks of the cluster members (by parity)
    int *violw = cflag + 16;                               // 4 ints: my violation mask (+ padding)
    int *grp_ptr = violw + 4;                              // ngroups + 1
    int *grp_unique = grp_ptr + a.ngroups + 1;             // ngroups
    int *grp_idx = grp_unique + a.ngroups;                 // ngidx
    int *cover = grp_idx + a.ngidx;                        // q (only with groups)

    unsigned *bar = a.barriers + team;
    unsigned bar_target = 0;
    double *ub = a.ubuf ? a.ubuf + (size_t)team * 2 * a.max_ct * q : nullptr;
    int *gflag = a.gflags ? a.gflags + (size_t)team * 2 * a.team_size : nullptr;
    const double *XXg = a.XX + (size_t)team * q * q;
    double *Amine = RPT > 0 ? nullptr : a.a_in_smem ? Asl : a.Abuf + ((size_t)team * a.team_size + rank) * a.cpc_pad * qs;

    // ---- one-time loads: my column slice of XX (zero padded to cpc_pad x qs) and every table ----
    // register variant: rows t, t + 256, ... of my 8 columns, straight from L2 (8 * RPT independent loads per thread)
    double areg[8][RPT > 0 ? RPT : 1];
    if (RPT > 0) {
#pragma unroll
        for (int jl = 0; jl < 8; ++jl)
#pragma unroll
            for (int r = 0; r < (RPT > 0 ? RPT : 1); ++r) {
                const int j = c0 + jl, i = threadIdx.x + r * PK_THREADS;
                areg[jl][r] = (j < c1 && i < q) ? __ldg(XXg + (size_t)j * q + i) : 0.0;
            }
    }
    for (int jl = warp; jl < (RPT > 0 ? 0 : a.cpc_pad); jl += PK_WARPS) {
        const int j = c0 + jl;
        double *dst = Amine + (size_t)jl * qs;
        const double *src = XXg + (size_t)j * q;
        // eight loads in flight per lane: one L2 round trip per 256 rows instead of one per 32 (this copy was ~10 us of
        // every launch of the logistic inner loop at q = 1001)
        for (int i0 = lane; i0 < qs; i0 += 32 * 8) {
            double tmp[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + 32 * u;
                tmp[u] = (j < c1 && i < q) ? __ldg(src + i) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + 32 * u;
                if (i < qs) dst[i] = tmp[u];
            }
        }
    }
    for (int e = threadIdx.x; e < 2 * nvec * qs; e += PK_THREADS) B0[e] = 0.0;
    for (int j = threadIdx.x; j < q; j += PK_THREADS) {
        xy[j] = (RPT > 0 && a.xy_grad) ? 0.0 : a.XY[(size_t)team * q + j];
        pf[j] = a.pen_fact ? a.pen_fact[j] : 1.0;
        if (a.ngroups) cover[j] = a.grp_cover[j];
        if (a.post_scale) psm[j] = a.post_scale[j];
    }
    for (int gi = threadIdx.x; gi < a.ngroups; gi += PK_THREADS) {
        gw[gi] = a.group_weights[gi];
        grp_unique[gi] = a.unique_groups[gi];
    }
    for (int gi = threadIdx.x; gi < a.ngroups + 1 && a.ngroups; gi += PK_THREADS) grp_ptr[gi] = a.grp_ptr[gi];
    for (int k = threadIdx.x; k < a.ngidx; k += PK_THREADS) grp_idx[k] = a.grp_idx[k];
    for (int c = threadIdx.x; c < nct; c += PK_THREADS) {
        const ChainDev ch = a.chains[a.team_idx[ct0 + c]];
        chi[c] = ch.penalty; chi[PK_MAXCT + c] = ch.nlam; chi[2 * PK_MAXCT + c] = ch.out_off;
        chd[c] = ch.alpha; chd[PK_MAXCT + c] = ch.gamma; chd[2 * PK_MAXCT + c] = ch.tau;
        lam_idx[c] = 0; iter[c] = 0; ak[c] = 1.0;
        done[c] = (ch.nlam <= 0) ? 1 : 0;
        const int pen = ch.penalty;
        kind[c] = (pen >= OEMB200_PEN_GRP_LASSO || a.accelerate) ? 4
                : pen == OEMB200_PEN_OLS ? 3
                : (pen == OEMB200_PEN_SCAD || pen == OEMB200_PEN_SCAD_NET) ? 2
                : (pen == OEMB200_PEN_MCP || pen == OEMB200_PEN_MCP_NET) ? 1 : 0;
    }
    for (int e = threadIdx.x; e < nct * a.Lmax; e += PK_THREADS) {
        const int c = e / a.Lmax, l = e - c * a.Lmax;
        const ChainDev ch = a.chains[a.team_idx[ct0 + c]];
        lam_sm[e] = l < ch.nlam ? a.lambdas[ch.lam_off + l] : 0.0;
    }
    if (threadIdx.x < 16) cflag[threadIdx.x] = 0;
    if (threadIdx.x == 0) violw[0] = 0;
    if (MODE == MODE_CLUSTER) cluster_sync_all();   // peers may start storing into my buffers
    else __syncthreads();
    SmemTabs tb{pf, gw, grp_ptr, grp_unique, grp_idx, cover, a.ngroups};

    // ---- exchange: barrier (+ in global mode the copy of the published vectors into my shared memory) ----
    // Global mode: one arrival counter per team (bar.sync orders the CTA's publications before thread 0's gpu-scope
    // release; the acquire poll + bar.sync makes the other members' publications visible to the whole CTA).  After the
    // barrier everything a member needs -- the published vectors AND the members' violation masks -- is requested in
    // ONE batch of loads (up to 12 doubles + 1 word in flight per thread) before the first use: one L2 round trip per
    // exchange (the chain-by-chain copy of round 1 paid one per chain, the masks one more).  A bulk-copy (cp.async.bulk
    // + mbarrier) version of this fetch was measured and is slower: 2.5 k cycles against 1.8 k for 24 KB.
    auto exchange = [&](int par, double *dst, int nv, const int *inactive, unsigned *flags_out) {
        if (MODE == MODE_SINGLE) __syncthreads();
        else if (MODE == MODE_CLUSTER) cluster_sync_all();
        else {
            const long long te0 = (a.prof && blockIdx.x == 0) ? clock64() : 0;
            __syncthreads();
            if (a.team_size > 1) {
                if (threadIdx.x == 0) {
                    bar_target += (unsigned)a.team_size;
                    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
                    unsigned v;
                    do {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
                    } while ((int)(v - bar_target) < 0);
                }
                __syncthreads();
            }
            if (a.prof && blockIdx.x == 0 && threadIdx.x == 0) a.prof[17] += clock64() - te0;
            const double *src = ub + (size_t)par * a.max_ct * q;
            unsigned fl = 0u;
            if (flags_out)
                for (int r = threadIdx.x; r < a.team_size; r += PK_THREADS) fl |= (unsigned)__ldcg(gflag + (size_t)par * a.team_size + r);
            constexpr int XB = 3;
            for (int cb = 0; cb < nv; cb += XB) {
                for (int j0 = threadIdx.x; j0 < q; j0 += 4 * PK_THREADS) {
                    double tmp[XB][4];
#pragma unroll
                    for (int cc = 0; cc < XB; ++cc) {
                        const int c = cb + cc;
                        const bool live = c < nv && !(inactive && inactive[c]);
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int j = j0 + u * PK_THREADS;
                            tmp[cc][u] = (live && j < q) ? ld_cg(src + (size_t)c * q + j) : 0.0;
                        }
                    }
#pragma unroll
                    for (int cc = 0; cc < XB; ++cc) {
                        const int c = cb + cc;
                        const bool live = c < nv && !(inactive && inactive[c]);
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int j = j0 + u * PK_THREADS;
                            if (live && j < q) dst[(size_t)c * qs + j] = tmp[cc][u];
                        }
                    }
                }
            }
            if (flags_out) *flags_out = fl;
            __syncthreads();
        }
    };

    MvCtx mv;
    mv.Amine = Amine; mv.xy = xy; mv.pf = pf; mv.cpar = cpar; mv.gam = chd + PK_MAXCT; mv.kind = kind;
    mv.part = part; mv.ub = ub; mv.violw = violw;
    mv.q = q; mv.qs = qs; mv.c0 = c0; mv.c1 = c1; mv.natm = a.cpc_pad >> 3; mv.max_ct = a.max_ct;
    mv.team_size = a.team_size; mv.tol = a.tol; mv.prof = (a.prof && blockIdx.x == 0) ? a.prof : nullptr;

    // =========================== phase 0: top eigenvalue ===========================
    double dval;
    int par = 0;
    if (a.compute_eig) {
        double *v = B0, *vprev = B0 + qs;      // w alternates between the two rows of B1 (remote stores need the parity)
        // deterministic pseudo-random start vector (fixed seed), normalised
        double ss = 0.0;
        for (int i = threadIdx.x; i < q; i += PK_THREADS) {
            unsigned h = (unsigned)i * 2654435761u + 0x9E3779B9u;
            h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
            const double x = (double)(h & 0xFFFFFF) / 16777216.0 + 0.25;
            v[i] = x; vprev[i] = 0.0;
            ss += x * x;
        }
        ss = block_sum(ss, red);
        const double inv = 1.0 / sqrt(ss);
        for (int i = threadIdx.x; i < q; i += PK_THREADS) v[i] *= inv;
        __syncthreads();
        double beta_prev = 0.0, theta = 0.0, lo_hint = -1e300, res_last = 0.0;
        bool capped = false;
        int k = 0;
        const long long tl0 = clock64();
        long long ttri = 0;
        const int kmax = min(LZ_MAX, max(q, 1));
        bool conv = false;
        while (!conv) {
            double *w = B1 + (size_t)par * qs;
            if constexpr (RPT > 0) matvec_reg<RPT, 1>(areg, mv, v, nullptr, 0, 0u, par, nullptr);
            else matvec_dmma<MODE>(mv, v, w, 1, nullptr, 0, 0u, par);
            exchange(par, w, 1, nullptr, nullptr);
            par ^= 1;
            double dot = 0.0;
            for (int i = threadIdx.x; i < q; i += PK_THREADS) dot = fma(v[i], w[i], dot);
            const double alpha_k = block_sum(dot, red);
            double nn = 0.0;
            for (int i = threadIdx.x; i < q; i += PK_THREADS) {
                const double x = w[i] - alpha_k * v[i] - beta_prev * vprev[i];
                w[i] = x;
                nn = fma(x, x, nn);
            }
            const double beta_k = sqrt(block_sum(nn, red));
            if (threadIdx.x == 0) { lz_al[k] = alpha_k; lz_be[k] = beta_k; lz_ib[k] = 1.0 / beta_k; }
            ++k;
            __syncthreads();
            // convergence check: every step while the tridiagonal is tiny, then every 8th
            const bool breakdown = !(beta_k > 1e-14 * fabs(alpha_k));
            if (k <= 4 || (k & 7) == 0 || breakdown || k >= kmax) {
                const long long tq = clock64();
                // a coarse Ritz value (bracket / 1.7e7) decides whether to look closer; the value that is used is exact
                tridiag_top(lz_al, lz_be, lz_ib, k, lo_hint, misc, red, reinterpret_cast<int *>(cpar), 3);
                __syncthreads();
                theta = misc[0];
                lo_hint = misc[2];
                double res = beta_k * misc[1];
                if (breakdown || k >= kmax || (res <= 4.0 * a.eig_tol * fabs(theta))) {
                    __syncthreads();
                    tridiag_top(lz_al, lz_be, lz_ib, k, lo_hint, misc, red, reinterpret_cast<int *>(cpar), 9);
                    __syncthreads();
                    theta = misc[0];
                    lo_hint = misc[2];
                    res = beta_k * misc[1];
                }
                ttri += clock64() - tq;
                res_last = res;
                conv = breakdown || k >= kmax || (res <= a.eig_tol * fabs(theta));
                // step cap reached before the Ritz value converged (q > LZ_MAX with a clustered top spectrum): an
                // unconverged Ritz value UNDER-estimates lambda_max, and d = factor * theta is the only margin that keeps
                // A = dI - XX positive semi-definite (1.0005 for the logistic entries), so the residual bound is added below
                capped = !breakdown && k >= kmax && k < q && !(res <= a.eig_tol * fabs(theta));
                __syncthreads();
            }
            if (!conv) {
                const double ib = 1.0 / beta_k;
                for (int i = threadIdx.x; i < q; i += PK_THREADS) {
                    vprev[i] = v[i];
                    v[i] = w[i] * ib;
                }
                beta_prev = beta_k;
                __syncthreads();
            }
        }
        dval = (capped ? theta + res_last : theta) * a.eig_factor;
        if (a.prof && blockIdx.x == 0 && threadIdx.x == 0) { a.prof[4] += clock64() - tl0; a.prof[5] += ttri; a.prof[6] += k; }
        if (rank == 0 && threadIdx.x == 0) {
            a.d[team] = dval;
            if (a.lanczos_steps) a.lanczos_steps[team] = k;
        }
    } else {
        dval = a.d[team];
    }

    // ---- logistic inner loop: XY = XX beta_init + grad for MY columns, from the XX slice in registers (the only entries of
    //      XY this member ever reads are its own; they also go to xy_out, which a later launch without a data pass reuses) ----
    if constexpr (RPT > 0) {
        if (a.xy_grad && nct > 0) {
            __syncthreads();
            for (int e = threadIdx.x; e < qs; e += PK_THREADS)
                B0[e] = (e < q && a.beta_init) ? a.beta_init[(size_t)a.chains[a.team_idx[ct0]].out_off * q + e] : 0.0;
            __syncthreads();
            double acc1[1][8], tot1[1];
#pragma unroll
            for (int jl = 0; jl < 8; ++jl) acc1[0][jl] = 0.0;
#pragma unroll
            for (int r = 0; r < RPT; ++r) {
                const int i = threadIdx.x + r * PK_THREADS;
                if (i < qs) {
                    const double b = B0[i];
#pragma unroll
                    for (int jl = 0; jl < 8; ++jl) acc1[0][jl] = fma(areg[jl][r], b, acc1[0][jl]);
                }
            }
            reduce_cols<1, 8>(acc1, tot1, lane);
            if ((lane & 3) == 0) part[warp * 8 + (lane >> 2)] = tot1[0];
            __syncthreads();
            if (threadIdx.x < 8 && c0 + (int)threadIdx.x < c1) {
                const int jr = c0 + threadIdx.x;
                double sxy = part[threadIdx.x];
#pragma unroll
                for (int w = 1; w < PK_WARPS; ++w) sxy += part[w * 8 + threadIdx.x];
                double gr;
                if (a.xy_icpt && jr == 0) gr = a.xy_grad[0] / a.xy_n;
                else {
                    const int jx = jr - a.xy_icpt;
                    gr = a.xy_grad[1 + jx] / a.xy_n;
                    if (a.xy_cinv) gr *= a.xy_cinv[jx];
                }
                xy[jr] = sxy + gr;
                a.xy_out[(size_t)team * q + jr] = sxy + gr;
            }
            __syncthreads();
        }
    }

    if (nct > 0) {
        // per-lambda derived constants of chain c (thread c): thresholds, denominators and their reciprocals
        auto set_cpar = [&](int c) {
            const int pen = chi[c];
            const double alpha = chd[c], gamma = chd[PK_MAXCT + c];
            const double lambda = lam_sm[(size_t)c * a.Lmax + min(lam_idx[c], a.Lmax - 1)];
            double denom = dval + (1.0 - alpha) * lambda, lam = lambda * alpha;
            if (pen == OEMB200_PEN_SCAD_NET && alpha == 0.0) { lam = 0.0; denom = dval + lambda; }
            const bool net = (pen == OEMB200_PEN_ENET || pen == OEMB200_PEN_SCAD_NET || pen == OEMB200_PEN_MCP_NET);
            const double lp = net ? lam : lambda, dp = net ? denom : dval;
            const bool is_scad = (pen == OEMB200_PEN_SCAD || pen == OEMB200_PEN_SCAD_NET);
            const bool is_mcp = (pen == OEMB200_PEN_MCP || pen == OEMB200_PEN_MCP_NET);
            const double gammad = gamma * dp;
            const double den2 = is_mcp ? dp - 1.0 / gamma : (gamma - 1.0) * dp - 1.0;   // second denominator
            double *cp = cpar + c * 8;
            cp[0] = lp; cp[1] = dp; cp[2] = (is_scad || is_mcp) ? fmin(1.0, gammad) : 1.0; cp[3] = lambda;
            cp[4] = __drcp_rn(dp); cp[5] = gammad; cp[6] = den2; cp[7] = __drcp_rn(den2);   // correctly rounded, like 1.0 / x
        };
        __syncthreads();      // the Lanczos scratch aliases cpar
        // ---- A = d I - XX on my slice; iterate buffers; first-lambda constants ----
        if (RPT > 0) {
#pragma unroll
            for (int jl = 0; jl < 8; ++jl)
#pragma unroll
                for (int r = 0; r < (RPT > 0 ? RPT : 1); ++r) {
                    const int i = threadIdx.x + r * PK_THREADS;
                    const double x = -areg[jl][r];
                    areg[jl][r] = (i == c0 + jl && i < c1) ? x + dval : x;
                }
        }
        for (int jl = warp; jl < (RPT > 0 ? 0 : a.cpc_pad); jl += PK_WARPS) {
            const int j = c0 + jl;
            double *col = Amine + (size_t)jl * qs;
            if (j < c1)
                for (int i = lane; i < q; i += 32) {
                    const double x = -col[i];
                    col[i] = (i == j) ? x + dval : x;
                }
        }
        for (int e = threadIdx.x; e < nvec * qs; e += PK_THREADS) {
            const int c = e / qs, j = e - c * qs;
            B0[e] = (c < nct && j < q && a.beta_init) ? a.beta_init[(size_t)chi[2 * PK_MAXCT + c] * q + j] : 0.0;
            B1[e] = 0.0;
        }
        if (threadIdx.x < nct) set_cpar(threadIdx.x);
        unsigned fastmask = 0u;
        bool any_slow = false;
        for (int c = 0; c < nct; ++c) {
            if (kind[c] < 4) fastmask |= 1u << c;
            else any_slow = true;
        }
        if (MODE == MODE_CLUSTER) cluster_sync_all();
        else __syncthreads();

        // =========================== phase 1: lambda paths ===========================
        // beta lives in Bc; the next iterate is assembled in Bn by the members that own its coordinates (the
        // coordinate-wise prox + stop rule run in the mat-vec epilogue), exchanged with ONE barrier, and the buffers
        // swap.  Group penalties / Nesterov publish u instead and every member applies the prox redundantly.
        int cur = 0;
        int *flagw = reinterpret_cast<int *>(red);      // 8 words: per-warp masks
        for (;;) {
            int nactive = 0;
            for (int c = 0; c < nct; ++c) nactive += done[c] ? 0 : 1;
            if (nactive == 0) break;
            long long t0 = clock64();
            double *Bc = cur ? B1 : B0, *Bn = cur ? B0 : B1;
            if constexpr (RPT > 0) {
                // the finishing warp publishes my violation mask itself (the exchange's bar.sync orders it)
                int *slot = gflag + (size_t)cur * a.team_size + rank;
                switch (nct) {
                    case 1: matvec_reg<RPT, 1>(areg, mv, Bc, done, 1, fastmask, cur, slot); break;
                    case 2: matvec_reg<RPT, 2>(areg, mv, Bc, done, 1, fastmask, cur, slot); break;
                    case 3: matvec_reg<RPT, 3>(areg, mv, Bc, done, 1, fastmask, cur, slot); break;
                    default: matvec_reg<RPT, 4>(areg, mv, Bc, done, 1, fastmask, cur, slot); break;
                }
            } else {
            matvec_dmma<MODE>(mv, Bc, Bn, nct, done, 1, fastmask, cur);
            __syncthreads();
            }
            // my violation mask -> every member (same parity slot scheme as the vectors)
            if (RPT == 0 && threadIdx.x == 0) {
                const int vm = violw[0];
                violw[0] = 0;
                if (MODE == MODE_SINGLE) cflag[cur * 8] = vm;
                else if (MODE == MODE_CLUSTER) {
                    for (int r = 0; r < a.team_size; ++r) {
                        unsigned remote;
                        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(&cflag[cur * 8 + rank])), "r"(r));
                        asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(remote), "r"(vm) : "memory");
                    }
                } else gflag[(size_t)cur * a.team_size + rank] = vm;
            }
            long long t1 = clock64();
            unsigned bad = 0u;
            exchange(cur, Bn, nct, done, &bad);
            long long t2 = clock64();
            if (MODE != MODE_GLOBAL && threadIdx.x < a.team_size) bad = (unsigned)cflag[cur * 8 + threadIdx.x];
            const long long tA = clock64();
            if (any_slow) {
                for (int c = 0; c < nct; ++c) {
                    if (done[c] || kind[c] < 4) continue;
                    double *bn = Bn + (size_t)c * qs;
                    const double *bo = Bc + (size_t)c * qs;
                    prox_inplace(q, tb, chi[c], chd[c], chd[PK_MAXCT + c], chd[2 * PK_MAXCT + c], cpar[c * 8 + 3], dval, bn);
                    if (a.accelerate) {     // Nesterov step, src/oem_dense.h:633-651
                        const double ak_prev = ak[c];
                        const double ak_new = 0.5 * (1.0 + sqrt(1.0 + 4.0 * ak_prev * ak_prev));
                        const double ratio = (ak_prev - 1.0) / ak_new;
                        double adv = 0.0;
                        for (int j = threadIdx.x; j < q; j += PK_THREADS) {
                            const double upd = bn[j];
                            const double diff = upd - bo[j];
                            const double acc = upd + ratio * diff;
                            bn[j] = acc;
                            adv += (acc - upd) * diff;
                        }
                        adv = block_sum(adv, red);
                        if (threadIdx.x == 0) ak[c] = (adv > 0.0) ? 1.0 : ak_new;
                    }
                    bool viol = false;      // stop rule, src/utils.cpp:537-549
                    for (int j = threadIdx.x; j < q; j += PK_THREADS) {
                        const double cv = bn[j], pv = bo[j];
                        if (__double_as_longlong(cv) == __double_as_longlong(pv)) continue;
                        const bool bc = abs_gt(cv, 1e-13), bp = abs_gt(pv, 1e-13);
                        if (bc != bp || (bc && abs_gt(cv - pv, a.tol * fabs(pv)))) viol = true;
                    }
                    if (viol) bad |= 1u << c;
                }
            }
            const long long tB = clock64();
            bad = __reduce_or_sync(0xffffffffu, bad);
            if (lane == 0) flagw[warp] = (int)bad;
            __syncthreads();
            bad = 0u;
#pragma unroll
            for (int w = 0; w < PK_WARPS; ++w) bad |= (unsigned)flagw[w];
            const long long tC = clock64();
            // nothing finished (the common iteration): only the iteration counters move.  In the global mode the
            // iterate buffers are written by the exchange alone, so no further CTA barrier is needed either.
            bool anyfin = false;
            for (int c = 0; c < nct; ++c)
                if (!done[c] && (!((bad >> c) & 1u) || iter[c] + 1 >= a.maxit)) anyfin = true;
            if (MODE == MODE_GLOBAL && !anyfin) {
                if (threadIdx.x < nct && !done[threadIdx.x]) iter[threadIdx.x] += 1;
                cur ^= 1;
                if (a.prof && blockIdx.x == 0 && threadIdx.x == 0) {
                    const long long t3 = clock64();
                    a.prof[0] += t1 - t0; a.prof[1] += t2 - t1; a.prof[2] += t3 - t2; a.prof[3] += 1;
                    a.prof[8] += tA - t2; a.prof[9] += tB - tA; a.prof[10] += tC - tB; a.prof[16] += 1;
                }
                continue;
            }
            // ---- finished chains (rare): scale.factor quirk of oem_xtx, then their column of the path ----
            for (int c = 0; c < nct; ++c) {
                if (done[c]) continue;
                const bool conv = !((bad >> c) & 1u);
                if (!(conv || iter[c] + 1 >= a.maxit)) continue;
                double *bn = Bn + (size_t)c * qs;
                double *bo = Bc + (size_t)c * qs;
                const bool last = lam_idx[c] + 1 >= chi[PK_MAXCT + c];
                double *gout = a.beta_out + ((size_t)chi[2 * PK_MAXCT + c] * a.Lmax + lam_idx[c]) * q;
                // every member holds the whole iterate and writes its own slice of the path column
                for (int j = threadIdx.x; j < q; j += PK_THREADS) {
                    double x = bn[j];
                    if (a.post_scale) { x *= psm[j]; bn[j] = x; }            // get_beta() mutates the iterate: src/oem_xtx.h:576-581
                    if (last) bo[j] = x;                                       // a finished chain keeps its beta in both buffers
                    if (j >= c0 && j < c1) gout[j] = x;
                }
            }
            __syncthreads();
            const long long tD = clock64();
            if (threadIdx.x < nct && !done[threadIdx.x]) {
                const int c = threadIdx.x;
                const int li = lam_idx[c], it = iter[c] + 1;
                const bool conv = !((bad >> c) & 1u);
                if (conv || it >= a.maxit) {
                    if (rank == 0) a.niter_out[(size_t)chi[2 * PK_MAXCT + c] * a.Lmax + li] = conv ? it : a.maxit + 1;
                    iter[c] = 0;
                    lam_idx[c] = li + 1;
                    if (li + 1 >= chi[PK_MAXCT + c]) done[c] = 1;
                    else set_cpar(c);
                } else {
                    iter[c] = it;
                }
            }
            cur ^= 1;
            // with replicated (group / Nesterov) chains a member still reads the old buffer after the exchange: keep the
            // cluster in step before peers overwrite it remotely
            if (MODE == MODE_CLUSTER && any_slow) cluster_sync_all();
            else __syncthreads();
            if (a.prof && blockIdx.x == 0 && threadIdx.x == 0) {
                const long long t3 = clock64();
                a.prof[0] += t1 - t0; a.prof[1] += t2 - t1; a.prof[2] += t3 - t2; a.prof[3] += 1;
                a.prof[8] += tA - t2; a.prof[9] += tB - tA; a.prof[10] += tC - tB; a.prof[11] += tD - tC; a.prof[12] += t3 - tD;
            }
        }
        // ---- IRLS epilogue: the outer loop's stop rule on (final iterate, warm start), verdicts, next pass's coefficients ----
        if (a.irls_conv && blockIdx.x == 0) {
            __syncthreads();
            const double *Bc = cur ? B1 : B0;                                   // chain 0 (the only one)
            const double *prev = a.beta_init + (size_t)chi[2 * PK_MAXCT] * q;
            int v = 0;
            for (int i = threadIdx.x; i < q; i += PK_THREADS) {
                const double cv = Bc[i], pv = prev[i];
                const double ac = fabs(cv), ap = fabs(pv);
                if ((ac > 1e-13 && ap <= 1e-13) || (ac <= 1e-13 && ap > 1e-13)) v = 1;
                else if (ac > 1e-13 && ap > 1e-13 && fabs((cv - pv) / pv) > a.irls_tol) v = 1;
                const int j = i - a.irls_icpt;
                if (a.irls_b && j >= 0 && j < a.irls_p) a.irls_b[j] = a.irls_cinv ? cv * a.irls_cinv[j] : cv;
            }
            v = __syncthreads_or(v);
            if (threadIdx.x == 0) {
                if (a.irls_b0) *a.irls_b0 = a.irls_icpt ? Bc[0] : 0.0;
                if (a.irls_iters_total) *a.irls_iters_total += a.niter_out[(size_t)chi[2 * PK_MAXCT] * a.Lmax];
                if (!v) *a.irls_conv = 1;
                if (a.irls_host_flag) *a.irls_host_flag = v ? 0 : 1;      // read by the host after this launch's event
            }
        }
    }
    if (MODE == MODE_CLUSTER) cluster_sync_all();   // no member may exit while peers can still write its shared memory
    if (a.t_acc && blockIdx.x == 0 && threadIdx.x == 0) *a.t_acc += global_timer_ns() - t_in;
}

// ---------------------------------------------------------------------------------------------
// Register-resident variant for the common small problem: q <= 256, coordinate-wise penalties only
// (lasso / ols / elastic.net / mcp / scad and their .net forms), no Nesterov, no scale.factor, cold start.
//
// A team is a cluster of NC <= 8 CTAs (1 CTA for q <= 128).  A CTA owns 8 * CPW columns of A = dI - XX; warp w owns
// CPW of them and keeps its CPW x q block IN REGISTERS for the whole path (lane l holds rows l, l + 32, ...:
// CPW * KPL <= 64 doubles per thread), so an OEM iteration reads nothing but the iterate from shared memory:
//     b[i]     = beta_c[l + 32 i]                       KPL conflict-free LDS per chain
//     acc[cc]  = sum_i A[cc][i] b[i]                    CPW independent DFMA chains (the FP64 CUDA-core pipe runs at
//                                                       the same rate as DMMA on this part, and a 1..4-column B
//                                                       operand would waste 4/8..7/8 of every DMMA)
//     multi-value butterfly over the 32 lanes           CPW - 1 + log2(32 / CPW) shuffles, fixed order
//     the 32 / CPW lanes that end up with column j's sum apply u = sum + XY_j, the coordinate-wise prox and the stop
//     rule (XY_j, pf_j and the previous beta_j live in their registers) and store the new beta_j into every member's
//     next-iterate buffer (DSMEM), each lane serving a different member
// then ONE cluster barrier per iteration (a __syncthreads for one CTA).  The per-warp violation masks travel with
// the same barrier; all threads keep the per-chain state (iteration count, lambda index) redundantly in registers,
// so nothing else is synchronised until a chain moves to its next lambda.
constexpr int PR_MAXCT = 4;       // chains per Gram handled by the register variant

template <int CPW, int KPL, int NCT>
__global__ void __launch_bounds__(PK_THREADS, 1) oem_path_reg_kernel(const PathArgs a) {
    constexpr int LPC = 32 / CPW;             // lanes that share one column after the butterfly
    constexpr int QP = KPL * 32;              // padded vector length
    extern __shared__ __align__(16) double sm[];
    const int q = a.q, NC = a.team_size;
    const int team = blockIdx.x / NC, rank = blockIdx.x - team * NC;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ct0 = a.team_ptr[team], nct = a.team_ptr[team + 1] - ct0;      // nct <= NCT (teams may have fewer chains)

    double *Bsm = sm;                                         // [2][NCT][QP]
    double *lam_sm = Bsm + 2 * NCT * QP;                      // [NCT][Lmax]
    double *cpar = lam_sm + (size_t)NCT * a.Lmax;             // [NCT][8]
    double *chd = cpar + NCT * 8;                             // alpha, gamma per chain: [2][NCT]
    uint64_t *xbar = reinterpret_cast<uint64_t *>(chd + 2 * NCT);   // [2]: per-parity transaction barriers of the exchange
    int *flags = reinterpret_cast<int *>(xbar + 2);           // [2][64]: violation masks by (parity, member, warp)
    int *chi = flags + 128;                                   // penalty, nlam, out_off, kind: [4][NCT]

    const int j = rank * (8 * CPW) + warp * CPW + lane / LPC; // the column this lane finishes
    const int sub = lane % LPC;
    const bool jvalid = j < q;
    const double dval = a.d[team];
    const double *XXg = a.XX + (size_t)team * q * q;

    // ---- one-time loads ----
    double A[CPW][KPL];
#pragma unroll
    for (int cc = 0; cc < CPW; ++cc) {
        const int jj = rank * (8 * CPW) + warp * CPW + cc;
#pragma unroll
        for (int i = 0; i < KPL; ++i) {
            const int k = lane + 32 * i;
            double x = 0.0;
            if (jj < q && k < q) { x = -XXg[(size_t)jj * q + k]; if (k == jj) x += dval; }
            A[cc][i] = x;
        }
    }
    const double xyj = jvalid ? a.XY[(size_t)team * q + j] : 0.0;
    const double pfj = jvalid ? (a.pen_fact ? a.pen_fact[j] : 1.0) : 0.0;
    for (int e = threadIdx.x; e < 2 * NCT * QP; e += PK_THREADS) Bsm[e] = 0.0;
    for (int e = threadIdx.x; e < 128; e += PK_THREADS) flags[e] = 0;
    if (threadIdx.x == 0) { mbar_init(&xbar[0], 1); mbar_init(&xbar[1], 1); mbar_fence_init(); }
    if (threadIdx.x < NCT) {
        const int c = threadIdx.x;
        if (c < nct) {
            const ChainDev ch = a.chains[a.team_idx[ct0 + c]];
            const int pen = ch.penalty;
            chi[c] = pen; chi[NCT + c] = ch.nlam; chi[2 * NCT + c] = ch.out_off;
            chi[3 * NCT + c] = pen == OEMB200_PEN_OLS ? 3
                             : (pen == OEMB200_PEN_SCAD || pen == OEMB200_PEN_SCAD_NET) ? 2
                             : (pen == OEMB200_PEN_MCP || pen == OEMB200_PEN_MCP_NET) ? 1 : 0;
            chd[c] = ch.alpha; chd[NCT + c] = ch.gamma;
            for (int l = 0; l < a.Lmax; ++l) lam_sm[(size_t)c * a.Lmax + l] = l < ch.nlam ? a.lambdas[ch.lam_off + l] : 0.0;
        } else {
            chi[c] = 0; chi[NCT + c] = 0; chi[2 * NCT + c] = 0; chi[3 * NCT + c] = 0;
            chd[c] = 1.0; chd[NCT + c] = 3.0;
            for (int l = 0; l < a.Lmax; ++l) lam_sm[(size_t)c * a.Lmax + l] = 0.0;
        }
    }
    __syncthreads();
    // per-lambda derived constants of chain c: thresholds, denominators and their reciprocals (as in the generic kernel)
    auto set_cpar = [&](int c, int li) {
        const int pen = chi[c];
        const double alpha = chd[c], gamma = chd[NCT + c];
        const double lambda = lam_sm[(size_t)c * a.Lmax + min(li, a.Lmax - 1)];
        double denom = dval + (1.0 - alpha) * lambda, lam = lambda * alpha;
        if (pen == OEMB200_PEN_SCAD_NET && alpha == 0.0) { lam = 0.0; denom = dval + lambda; }
        const bool net = (pen == OEMB200_PEN_ENET || pen == OEMB200_PEN_SCAD_NET || pen == OEMB200_PEN_MCP_NET);
        const double lp = net ? lam : lambda, dp = net ? denom : dval;
        const bool is_scad = (pen == OEMB200_PEN_SCAD || pen == OEMB200_PEN_SCAD_NET);
        const bool is_mcp = (pen == OEMB200_PEN_MCP || pen == OEMB200_PEN_MCP_NET);
        const double gammad = gamma * dp;
        const double den2 = is_mcp ? dp - 1.0 / gamma : (gamma - 1.0) * dp - 1.0;
        double *cp = cpar + c * 8;
        cp[0] = lp; cp[1] = dp; cp[2] = (is_scad || is_mcp) ? fmin(1.0, gammad) : 1.0; cp[3] = lambda;
        cp[4] = 1.0 / dp; cp[5] = gammad; cp[6] = den2; cp[7] = 1.0 / den2;
    };
    if (threadIdx.x < NCT) set_cpar(threadIdx.x, 0);

    // replicated per-chain state (identical in every thread of the team)
    int iter[NCT], lidx[NCT], kind[NCT];
    double prev[NCT], gam[NCT];
    unsigned done = 0u;
#pragma unroll
    for (int c = 0; c < NCT; ++c) {
        iter[c] = 0; lidx[c] = 0; prev[c] = 0.0;
        kind[c] = chi[3 * NCT + c];
        gam[c] = chd[NCT + c];
        if (c >= nct || chi[NCT + c] <= 0) done |= 1u << c;
    }
    if (NC > 1) cluster_sync_all();      // peers may start storing into my buffers
    else __syncthreads();
    // per-lambda constants of every chain live in registers; refreshed when a chain moves to its next lambda
    // ... as the thresholds of the region tests of THIS lane's column (prox_select), so that an iteration's prox is a few
    // integer comparisons, one select and one Markstein division after the column sum arrives
    ProxPre pk[NCT];
    auto load_pre = [&](int c) {
        const double *cp = cpar + c * 8;
        const double gamma = gam[c];
        pk[c].kind = kind[c];
        pk[c].tp = pfj * cp[0]; pk[c].dp = cp[1]; pk[c].rdp = cp[4]; pk[c].den2 = cp[6]; pk[c].rden2 = cp[7];
        pk[c].thr_big = cp[5] * pk[c].tp;
        pk[c].thr_mid = (pk[c].dp + 1.0) * pk[c].tp;
        pk[c].gpen = gamma * pk[c].tp; pk[c].gm1 = gamma - 1.0;
        pk[c].pv = 0.0; pk[c].tolpv = 0.0;
    };
#pragma unroll
    for (int c = 0; c < NCT; ++c) load_pre(c);

    const unsigned all = (1u << NCT) - 1u;
    int par = 0;
    long long niters = 0, tmv = 0, tbar = 0;
    const bool prof = a.prof != nullptr;
    const long long tstart = clock64();
    while (done != all) {
        const double *Bc = Bsm + (size_t)par * NCT * QP;
        double *Bn = Bsm + (size_t)(par ^ 1) * NCT * QP;
        const long long tp0 = prof ? clock64() : 0;
        // ---- u = A' beta + XY for all chains (finished chains ride along: their results are discarded) ----
        double acc[NCT][CPW], tot[NCT];
        {
            double b[NCT][KPL];
#pragma unroll
            for (int c = 0; c < NCT; ++c)
#pragma unroll
                for (int i = 0; i < KPL; ++i) b[c][i] = Bc[c * QP + lane + 32 * i];
#pragma unroll
            for (int c = 0; c < NCT; ++c)
#pragma unroll
                for (int cc = 0; cc < CPW; ++cc) {
                    double s = 0.0;
#pragma unroll
                    for (int i = 0; i < KPL; ++i) s = fma(A[cc][i], b[c][i], s);
                    acc[c][cc] = s;
                }
        }
        reduce_cols<NCT, CPW>(acc, tot, lane);
        // ---- coordinate-wise prox (src/oem_dense.h:527-629) and stop rule (src/utils.cpp:537-549) on the owner lanes ----
        unsigned viol = 0u;
        double rnew[NCT];
#pragma unroll
        for (int c = 0; c < NCT; ++c) {
            double r = prox_select(pk[c], tot[c] + xyj);
            if (!jvalid) r = 0.0;
            const double pv = prev[c];
            if (__double_as_longlong(r) != __double_as_longlong(pv)) {
                const bool bc = abs_gt(r, 1e-13), bp = abs_gt(pv, 1e-13);
                if (bc != bp || (bc && abs_gt(r - pv, a.tol * fabs(pv)))) viol |= 1u << c;
            }
            rnew[c] = r;
        }
        viol &= ~done;
#pragma unroll
        for (int c = 0; c < NCT; ++c) {
            if ((done >> c) & 1u) continue;
            prev[c] = rnew[c];
            if (jvalid) {
                double *dst = Bn + c * QP + j;
                if (NC == 1) { if (sub == 0) *dst = rnew[c]; }
                else
                    for (int rr = sub; rr < NC; rr += LPC)
                        st_async_f64(map_cluster(dst, (unsigned)rr), rnew[c], map_cluster(&xbar[par], (unsigned)rr));
            }
        }
        viol = __reduce_or_sync(0xffffffffu, viol);
        const long long tp1 = prof ? clock64() : 0;
        if (NC == 1) {
            if (lane == 0) flags[par * 64 + warp] = (int)viol;
            __syncthreads();
        } else {
            // every member receives q values per live chain and NC * 8 warp masks on its parity barrier
            if (lane < NC)
                st_async_u32(map_cluster(&flags[par * 64 + rank * 8 + warp], (unsigned)lane), viol,
                             map_cluster(&xbar[par], (unsigned)lane));
            if (threadIdx.x == 0)
                mbar_arrive_expect_tx(&xbar[par], (uint32_t)(q * __popc(~done & all) * 8 + NC * 8 * 4));
            mbar_wait_cluster(&xbar[par], (uint32_t)((niters >> 1) & 1));
        }
        const long long tp2 = prof ? clock64() : 0;
        unsigned bad = 0u;
        if (lane < NC * 8) bad = (unsigned)flags[par * 64 + lane];
        if (lane + 32 < NC * 8) bad |= (unsigned)flags[par * 64 + lane + 32];
        bad = __reduce_or_sync(0xffffffffu, bad);
        // ---- chain state (every thread, identically) ----
        unsigned advanced = 0u;
#pragma unroll
        for (int c = 0; c < NCT; ++c) {
            if ((done >> c) & 1u) continue;
            const int it = iter[c] + 1;
            const bool conv = !((bad >> c) & 1u);
            if (conv || it >= a.maxit) {
                const int li = lidx[c];
                const size_t col = (size_t)chi[2 * NCT + c] * a.Lmax + li;
                if (jvalid && sub == 0) a.beta_out[col * q + j] = prev[c];
                if (blockIdx.x == team * NC && threadIdx.x == 0) a.niter_out[col] = conv ? it : a.maxit + 1;
                iter[c] = 0;
                lidx[c] = li + 1;
                if (li + 1 >= chi[NCT + c]) done |= 1u << c;
                else advanced |= 1u << c;
            } else {
                iter[c] = it;
            }
        }
        if (advanced) {        // uniform over the whole team: new per-lambda constants before the next epilogue reads them
            // (the exchange wait already orders every warp's earlier reads of cpar before this point; the explicit
            // barrier keeps the write-after-read visible to tools and costs nothing at one event per lambda)
            __syncthreads();
#pragma unroll
            for (int c = 0; c < NCT; ++c)
                if (((advanced >> c) & 1u) && threadIdx.x == c) set_cpar(c, lidx[c]);
            __syncthreads();
#pragma unroll
            for (int c = 0; c < NCT; ++c)
                if ((advanced >> c) & 1u) load_pre(c);
        }
        par ^= 1;
        ++niters;
        if (prof) { tmv += tp1 - tp0; tbar += tp2 - tp1; }
    }
    if (prof && blockIdx.x == 0 && threadIdx.x == 0) {
        a.prof[0] += clock64() - tstart; a.prof[3] += niters; a.prof[1] += tmv; a.prof[2] += tbar;
    }
    if (NC > 1) cluster_sync_all();      // no member may exit while peers can still write its shared memory
}

// Shared memory every member of a generic path launch needs besides its slice of A: the ping-pong iterates of all the
// team's chains, XY, per-lambda tables, the Lanczos tridiagonal, group tables.
// XY = XX beta + grad with grad = [g0 / n, (g_j / n) o colsq_inv] (oem_logistic_dense.h:970-999).  One warp per row.
__global__ void path_xy_kernel(int q, int icpt, const double *__restrict__ XX, const double *__restrict__ beta,
                               const double *__restrict__ g, const double *__restrict__ cinv, double n_tot,
                               double *__restrict__ XY, const int *__restrict__ skip) {
    if (skip && *skip) return;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= q) return;
    const int lane = threadIdx.x & 31;
    // four independent partial sums per lane: the 8 MB of XX come from L2, one dependent FMA chain per lane left the loads
    // of a row serialised (12 us per call at q = 1001, once per IRLS data pass)
    const double *row = XX + (size_t)r * q;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int c = lane;
    for (; c + 96 < q; c += 128) {
        const double x0 = __ldg(row + c), x1 = __ldg(row + c + 32), x2 = __ldg(row + c + 64), x3 = __ldg(row + c + 96);
        s0 = fma(x0, beta[c], s0); s1 = fma(x1, beta[c + 32], s1);
        s2 = fma(x2, beta[c + 64], s2); s3 = fma(x3, beta[c + 96], s3);
    }
    for (; c < q; c += 32) s0 = fma(__ldg(row + c), beta[c], s0);
    double s = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
        double gr;
        if (icpt && r == 0) gr = g[0] / n_tot;
        else {
            const int j = r - icpt;
            gr = g[1 + j] / n_tot;
            if (cinv) gr *= cinv[j];
        }
        XY[r] = s + gr;
    }
}

static void path_xy_launch(Ctx &cx, int q, int icpt, const double *XX, const double *beta, const double *g, const double *cinv,
                           double n_tot, double *XY, const int *skip) {
    path_xy_kernel<<<(q + 7) / 8, 256, 0, cx.stream>>>(q, icpt, XX, beta, g, cinv, n_tot, XY, skip);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

static size_t path_fixed_smem_bytes(int q, int max_ct, int Lmax, int ng, int ngidx, bool post = false) {
    const int nvec = std::max(max_ct, 2);
    const int q4 = (q + 3) / 4 * 4;
    const int qs = q4 + (((4 - q4) % 16) + 16) % 16;
    return ((size_t)2 * nvec * qs + 2 * (size_t)q + (size_t)max_ct * std::max(Lmax, 1) + ng + PK_PART * 64 + 16 +
            3 * LZ_MAX + PK_MAXCT + 3 * PK_MAXCT + 8 + 8 * PK_MAXCT + (post ? (size_t)q : 0)) * 8 +
           ((size_t)7 * PK_MAXCT + 20 + (ng ? 2 * (size_t)ng + 1 + ngidx + q : 0)) * 4 + 16;
}

// Entry drivers call this BEFORE their passes over X: a beta dimension the path kernel cannot hold (p in the several
// thousands -- the n <= p use of oem_fit_dense is where that happens) is refused up front instead of after a p x p Gram
// has been allocated and computed.
void path_check_fits(Ctx &cx, int q, int chains_per_gram, int Lmax, int ngroups, int ngidx) {
    const int ct = std::max(1, std::min(chains_per_gram, PK_MAXCT));
    if (chains_per_gram > PK_MAXCT) fail(OEMB200_EUNSUPPORTED, "path: more than %d penalties in one call", PK_MAXCT);
    const size_t need = path_fixed_smem_bytes(q, ct, Lmax, ngroups, ngroups ? ngidx : 0);
    if (need > cx.smem_optin)
        fail(OEMB200_EUNSUPPORTED, "beta has %d coefficients: with %d penalties per call and %d lambdas the path kernel needs %zu bytes "
             "of shared memory per CTA (%zu available); fit fewer penalties per call or reduce p (about %d coefficients fit)", q, ct,
             std::max(Lmax, 1), need, cx.smem_optin, (int)((cx.smem_optin - 16000) / (8 * (2 * std::max(ct, 2) + 2))));
}

// ---------------------------------------------------------------------------------------------
void path_launch(Ctx &cx, const PathProblem &pp) {
    const int q = pp.q, G = pp.ngram;
    if (q <= 0 || G <= 0) fail(OEMB200_EINVAL, "path: empty problem");
    // chains per team
    std::vector<int> tptr(G + 1, 0), tidx(pp.chains.size());
    for (auto &c : pp.chains) {
        if (c.gram < 0 || c.gram >= G) fail(OEMB200_EINVAL, "path: chain refers to Gram %d of %d", c.gram, G);
        tptr[c.gram + 1]++;
    }
    int max_ct = 1;
    for (int g = 0; g < G; ++g) { max_ct = std::max(max_ct, tptr[g + 1]); tptr[g + 1] += tptr[g]; }
    if (max_ct > PK_MAXCT) fail(OEMB200_EUNSUPPORTED, "path: more than %d chains on one Gram", PK_MAXCT);
    {
        std::vector<int> fill(tptr.begin(), tptr.end() - 1);
        for (size_t i = 0; i < pp.chains.size(); ++i) tidx[fill[pp.chains[i].gram]++] = (int)i;
    }
    std::vector<ChainDev> cd(pp.chains.size());
    for (size_t i = 0; i < pp.chains.size(); ++i) {
        const ChainDesc &c = pp.chains[i];
        if (c.nlam > pp.Lmax) fail(OEMB200_EINVAL, "path: chain has more lambdas than Lmax");
        cd[i] = ChainDev{c.gram, c.penalty, c.nlam, c.lam_off, c.alpha, c.gamma, c.tau, c.out_off, 0};
    }

    // ---- small coordinate-wise problems: register-resident variant (d comes from a Lanczos-only generic launch) ----
    {
        bool reg_ok = q <= 256 && !pp.accelerate && !pp.post_scale && !pp.beta_init && !pp.skip &&
                      !pp.irls_conv && max_ct <= PR_MAXCT && !pp.chains.empty();
        for (auto &c : pp.chains) reg_ok = reg_ok && c.penalty < OEMB200_PEN_GRP_LASSO;
        const int NC = q <= 128 ? 1 : (q + 31) / 32;
        const int QP = q <= 128 ? 128 : 256;
        const int Lm = std::max(pp.Lmax, 1);
        const int nctt = std::max(1, std::min(max_ct, PR_MAXCT));
        const size_t smem_bytes = ((size_t)2 * nctt * QP + (size_t)nctt * Lm + nctt * 8 + 2 * nctt + 2) * 8 + (128 + 4 * nctt) * 4;
        void *kern = nullptr;
        if (reg_ok && G * NC <= cx.num_sms && smem_bytes <= cx.smem_optin) {
#define PR_PICK(N)                                                                                                   \
    case N: kern = q <= 128 ? (void *)oem_path_reg_kernel<16, 4, N> : (void *)oem_path_reg_kernel<4, 8, N>; break
            switch (nctt) { PR_PICK(1); PR_PICK(2); PR_PICK(3); default: PR_PICK(4); }
#undef PR_PICK
            OEM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
            // a cluster shape this device cannot schedule (MIG slices, odd GPC sizes) falls back to the generic kernel
            cudaLaunchConfig_t probe;
            memset(&probe, 0, sizeof probe);
            probe.gridDim = dim3(G * NC); probe.blockDim = dim3(PK_THREADS); probe.dynamicSmemBytes = smem_bytes;
            cudaLaunchAttribute pat[1];
            pat[0].id = cudaLaunchAttributeClusterDimension;
            pat[0].val.clusterDim.x = NC; pat[0].val.clusterDim.y = 1; pat[0].val.clusterDim.z = 1;
            probe.attrs = pat; probe.numAttrs = 1;
            int nclusters = 0;
            if (cudaOccupancyMaxActiveClusters(&nclusters, kern, &probe) != cudaSuccess || nclusters < 1) {
                (void)cudaGetLastError();
                kern = nullptr;
            }
        }
        if (kern) {
            if (pp.compute_eig) {
                PathProblem eig = pp;
                eig.chains.clear();
                path_launch(cx, eig);
            }
            DBuf<ChainDev> d_chains(cd.size());
            DBuf<int> d_tptr(tptr.size()), d_tidx(tidx.size());
            d_chains.upload(cd.data(), cd.size(), cx.stream);
            d_tptr.upload(tptr.data(), tptr.size(), cx.stream);
            d_tidx.upload(tidx.data(), tidx.size(), cx.stream);
            PathArgs a;
            memset(&a, 0, sizeof a);
            a.q = q; a.qs = QP; a.ngram = G; a.team_size = NC; a.cpc = q <= 128 ? 128 : 32; a.max_ct = max_ct; a.Lmax = Lm;
            a.maxit = pp.maxit; a.tol = pp.tol;
            a.XX = pp.XX; a.XY = pp.XY; a.d = pp.d;
            a.chains = d_chains.p; a.team_ptr = d_tptr.p; a.team_idx = d_tidx.p;
            a.lambdas = pp.lambdas; a.pen_fact = pp.pen_fact; a.beta_out = pp.beta_out; a.niter_out = pp.niter_out;
            DBuf<long long> d_prof;
            const bool prof = getenv("OEMB200_PATH_PROF") != nullptr;
            if (prof) { d_prof.alloc(32); d_prof.zero(cx.stream); a.prof = d_prof.p; }
            void *kargs[] = {&a};
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof cfg);
            cfg.gridDim = dim3(G * NC); cfg.blockDim = dim3(PK_THREADS); cfg.dynamicSmemBytes = smem_bytes; cfg.stream = cx.stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = NC; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            OEM_CUDA(cudaLaunchKernelExC(&cfg, kern, kargs));
            cx.st.kernel_launches += 1;
            if (prof) {
                long long h[32];
                d_prof.download(h, 32, cx.stream);
                OEM_CUDA(cudaStreamSynchronize(cx.stream));
                fprintf(stderr, "[path prof] register variant: team=%d q=%d nct=%d | iters=%lld cyc/iter=%.0f (matvec+prox %.0f, barrier %.0f)\n",
                        NC, q, max_ct, h[3], h[3] ? (double)h[0] / h[3] : 0.0, h[3] ? (double)h[1] / h[3] : 0.0,
                        h[3] ? (double)h[2] / h[3] : 0.0);
            }
            return;
        }
    }

    // ---- geometry: mode, team size, column slice, shared memory ----
    const int nvec = std::max(max_ct, 2);
    const int q4 = (q + 3) / 4 * 4;
    const int qs = q4 + (((4 - q4) % 16) + 16) % 16;      // smallest value >= roundup(q,4) that is 4 (mod 16)
    const int ng = pp.ngroups, ngidx = ng ? pp.ngidx : 0;
    const size_t fixed_bytes = path_fixed_smem_bytes(q, max_ct, pp.Lmax, ng, ngidx, pp.post_scale != nullptr);
    const size_t smem_cap = cx.smem_optin;
    if (fixed_bytes > smem_cap)
        fail(OEMB200_EUNSUPPORTED, "path: q=%d with %d chains per Gram and %d lambdas exceeds shared memory", q, max_ct, pp.Lmax);
    auto slice_bytes = [&](int members) {
        const int cpc_ = (q + members - 1) / members;
        return (size_t)((cpc_ + 7) / 8 * 8) * qs * 8;
    };
    int mode, team;
    if (slice_bytes(1) + fixed_bytes <= smem_cap) { mode = MODE_SINGLE; team = 1; }
    else {
        int cs = 0;
        for (int c : {8, 4, 2})      // more members = less mat-vec work each; the cluster barrier costs the same
            if (slice_bytes(c) + fixed_bytes <= smem_cap && (q + c - 1) / c >= 16) { cs = c; break; }
        if (cs && G * cs <= cx.num_sms) { mode = MODE_CLUSTER; team = cs; }
        else { mode = MODE_GLOBAL; team = 0; }
    }
    void *kern = mode == MODE_SINGLE ? (void *)oem_path_kernel<MODE_SINGLE, 0>
               : mode == MODE_CLUSTER ? (void *)oem_path_kernel<MODE_CLUSTER, 0> : (void *)oem_path_kernel<MODE_GLOBAL, 0>;
    // the attribute and the occupancy answer are per (kernel, device): asked once, not on every launch of an IRLS loop
    static int per_sm_cache[3 + 4][64];
    static bool attr_set[3 + 4][64];
    const int dslot = cx.device & 63;
    auto prepare_kernel = [&](void *k, int slot) {
        if (attr_set[slot][dslot]) return;
        OEM_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
        int ps = 0;
        OEM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ps, k, PK_THREADS, smem_cap));
        per_sm_cache[slot][dslot] = ps;
        attr_set[slot][dslot] = true;
    };
    prepare_kernel(kern, mode);
    if (mode == MODE_GLOBAL) {
        const int per_sm = per_sm_cache[mode][dslot];
        const int max_ctas = std::max(1, per_sm) * cx.num_sms;
        if (G > max_ctas) fail(OEMB200_EUNSUPPORTED, "path: %d Grams exceed the %d co-resident CTAs", G, max_ctas);
        team = std::max(1, std::min(max_ctas / G, (q + 7) / 8));       // at least one 8-column MMA atom per member
    }
    int cpc = (q + team - 1) / team;
    if (mode == MODE_GLOBAL) {
        cpc = (cpc + 7) / 8 * 8;                                       // whole atoms: no padded tensor work
        team = (q + cpc - 1) / cpc;                                    // drop members that would own nothing
    }
    const int cpc_pad = (cpc + 7) / 8 * 8;
    // one 8-column atom per member and <= 4 chains: the register-resident mat-vec (matvec_reg)
    int rpt = 0;
    if (mode == MODE_GLOBAL && cpc_pad == 8 && max_ct <= 4 && qs <= 5 * PK_THREADS) {
        rpt = std::max(2, (qs + PK_THREADS - 1) / PK_THREADS);
        void *kr = rpt == 2 ? (void *)oem_path_kernel<MODE_GLOBAL, 2> : rpt == 3 ? (void *)oem_path_kernel<MODE_GLOBAL, 3>
                 : rpt == 4 ? (void *)oem_path_kernel<MODE_GLOBAL, 4> : (void *)oem_path_kernel<MODE_GLOBAL, 5>;
        prepare_kernel(kr, 3 + rpt - 2);
        if (per_sm_cache[3 + rpt - 2][dslot] >= 1 && G * team <= per_sm_cache[3 + rpt - 2][dslot] * cx.num_sms) kern = kr;
        else rpt = 0;
    }
    const bool a_in_smem = rpt == 0 && (size_t)cpc_pad * qs * 8 + fixed_bytes <= smem_cap;
    const size_t smem_bytes = fixed_bytes + (a_in_smem ? (size_t)cpc_pad * qs * 8 : 0);

    // device tables: rebuilt unless the caller's scratch already holds exactly this layout
    PathScratch local_scratch;
    PathScratch &S = pp.scratch ? *pp.scratch : local_scratch;
    std::vector<unsigned char> key;
    {
        auto put = [&](const void *ptr, size_t bytes) {
            const unsigned char *b = static_cast<const unsigned char *>(ptr);
            key.insert(key.end(), b, b + bytes);
        };
        const int geo[11] = {q, qs, G, team, cpc_pad, max_ct, mode, a_in_smem ? 1 : 0, (int)cd.size(), cx.device, rpt};
        put(geo, sizeof geo);
        if (!cd.empty()) put(cd.data(), cd.size() * sizeof(ChainDev));
        put(tptr.data(), tptr.size() * sizeof(int));
        if (!tidx.empty()) put(tidx.data(), tidx.size() * sizeof(int));
    }
    if (S.key != key) {
        S.chains.alloc(std::max<size_t>(1, cd.size()));
        S.tptr.alloc(tptr.size());
        S.tidx.alloc(std::max<size_t>(1, tidx.size()));
        // barrier words and violation flags share one allocation so that one memset clears both before a launch
        S.ubuf.release(); S.A.release();
        S.nflags = mode == MODE_GLOBAL ? (size_t)G * 2 * team : 0;
        S.bar.alloc((size_t)G + S.nflags);
        if (mode == MODE_GLOBAL) S.ubuf.alloc((size_t)G * 2 * max_ct * q);
        if (!a_in_smem && rpt == 0) S.A.alloc((size_t)G * team * cpc_pad * qs);
        if (!cd.empty()) S.chains.upload(cd.data(), cd.size(), cx.stream);
        S.tptr.upload(tptr.data(), tptr.size(), cx.stream);
        if (!tidx.empty()) S.tidx.upload(tidx.data(), tidx.size(), cx.stream);
        S.key = key;
    }
    DBuf<ChainDev> &d_chains = S.chains;
    DBuf<int> &d_tptr = S.tptr, &d_tidx = S.tidx;
    DBuf<double> &d_ubuf = S.ubuf, &d_A = S.A;
    DBuf<unsigned> &d_bar = S.bar;
    int *const d_gflags_p = S.nflags ? reinterpret_cast<int *>(S.bar.p + G) : nullptr;
    d_bar.zero(cx.stream);

    PathArgs a;
    memset(&a, 0, sizeof a);
    a.q = q; a.qs = qs; a.ngram = G; a.team_size = team; a.cpc = cpc; a.cpc_pad = cpc_pad; a.max_ct = max_ct;
    a.Lmax = std::max(pp.Lmax, 1);
    a.maxit = pp.maxit; a.accelerate = pp.accelerate ? 1 : 0; a.compute_eig = pp.compute_eig ? 1 : 0;
    a.a_in_smem = a_in_smem ? 1 : 0; a.ngroups = ng; a.mode = mode; a.ngidx = ngidx;
    a.tol = pp.tol; a.eig_factor = pp.eig_factor; a.eig_tol = pp.eig_tol;
    a.XX = pp.XX; a.XY = pp.XY; a.d = pp.d; a.Abuf = d_A.p;
    a.chains = d_chains.p; a.team_ptr = d_tptr.p; a.team_idx = d_tidx.p;
    a.lambdas = pp.lambdas; a.pen_fact = pp.pen_fact;
    a.unique_groups = pp.unique_groups; a.grp_ptr = pp.grp_ptr; a.grp_idx = pp.grp_idx; a.grp_cover = pp.grp_cover;
    a.group_weights = pp.group_weights; a.post_scale = pp.post_scale; a.beta_init = pp.beta_init;
    a.beta_out = pp.beta_out; a.niter_out = pp.niter_out;
    a.lanczos_steps = pp.lanczos_steps; a.ubuf = d_ubuf.p; a.barriers = d_bar.p; a.gflags = d_gflags_p;
    a.skip = pp.skip; a.t_acc = pp.t_acc;
    if (pp.irls_conv) {
        if (G != 1 || pp.chains.size() != 1 || pp.chains[0].nlam != 1 || !pp.beta_init)
            fail(OEMB200_EINVAL, "path: the IRLS epilogue needs one Gram, one chain, one lambda and a warm start");
        a.irls_conv = pp.irls_conv; a.irls_host_flag = pp.irls_host_flag; a.irls_iters_total = pp.irls_iters_total;
        a.irls_tol = pp.irls_tol; a.irls_cinv = pp.irls_cinv; a.irls_p = pp.irls_p; a.irls_icpt = pp.irls_icpt;
        a.irls_b = pp.irls_b; a.irls_b0 = pp.irls_b0;
    }

    if (pp.xy_grad) {
        if (G != 1 || pp.chains.size() != 1 || !pp.xy_out || pp.xy_out != pp.XY || !pp.beta_init)
            fail(OEMB200_EINVAL, "path: xy_grad needs one Gram, one chain, a warm start and xy_out == XY");
        if (rpt > 0) {
            a.xy_grad = pp.xy_grad; a.xy_cinv = pp.xy_cinv; a.xy_n = pp.xy_n; a.xy_icpt = pp.xy_icpt; a.xy_out = pp.xy_out;
        } else {
            path_xy_launch(cx, q, pp.xy_icpt, pp.XX, pp.beta_init + (size_t)pp.chains[0].out_off * q, pp.xy_grad, pp.xy_cinv, pp.xy_n,
                           pp.xy_out, pp.skip);
        }
    }

    DBuf<long long> d_prof;
    const bool prof = getenv("OEMB200_PATH_PROF") != nullptr;
    if (prof) { d_prof.alloc(32); d_prof.zero(cx.stream); a.prof = d_prof.p; }
    void *kargs[] = {&a};
    if (mode == MODE_GLOBAL) {
        OEM_CUDA(cudaLaunchCooperativeKernel(kern, dim3(G * team), dim3(PK_THREADS), kargs, smem_bytes, cx.stream));
    } else {
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3(G * team); cfg.blockDim = dim3(PK_THREADS); cfg.dynamicSmemBytes = smem_bytes; cfg.stream = cx.stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = team; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        OEM_CUDA(cudaLaunchKernelExC(&cfg, kern, kargs));
    }
    cx.st.kernel_launches += 1;
    if (prof) {
        long long h[32];
        d_prof.download(h, 32, cx.stream);
        OEM_CUDA(cudaStreamSynchronize(cx.stream));
        fprintf(stderr, "[path prof] mode=%d rpt=%d team=%d cpc=%d q=%d nct=%d | iters=%lld cyc/iter: matvec=%.0f exchange=%.0f prox+update=%.0f | "
                "lanczos: steps=%lld total=%lld cyc (tridiag %lld)\n", mode, rpt, team, cpc, q, max_ct, h[3],
                h[3] ? (double)h[0] / h[3] : 0.0, h[3] ? (double)h[1] / h[3] : 0.0, h[3] ? (double)h[2] / h[3] : 0.0, h[6], h[4], h[5]);
        if (h[3]) fprintf(stderr, "[path prof]   flags=%.0f replicated=%.0f reduce=%.0f finished=%.0f state=%.0f | matvec: kloop=%.0f butterfly|sync=%.0f "
                          "reduce+prox+publish=%.0f (reg: sync %.0f) | team barrier=%.0f of the exchange, %lld iterations without a finished chain\n", (double)h[8] / h[3],
                          (double)h[9] / h[3], (double)h[10] / h[3], (double)h[11] / h[3], (double)h[12] / h[3],
                          (double)h[13] / h[3], (double)h[14] / h[3], (double)h[15] / h[3], (double)h[7] / h[3], (double)h[17] / h[3], h[16]);
    }
}

}  // namespace oemb200
