// gram_syrk.cu -- symmetric lower-triangle FP64 Gram  G = X' diag(w) X  over row tiles of a
// column-major n x p matrix, on the FP64 tensor pipe (mma.sync m8n8k4 -> SASS DMMA.8x8x4),
// operands staged into shared memory by TMA (cp.async.bulk.tensor -> SASS UTMALDG).
//
// Replaces (paths relative to the reference tree):
//   oemDense::XtX()              src/oem_dense.h:318-361   (incl. the OpenMP row-slice sum :328-358)
//   oemBig::XtX() sliced         src/oem_big.h:319-361
//   oemLogisticDense::XtWX()     src/oem_logistic_dense.h:334-381
//   oemXvalDense::XtX_xval       src/oem_xval_dense.h:358-484  (per-fold Grams = row segments here)
// and fuses DataStd's column centring (src/DataStd.h:216-261) into the fragment load.
//
// Layout.  X is column-major, so for G = X'X the contraction index (rows) is the contiguous one
// for BOTH mma operands.  A TMA box is [KT rows x 128 columns]; it lands in shared memory as a
// dense column-major panel with column stride KT = 36 doubles.  36 = 4 (mod 16) makes the
// 64-bit fragment loads (lane -> column 8*atom + lane/4, row 4*kstep + lane%4) hit 16 distinct
// bank pairs per half-warp: conflict-free without swizzling.
//
// Work decomposition.  Output tile = 128 x 128 (pair of column panels pi >= pj), 8 consumer warps
// in a 2 x 4 grid with 64 x 32 warp tiles (64 accumulator doubles per thread); thread 0 doubles as the
// TMA producer (a 9th warp would cap the kernel at 168 registers).  Diagonal tiles (pi == pj) compute
// only their lower triangle: warp w owns atom rows w and 15-w of the 16 x 16 atom grid (17 atoms each),
// so a diagonal tile costs 17/32 of an off-diagonal one instead of wasting its upper half.
// A work item = (tile, row range); the host builds the item list row-range-major so CTAs that run
// together stream the same rows (panel reuse in L2).  Every item writes its partial tile to a
// workspace slot; gram_reduce_kernel sums the slots of a tile in a fixed order (deterministic,
// no atomics) and mirrors the lower triangle.
#include <algorithm>
#include <functional>
#include <type_traits>
#include <mutex>
#include "runtime.h"

namespace oemb200 {

constexpr int G_TILE = 128;
constexpr int G_KT = 36;
constexpr int G_KSTEPS = G_KT / 4;
constexpr int G_STAGES = 3;
constexpr int G_CWARPS = 8;
constexpr int G_THREADS = G_CWARPS * 32;   // 9 warps would cap ptxas at 168 regs (4-warp allocation granularity)
constexpr int G_PANEL = G_TILE * G_KT;                       // doubles per panel
constexpr int G_PANEL_BYTES = G_PANEL * 8;                   // 36864
constexpr int G_STAGE_BYTES = 2 * G_PANEL_BYTES;             // 73728
constexpr int G_SMEM_BYTES = G_STAGES * G_STAGE_BYTES + 128; // + barriers

int gram_kt() { return G_KT; }

struct GramItem {
    int pi, pj, slot, pad;
    long long row0, row1;
};
struct GramTile {
    int pi, pj, slot0, nslots, out, pad;
};

// STATS: the diagonal-tile CTAs also accumulate, for the 128 columns of their panel, sum x and sum x*y over the item's
// rows (the column sweeps of src/oem_big.h:743-837; sum x^2 is the Gram's own diagonal) from the A fragments they load
// anyway: warp w owns atom rows w and 15-w, so the 8 warps cover the panel's 16 column atoms exactly once.  A separate
// HBM sweep of X (colstats_kernel) is no longer needed.  The statistics are those of the raw columns: STATS excludes
// CENTER and WEIGHT (gram_launch refuses the combinations).
template <bool CENTER, bool WEIGHT, bool USE_TMA, bool STATS>
__global__ void __launch_bounds__(G_THREADS, 1)
gram_syrk_kernel(const __grid_constant__ CUtensorMap tmap, const double *__restrict__ X, long long ld,
                 long long nrows, int q, const GramItem *__restrict__ items, const double *__restrict__ mean,
                 const double *__restrict__ roww, double *__restrict__ ws, const double *__restrict__ yvec,
                 double *__restrict__ stats_ws, int npanels) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *panels = reinterpret_cast<double *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + G_STAGES * G_STAGE_BYTES);
    uint64_t *empty = full + G_STAGES;

    const GramItem it = items[blockIdx.x];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool diag = (it.pi == it.pj);
    const int nk = static_cast<int>((it.row1 - it.row0 + G_KT - 1) / G_KT);

    if (threadIdx.x == 0) {
        for (int s = 0; s < G_STAGES; ++s) {
            mbar_init(&full[s], USE_TMA ? 1 : G_CWARPS);
            mbar_init(&empty[s], G_CWARPS);
        }
        mbar_fence_init();
        if (USE_TMA) tma_prefetch_desc(&tmap);
    }
    __syncthreads();

    // Stage loader.  TMA mode: one elected thread arms the barrier and issues two box loads.
    // Fallback mode (odd leading dimension / unaligned base): the 8 warps copy 1/8 of the panels each.
    auto load_tile = [&](int kt) {
        const int s = kt % G_STAGES;
        double *pa = panels + (size_t)s * 2 * G_PANEL;
        const long long r0 = it.row0 + (long long)kt * G_KT;
        if (USE_TMA) {
            if (threadIdx.x == 0) {
                mbar_arrive_expect_tx(&full[s], diag ? G_PANEL_BYTES : 2 * G_PANEL_BYTES);
                tma_load_2d(pa, &tmap, &full[s], static_cast<int>(r0), it.pi * G_TILE);
                if (!diag) tma_load_2d(pa + G_PANEL, &tmap, &full[s], static_cast<int>(r0), it.pj * G_TILE);
            }
        } else {
            const int npan = diag ? 1 : 2;
            for (int pn = 0; pn < npan; ++pn) {
                const int c0 = (pn == 0 ? it.pi : it.pj) * G_TILE;
                double *dst = pa + pn * G_PANEL;
                for (int e = threadIdx.x; e < G_PANEL; e += G_THREADS) {
                    const int c = e / G_KT, r = e - c * G_KT;
                    const long long gr = r0 + r;
                    const int gc = c0 + c;
                    dst[e] = (gr < nrows && gc < q) ? X[(size_t)gc * ld + gr] : 0.0;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
        }
    };
    for (int kt = 0; kt < G_STAGES && kt < nk; ++kt) load_tile(kt);

    // ===================== consumer warps =====================
    const int g = lane >> 2, t = lane & 3;
    if (!diag) {
    const int wm = warp >> 2, wn = warp & 3;
    int offA[8], offB[4];
#pragma unroll
    for (int ma = 0; ma < 8; ++ma) offA[ma] = (wm * 64 + ma * 8 + g) * G_KT + t;
#pragma unroll
    for (int na = 0; na < 4; ++na) offB[na] = (wn * 32 + na * 8 + g) * G_KT + t;

    double mA[8], mB[4];
    if (CENTER) {
#pragma unroll
        for (int ma = 0; ma < 8; ++ma) {
            const int c = it.pi * G_TILE + wm * 64 + ma * 8 + g;
            mA[ma] = c < q ? mean[c] : 0.0;
        }
#pragma unroll
        for (int na = 0; na < 4; ++na) {
            const int c = it.pj * G_TILE + wn * 32 + na * 8 + g;
            mB[na] = c < q ? mean[c] : 0.0;
        }
    }

    double acc[8][4][2];
#pragma unroll
    for (int ma = 0; ma < 8; ++ma)
#pragma unroll
        for (int na = 0; na < 4; ++na) acc[ma][na][0] = acc[ma][na][1] = 0.0;

    // Row atoms of the last panel beyond q are padding: a warp skips them (warp-uniform), which frees issue slots on
    // its scheduler for the other warp that shares it (warps w and w+4 = the two row halves of one column quarter).
    const int mav = max(0, min(8, (q - it.pi * G_TILE - wm * 64 + 7) >> 3));
    auto run = [&](auto full_tag) {
    constexpr int MAV = decltype(full_tag)::value;      // row atoms this warp computes (compile-time: keeps the
                                                        // straight-line LDS / DMMA schedule of the full tile)
    for (int kt = 0; kt < nk; ++kt) {
        const int s = kt % G_STAGES;
        const uint32_t ph = (kt / G_STAGES) & 1;
        const long long rbase = it.row0 + (long long)kt * G_KT + t;
        double wv[G_KSTEPS];
        if (WEIGHT) {
#pragma unroll
            for (int ks = 0; ks < G_KSTEPS; ++ks) {
                const long long r = rbase + ks * 4;
                wv[ks] = r < nrows ? __ldg(roww + r) : 0.0;
            }
        }
        const bool tail = CENTER && (it.row0 + (long long)(kt + 1) * G_KT > nrows);
        mbar_wait(&full[s], ph);
        const double *pA = panels + (size_t)s * 2 * G_PANEL;
        const double *pB = diag ? pA : pA + G_PANEL;
#pragma unroll
        for (int ks = 0; ks < G_KSTEPS; ++ks) {
            double a[8], b[4];
#pragma unroll
            for (int ma = 0; ma < 8; ++ma)
                if (ma < MAV) a[ma] = pA[offA[ma] + ks * 4];
#pragma unroll
            for (int na = 0; na < 4; ++na) b[na] = pB[offB[na] + ks * 4];
            if (CENTER) {
#pragma unroll
                for (int ma = 0; ma < 8; ++ma)
                    if (ma < MAV) a[ma] -= mA[ma];
                const bool valid = !tail || (rbase + ks * 4 < nrows);
#pragma unroll
                for (int na = 0; na < 4; ++na) b[na] = valid ? b[na] - mB[na] : 0.0;
            }
            if (WEIGHT) {
#pragma unroll
                for (int na = 0; na < 4; ++na) b[na] *= wv[ks];
            }
#pragma unroll
            for (int ma = 0; ma < 8; ++ma)
                if (ma < MAV) {
#pragma unroll
                    for (int na = 0; na < 4; ++na) dmma884(acc[ma][na][0], acc[ma][na][1], a[ma], b[na]);
                }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        // refill the stage just released with k-tile kt + STAGES once all 8 warps have let go of it
        if (kt + G_STAGES < nk) {
            if (USE_TMA) {
                if (threadIdx.x == 0) {
                    mbar_wait(&empty[s], ph);
                    load_tile(kt + G_STAGES);
                }
            } else {
                mbar_wait(&empty[s], ph);
                load_tile(kt + G_STAGES);
            }
        }
    }
    };
    switch (mav) {
        case 8: run(std::integral_constant<int, 8>{}); break;
        case 7: run(std::integral_constant<int, 7>{}); break;
        case 6: run(std::integral_constant<int, 6>{}); break;
        case 5: run(std::integral_constant<int, 5>{}); break;
        case 4: run(std::integral_constant<int, 4>{}); break;
        case 3: run(std::integral_constant<int, 3>{}); break;
        case 2: run(std::integral_constant<int, 2>{}); break;
        case 1: run(std::integral_constant<int, 1>{}); break;
        default: run(std::integral_constant<int, 0>{}); break;      // all padding: only keeps the barriers moving
    }

    // epilogue: partial tile -> workspace slot, [j][i] with i (panel pi column) contiguous
    double *slot = ws + (size_t)it.slot * (G_TILE * G_TILE);
#pragma unroll
    for (int ma = 0; ma < 8; ++ma) {
        const int i = wm * 64 + ma * 8 + g;
#pragma unroll
        for (int na = 0; na < 4; ++na) {
            const int j = wn * 32 + na * 8 + 2 * t;
            slot[(size_t)j * G_TILE + i] = acc[ma][na][0];
            slot[(size_t)(j + 1) * G_TILE + i] = acc[ma][na][1];
        }
    }
        return;
    }

    // ===================== diagonal tile: lower triangle only =====================
    // The 128 x 128 tile is 16 x 16 atoms of 8 x 8; only the 136 atoms on or below the diagonal are needed.
    // Warp w takes atom rows w and 15-w: (w+1) + (16-w) = 17 atoms each, a perfectly balanced triangle.
    // Slot s < = w is atom (w, s); slot s > w is atom (15-w, s-w-1).
    {
        const int rlo = warp, rhi = 15 - warp;
        const int offAlo = (rlo * 8 + g) * G_KT + t, offAhi = (rhi * 8 + g) * G_KT + t;
        int offS[17];
#pragma unroll
        for (int sl = 0; sl < 17; ++sl) {
            const int col = sl <= warp ? sl : sl - warp - 1;
            offS[sl] = (col * 8 + g) * G_KT + t;
        }
        double mlo = 0.0, mhi = 0.0, mS[17];
        if (CENTER) {
            const int clo = it.pi * G_TILE + rlo * 8 + g, chi = it.pi * G_TILE + rhi * 8 + g;
            mlo = clo < q ? mean[clo] : 0.0;
            mhi = chi < q ? mean[chi] : 0.0;
#pragma unroll
            for (int sl = 0; sl < 17; ++sl) {
                const int col = sl <= warp ? sl : sl - warp - 1;
                const int c = it.pi * G_TILE + col * 8 + g;
                mS[sl] = c < q ? mean[c] : 0.0;
            }
        }
        double acc[17][2];
#pragma unroll
        for (int sl = 0; sl < 17; ++sl) acc[sl][0] = acc[sl][1] = 0.0;
        double st_lo[2] = {0.0, 0.0}, st_hi[2] = {0.0, 0.0};      // sum x, sum x*y of my two columns
        double ynext[G_KSTEPS];
        if (STATS) {
#pragma unroll
            for (int ks = 0; ks < G_KSTEPS; ++ks) {
                const long long r = it.row0 + t + ks * 4;
                ynext[ks] = (yvec && r < it.row1) ? __ldg(yvec + r) : 0.0;
            }
        }

        for (int kt = 0; kt < nk; ++kt) {
            const int s = kt % G_STAGES;
            const uint32_t ph = (kt / G_STAGES) & 1;
            const long long rbase = it.row0 + (long long)kt * G_KT + t;
            double wv[G_KSTEPS];
            if (WEIGHT) {
#pragma unroll
                for (int ks = 0; ks < G_KSTEPS; ++ks) {
                    const long long r = rbase + ks * 4;
                    wv[ks] = r < nrows ? __ldg(roww + r) : 0.0;
                }
            }
            double yv[G_KSTEPS];
            if (STATS) {      // y of this k-tile was requested one k-tile ago; request the next one now
#pragma unroll
                for (int ks = 0; ks < G_KSTEPS; ++ks) {
                    yv[ks] = ynext[ks];
                    const long long r = rbase + G_KT + ks * 4;
                    ynext[ks] = (yvec && r < it.row1) ? __ldg(yvec + r) : 0.0;
                }
            }
            const bool tail = CENTER && (it.row0 + (long long)(kt + 1) * G_KT > nrows);
            mbar_wait(&full[s], ph);
            const double *pA = panels + (size_t)s * 2 * G_PANEL;
#pragma unroll
            for (int ks = 0; ks < G_KSTEPS; ++ks) {
                double alo = pA[offAlo + ks * 4], ahi = pA[offAhi + ks * 4];
                const bool valid = !tail || (rbase + ks * 4 < nrows);
                if (CENTER) { alo -= mlo; ahi -= mhi; }
                if (STATS) {
                    // rows past the item's end only occur in the matrix's last k-tile, where the loader zero-fills them
                    st_lo[0] += alo; st_lo[1] = fma(alo, yv[ks], st_lo[1]);       // sum x^2 is the Gram's own diagonal
                    st_hi[0] += ahi; st_hi[1] = fma(ahi, yv[ks], st_hi[1]);
                }
                if (WEIGHT) { alo *= wv[ks]; ahi *= wv[ks]; }
#pragma unroll
                for (int sl = 0; sl < 17; ++sl) {
                    double b = pA[offS[sl] + ks * 4];
                    if (CENTER) b = valid ? b - mS[sl] : 0.0;
                    dmma884(acc[sl][0], acc[sl][1], sl <= warp ? alo : ahi, b);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (kt + G_STAGES < nk) {
                if (USE_TMA) {
                    if (threadIdx.x == 0) {
                        mbar_wait(&empty[s], ph);
                        load_tile(kt + G_STAGES);
                    }
                } else {
                    mbar_wait(&empty[s], ph);
                    load_tile(kt + G_STAGES);
                }
            }
        }
        if (STATS) {
            // fixed-order sum over the 4 row lanes t of each column, then one partial per (row chunk, panel)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                st_lo[e] += __shfl_xor_sync(0xffffffffu, st_lo[e], 1);
                st_lo[e] += __shfl_xor_sync(0xffffffffu, st_lo[e], 2);
                st_hi[e] += __shfl_xor_sync(0xffffffffu, st_hi[e], 1);
                st_hi[e] += __shfl_xor_sync(0xffffffffu, st_hi[e], 2);
            }
            if (t == 0) {
                double *so = stats_ws + ((size_t)it.pad * npanels + it.pi) * (2 * G_TILE);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    so[e * G_TILE + rlo * 8 + g] = st_lo[e];
                    so[e * G_TILE + rhi * 8 + g] = st_hi[e];
                }
            }
        }
        double *slot = ws + (size_t)it.slot * (G_TILE * G_TILE);
#pragma unroll
        for (int sl = 0; sl < 17; ++sl) {
            const int row = sl <= warp ? rlo : rhi;
            const int col = sl <= warp ? sl : sl - warp - 1;
            const int i = row * 8 + g, j = col * 8 + 2 * t;
            slot[(size_t)j * G_TILE + i] = acc[sl][0];
            slot[(size_t)(j + 1) * G_TILE + i] = acc[sl][1];
        }
    }
}

// Fixed-order sum of a tile's partial slots; writes lower triangle and its mirror.
__global__ void __launch_bounds__(256)
gram_reduce_kernel(const double *__restrict__ ws, const GramTile *__restrict__ tiles, double *__restrict__ G, int q,
                   int accumulate) {
    const GramTile tl = tiles[blockIdx.y];
    const int e = blockIdx.x * 256 + threadIdx.x;
    const int i = e & (G_TILE - 1), j = e >> 7;
    const int gi = tl.pi * G_TILE + i, gj = tl.pj * G_TILE + j;
    if (gi >= q || gj >= q || gi < gj) return;
    const double *p = ws + (size_t)tl.slot0 * (G_TILE * G_TILE) + e;
    double s = 0.0;
    for (int k = 0; k < tl.nslots; ++k) s += p[(size_t)k * (G_TILE * G_TILE)];
    double *Go = G + (size_t)tl.out * q * q;
    if (accumulate) s += Go[(size_t)gj * q + gi];
    Go[(size_t)gj * q + gi] = s;
    Go[(size_t)gi * q + gj] = s;
}

// stats_out[o][e][j] (+)= sum over the row chunks of output o (in chunk order) of the diagonal CTAs' partial sums for
// e = 0 (sum x) and 1 (sum x*y); e = 2 (sum x^2) is the diagonal of the finished Gram G[o] (runs after gram_reduce_kernel)
__global__ void gram_stats_reduce_kernel(const double *__restrict__ stats_ws, const int *__restrict__ chunk_out, int nchunks,
                                         int npanels, int q, int nout, const double *__restrict__ G,
                                         double *__restrict__ stats_out, int accumulate) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int o = blockIdx.y;
    if (j >= q) return;
    const int pi = j / G_TILE, jl = j - pi * G_TILE;
    double s[2] = {0.0, 0.0};
    for (int c = 0; c < nchunks; ++c) {
        if (chunk_out[c] != o) continue;
        const double *so = stats_ws + ((size_t)c * npanels + pi) * (2 * G_TILE) + jl;
#pragma unroll
        for (int e = 0; e < 2; ++e) s[e] += so[e * G_TILE];
    }
    double *out = stats_out + (size_t)o * 3 * q;
#pragma unroll
    for (int e = 0; e < 2; ++e) out[(size_t)e * q + j] = accumulate ? out[(size_t)e * q + j] + s[e] : s[e];
    out[(size_t)2 * q + j] = G[(size_t)o * q * q + (size_t)j * q + j];
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

template <bool C, bool W, bool T, bool S>
static void launch_variant(Ctx &cx, const CUtensorMap &tm, const double *X, int64_t ld, int64_t n, int q,
                           const GramItem *d_items, int nitems, const double *mean, const double *roww, double *ws,
                           const double *yvec, double *stats_ws, int npanels) {
    auto kern = gram_syrk_kernel<C, W, T, S>;
    OEM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, G_SMEM_BYTES));
    kern<<<nitems, G_THREADS, G_SMEM_BYTES, cx.stream>>>(tm, X, ld, n, q, d_items, mean, roww, ws, yvec, stats_ws, npanels);
    OEM_CUDA(cudaGetLastError());
}

void gram_launch(Ctx &cx, const double *X, int64_t n, int q, int64_t ld, const std::vector<RowSegment> &segs,
                 int nout, const double *mean, const double *roww, double *G, bool accumulate, const double *stats_y,
                 double *stats_out) {
    if (stats_out && roww) fail(OEMB200_EINVAL, "gram: fused column statistics are not available with row weights");
    if (stats_out && mean) fail(OEMB200_EINVAL, "gram: fused column statistics are not available with centring");
    if (n <= 0 || q <= 0) fail(OEMB200_EINVAL, "gram: empty matrix (n=%lld, p=%d)", (long long)n, q);
    if (n >= (1ll << 31)) fail(OEMB200_EINVAL, "gram: more than 2^31-1 rows per call; shard or chunk the rows");
    const int P = (q + G_TILE - 1) / G_TILE;
    const int ntile_pairs = P * (P + 1) / 2;

    // ---- plan: split every segment into row chunks so that there are a few waves of items ----
    int64_t rows_total = 0;
    for (auto &s : segs) {
        if (s.row0 < 0 || s.row1 > n || s.row1 < s.row0 || s.out < 0 || s.out >= nout)
            fail(OEMB200_EINVAL, "gram: bad row segment");
        if ((s.row0 % G_KT) != 0 && s.row0 != 0) fail(OEMB200_EINVAL, "gram: segment start not a multiple of %d", G_KT);
        if (((s.row1 - s.row0) % G_KT) != 0 && s.row1 != n)
            fail(OEMB200_EINVAL, "gram: interior segment length not a multiple of %d", G_KT);
        rows_total += s.row1 - s.row0;
    }
    // Row-chunk length: a few waves of items, chosen by simulating the block scheduler (items in launch order onto the
    // earliest free SM) with the three tile-class costs, so that the class sizes divide well over the SMs and the tail
    // of cheap diagonal items is short.
    const int64_t min_rows = 32 * G_KT;
    auto round_chunk = [&](int64_t target_chunks) {
        int64_t cr = (rows_total + target_chunks - 1) / std::max<int64_t>(1, target_chunks);
        return std::max<int64_t>(min_rows, ((cr + G_KT - 1) / G_KT) * G_KT);
    };
    const bool partial = (q % G_TILE) != 0;
    const int nfull = partial ? (P - 1) * (P - 2) / 2 : P * (P - 1) / 2;       // tiles per class
    const int nlast = partial ? P - 1 : 0;
    const double cost_last = partial ? (8.0 + std::max(0, std::min(8, (q - (P - 1) * G_TILE - 64 + 7) / 8)) +
                                        std::min(8, (q - (P - 1) * G_TILE + 7) / 8) - 8.0) / 16.0 : 1.0;
    const double cost_diag = stats_out ? 0.60 : 0.54;
    auto makespan = [&](int64_t cr) {
        std::vector<double> cost;      // launch order: class by class, chunk-major
        std::vector<double> len;       // k-tiles (+3 for pipeline fill / epilogue) of every chunk
        for (auto &sg : segs) {
            const int64_t l = sg.row1 - sg.row0;
            if (l <= 0) continue;
            const int64_t nc = (l + cr - 1) / cr;
            const int64_t per = (((l + nc - 1) / nc) + G_KT - 1) / G_KT * G_KT;
            for (int64_t r = 0; r < l; r += per) len.push_back((double)((std::min(l, r + per) - r + G_KT - 1) / G_KT) + 3.0);
        }
        for (double c : {1.0, cost_last, cost_diag}) {
            const int nt = c == 1.0 ? nfull : (c == cost_diag ? P : nlast);
            for (double l : len)
                for (int t = 0; t < nt; ++t) cost.push_back(l * c);
        }
        std::vector<double> sm(cx.num_sms, 0.0);       // min-heap of SM free times
        std::make_heap(sm.begin(), sm.end(), std::greater<double>());
        double end = 0.0;
        for (double c : cost) {
            std::pop_heap(sm.begin(), sm.end(), std::greater<double>());
            sm.back() += c;
            end = std::max(end, sm.back());
            std::push_heap(sm.begin(), sm.end(), std::greater<double>());
        }
        return end;
    };
    const int64_t c_lo = std::max<int64_t>(1, (int64_t)6 * cx.num_sms / ntile_pairs);
    const int64_t c_hi = std::max<int64_t>(c_lo, (int64_t)14 * cx.num_sms / ntile_pairs);
    int64_t chunk_rows = round_chunk(c_lo);
    double best = makespan(chunk_rows);
    for (int64_t c = c_lo + 1; c <= c_hi; ++c) {
        const int64_t cr = round_chunk(c);
        if (cr == chunk_rows) continue;
        const double m = makespan(cr);
        if (m < best * 0.999) { best = m; chunk_rows = cr; }
    }
    // cap the workspace at ~1.5 GB of partial tiles
    const int64_t max_slots = (1536ll << 20) / (G_TILE * G_TILE * 8);
    for (;;) {
        int64_t nchunks = 0;
        for (auto &s : segs) nchunks += std::max<int64_t>(1, (s.row1 - s.row0 + chunk_rows - 1) / chunk_rows);
        if (nchunks * ntile_pairs <= max_slots) break;
        chunk_rows *= 2;
    }

    std::vector<GramItem> items;
    std::vector<GramTile> tiles;
    // slots of one (segment-out, tile) must be contiguous: slot = tilebase + chunk index
    // first count chunks per out
    std::vector<int> chunks_per_out(nout, 0);
    struct Chunk { int64_t r0, r1; int out, idx; };      // position in `chunks` = global chunk index (stats slot)
    std::vector<Chunk> chunks;
    for (auto &s : segs) {
        const int64_t len = s.row1 - s.row0;
        if (len == 0) continue;
        const int64_t nc = (len + chunk_rows - 1) / chunk_rows;
        // equal-size chunks, multiples of KT
        int64_t per = (((len + nc - 1) / nc) + G_KT - 1) / G_KT * G_KT;
        for (int64_t r = s.row0; r < s.row1; r += per) {
            Chunk c{r, std::min(s.row1, r + per), s.out, chunks_per_out[s.out]++};
            chunks.push_back(c);
        }
    }
    std::vector<int> out_base(nout + 1, 0);
    for (int o = 0; o < nout; ++o) out_base[o + 1] = out_base[o] + chunks_per_out[o] * ntile_pairs;
    const int nslots = out_base[nout];
    // Item order = launch order.  Tiles come in three cost classes (full off-diagonal 1.0, last-panel off-diagonal with
    // skipped padding, triangular diagonal ~0.6); CTAs of one class take equally long, so listing the items class by
    // class (row-range-major inside a class) makes the tiles of a row range start together and stream the same rows at
    // the same time -- that is what lets them share column panels through L2.  Mixed classes drift apart within a wave
    // and re-read the panels from HBM (measured 5.6x the matrix; class-major order: see profiles/gram_traffic.json).
    for (int cls = 0; cls < 3; ++cls)
        for (size_t ci = 0; ci < chunks.size(); ++ci) {
            const Chunk &c = chunks[ci];
            int tp = 0;
            for (int pi = 0; pi < P; ++pi)
                for (int pj = 0; pj <= pi; ++pj, ++tp) {
                    const int tcls = pi == pj ? 2 : (partial && pi == P - 1) ? 1 : 0;
                    if (tcls != cls) continue;
                    GramItem it;
                    it.pi = pi; it.pj = pj; it.pad = (int)ci;
                    it.slot = out_base[c.out] + tp * chunks_per_out[c.out] + c.idx;
                    it.row0 = c.r0; it.row1 = c.r1;
                    items.push_back(it);
                }
        }
    for (int o = 0; o < nout; ++o) {
        int tp = 0;
        for (int pi = 0; pi < P; ++pi)
            for (int pj = 0; pj <= pi; ++pj, ++tp) {
                GramTile tl;
                tl.pi = pi; tl.pj = pj; tl.pad = 0;
                tl.slot0 = out_base[o] + tp * chunks_per_out[o];
                tl.nslots = chunks_per_out[o];
                tl.out = o;
                tiles.push_back(tl);
            }
    }
    if (items.empty()) {
        if (!accumulate) {
            OEM_CUDA(cudaMemsetAsync(G, 0, (size_t)nout * q * q * 8, cx.stream));
            if (stats_out) OEM_CUDA(cudaMemsetAsync(stats_out, 0, (size_t)nout * 3 * q * 8, cx.stream));
        }
        return;
    }

    DBuf<GramItem> d_items(items.size());
    DBuf<GramTile> d_tiles(tiles.size());
    DBuf<double> ws((size_t)nslots * G_TILE * G_TILE);
    d_items.upload(items.data(), items.size(), cx.stream);
    d_tiles.upload(tiles.data(), tiles.size(), cx.stream);
    DBuf<double> stats_ws;
    DBuf<int> d_chunk_out;
    if (stats_out) {
        stats_ws.alloc(chunks.size() * (size_t)P * 2 * G_TILE);
        std::vector<int> co(chunks.size());
        for (size_t ci = 0; ci < chunks.size(); ++ci) co[ci] = chunks[ci].out;
        d_chunk_out.alloc(co.size());
        d_chunk_out.upload(co.data(), co.size(), cx.stream);
    }

    // ---- TMA descriptor (FP64, 2-D, box = 36 rows x 128 columns, no swizzle, zero OOB fill) ----
    CUtensorMap tm;
    memset(&tm, 0, sizeof tm);
    bool use_tma = (ld % 2 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && get_encode_fn() != nullptr;
    if (use_tma) {
        cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)q};
        cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
        cuuint32_t box[2] = {(cuuint32_t)G_KT, (cuuint32_t)G_TILE};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = get_encode_fn()(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(X), dims, strides,
                                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) use_tma = false;
    }

    const int ni = (int)items.size();
    const bool C = mean != nullptr, W = roww != nullptr;
    const size_t t_k = cx.tm->start(&cx.st.ms_gram);      // the DMMA kernel alone
#define OEM_GRAM_DISPATCH(CC, WW, SS)                                                                               \
    if (use_tma) launch_variant<CC, WW, true, SS>(cx, tm, X, ld, n, q, d_items.p, ni, mean, roww, ws.p, stats_y, stats_ws.p, P);  \
    else launch_variant<CC, WW, false, SS>(cx, tm, X, ld, n, q, d_items.p, ni, mean, roww, ws.p, stats_y, stats_ws.p, P)
    if (stats_out) { OEM_GRAM_DISPATCH(false, false, true); }
    else if (C && W) { OEM_GRAM_DISPATCH(true, true, false); }
    else if (C) { OEM_GRAM_DISPATCH(true, false, false); }
    else if (W) { OEM_GRAM_DISPATCH(false, true, false); }
    else { OEM_GRAM_DISPATCH(false, false, false); }
#undef OEM_GRAM_DISPATCH
    cx.tm->stop(t_k);
    const size_t t_r = cx.tm->start(&cx.st.ms_gram_reduce);

    dim3 rg(G_TILE * G_TILE / 256, (unsigned)tiles.size());
    gram_reduce_kernel<<<rg, 256, 0, cx.stream>>>(ws.p, d_tiles.p, G, q, accumulate ? 1 : 0);
    OEM_CUDA(cudaGetLastError());
    if (stats_out) {
        gram_stats_reduce_kernel<<<dim3((q + 127) / 128, nout), 128, 0, cx.stream>>>(
            stats_ws.p, d_chunk_out.p, (int)chunks.size(), P, q, nout, G, stats_out, accumulate ? 1 : 0);
        OEM_CUDA(cudaGetLastError());
        cx.st.kernel_launches += 1;
    }
    cx.tm->stop(t_r);
    cx.st.kernel_launches += 2;
    cx.st.gram_launches += 1;
    cx.st.gram_flops += (double)rows_total * q * (q + 1.0);
    // workspace / item lists go back to the pool on return; stream order protects them (runtime.h)
}

}  // namespace oemb200
