// assemble.cu -- O(q^2) glue between the data pass and the path kernel: turn raw sums
// (Gram, column sums, X'y, column sums of squares, counts) into the scaled XX, XY the OEM
// iteration runs on.  Three conventions exist in the reference (SURVEY.md Appendix A):
//
//   assemble_aug    explicit-intercept border + UNCENTRED scaling 1/sqrt(sum x^2/(n-1)):
//                   oemBig::compute_XtX_d_update_A      src/oem_big.h:469-566, init_oem :731-842
//                   oemXvalDense compute_/update_XtX_d_update_A   src/oem_xval_dense.h:667-853
//                   oemLogisticDense::compute_XtX_d_update_A      src/oem_logistic_dense.h:458-522
//   assemble_dense  DataStd centring / scaling folded into the Gram of centred columns:
//                   src/DataStd.h:94-267 + src/oem_dense.h:693-712,458-506
//   scale_sym       oem_xtx scale.factor: XX <- D^-1 XX D^-1, XY <- XY / s   src/oem_xtx.h:349-356,526-533
#include "runtime.h"

namespace oemb200 {

// out o uses all parts except part (o-1) (o = 0: all parts).  One thread per element of XX.
__global__ void assemble_aug_kernel(int p, int intercept, int standardize, int nparts, const double *__restrict__ G,
                                    const double *__restrict__ stats, const double *__restrict__ ysum, int ysum_stride,
                                    const double *__restrict__ corner, const double *__restrict__ nobs,
                                    double *__restrict__ XX, double *__restrict__ XY, double *__restrict__ colsq_inv,
                                    double *__restrict__ nobs_out) {
    const int q = p + intercept;
    const int o = blockIdx.y;
    const int skip = o - 1;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)q * q) return;
    const int r = (int)(e % q), c = (int)(e / q);
    double ns = 0.0;
    for (int k = 0; k < nparts; ++k)
        if (k != skip) ns += nobs[k];
    auto winv = [&](int j) -> double {
        if (!standardize) return 1.0;
        double sq = 0.0;
        for (int k = 0; k < nparts; ++k)
            if (k != skip) sq += stats[((size_t)k * 3 + 2) * p + j];
        sq = sq / (ns - 1.0);
        if (sq == 0.0) sq = 1.0;
        return 1.0 / sqrt(sq);
    };
    const int xr = r - intercept, xc = c - intercept;   // -1 = the intercept row / column
    double val;
    if (xr >= 0 && xc >= 0) {
        double g = 0.0;
        for (int k = 0; k < nparts; ++k)
            if (k != skip) g += G[((size_t)k * p + xc) * p + xr];
        val = standardize ? (winv(xr) * g) * winv(xc) : g;
    } else if (xr < 0 && xc < 0) {
        double g = 0.0;
        for (int k = 0; k < nparts; ++k)
            if (k != skip) g += corner[k];
        val = g;
    } else {
        const int j = xr < 0 ? xc : xr;
        double g = 0.0;
        for (int k = 0; k < nparts; ++k)
            if (k != skip) g += stats[((size_t)k * 3 + 0) * p + j];
        val = standardize ? g * winv(j) : g;
    }
    XX[(size_t)o * q * q + e] = val / ns;
    if (c == 0) {   // first column's threads also emit XY, colsq_inv, nobs
        if (XY) {
            double b = 0.0;
            if (xr < 0) {
                for (int k = 0; k < nparts; ++k)
                    if (k != skip) b += ysum[(size_t)k * ysum_stride];
            } else {
                for (int k = 0; k < nparts; ++k)
                    if (k != skip) b += stats[((size_t)k * 3 + 1) * p + xr];
                if (standardize) b *= winv(xr);
            }
            XY[(size_t)o * q + r] = b / ns;
        }
        if (xr >= 0 && colsq_inv) colsq_inv[(size_t)o * p + xr] = winv(xr);
        if (r == 0 && nobs_out) nobs_out[o] = ns;
    }
}

void assemble_aug_launch(Ctx &cx, int p, int intercept, int standardize, int nparts, int nout, const double *G_parts,
                         const double *stats_parts, const double *ysum_parts, int ysum_stride, const double *corner_parts,
                         const double *nobs_parts, double *XX, double *XY, double *colsq_inv, double *nobs_out) {
    const int q = p + intercept;
    dim3 grid((unsigned)(((long long)q * q + 255) / 256), nout);
    assemble_aug_kernel<<<grid, 256, 0, cx.stream>>>(p, intercept, standardize, nparts, G_parts, stats_parts,
                                                    ysum_parts, ysum_stride, corner_parts, nobs_parts, XX, XY, colsq_inv, nobs_out);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

// flag = standardize + 2*intercept.  G: Gram of raw (flag 0,1) or centred (flag 2,3) columns.
// xy: sum_i xs_ij ys_i with the same centring.  css: centred sums of squares (flag 1 only).
__global__ void assemble_dense_kernel(int p, int flag, double n, const double *__restrict__ G,
                                      const double *__restrict__ xy, const double *__restrict__ css,
                                      double *__restrict__ XX, double *__restrict__ XY, double *__restrict__ scalex) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)p * p) return;
    const int r = (int)(e % p), c = (int)(e / p);
    const double n_invsqrt = 1.0 / sqrt(n);
    auto sc = [&](int j) -> double {
        double s = 1.0;
        if (flag == 1) s = sqrt(css[j]) / sqrt(n);                    // sd_n: ||x - mean|| / sqrt(n)
        else if (flag == 3) s = sqrt(G[(size_t)j * p + j]) * n_invsqrt;   // ||x_c|| * n_invsqrt
        if (s == 0.0) s = 1.0;
        return s;
    };
    double val = G[e];
    if (flag == 1) val = (val * (1.0 / sc(r))) * (1.0 / sc(c));
    else if (flag == 3) val = (val / sc(r)) / sc(c);
    XX[e] = val / n;
    if (c == 0) {
        double b = xy[r];
        if (flag == 1) b *= (1.0 / sc(r));
        else if (flag == 3) b /= sc(r);
        XY[r] = b / n;
        scalex[r] = sc(r);
    }
}

void assemble_dense_launch(Ctx &cx, int p, int flag, double n, const double *G, const double *xy, const double *css,
                           double *XX, double *XY, double *scalex) {
    assemble_dense_kernel<<<(unsigned)(((long long)p * p + 255) / 256), 256, 0, cx.stream>>>(p, flag, n, G, xy, css,
                                                                                           XX, XY, scalex);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

__global__ void scale_sym_kernel(int p, const double *__restrict__ sinv, const double *__restrict__ XXin,
                                 const double *__restrict__ XYin, double *__restrict__ XX, double *__restrict__ XY) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)p * p) return;
    const int r = (int)(e % p), c = (int)(e / p);
    XX[e] = sinv ? (sinv[r] * XXin[e]) * sinv[c] : XXin[e];
    if (c == 0) XY[r] = sinv ? XYin[r] * sinv[r] : XYin[r];
}

void scale_sym_launch(Ctx &cx, int p, const double *sinv, const double *XXin, const double *XYin, double *XX,
                      double *XY) {
    scale_sym_kernel<<<(unsigned)(((long long)p * p + 255) / 256), 256, 0, cx.stream>>>(p, sinv, XXin, XYin, XX, XY);
    OEM_CUDA(cudaGetLastError());
    cx.st.kernel_launches += 1;
}

}  // namespace oemb200
