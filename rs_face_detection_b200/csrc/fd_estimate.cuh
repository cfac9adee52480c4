// fd_estimate.cuh — cv::estimateAffinePartial2D(from, to, LMEDS, 3.0, 2000, 0.99, 10) for 5 point pairs as device code
// (face_alignment.rs:50-59), shared by estimate_kernel (fd_align.cu) and the fused post-CNN kernel (fd_detect_fused.cu).
// fp64, the operation order of OpenCV's calib3d/ptsetreg.cpp: RNG reseeded per call, exact 2-point similarity per LMedS
// iteration, float32 squared errors, median, inlier threshold, then the least-squares similarity over the inliers that
// OpenCV's LM refinement converges to.
#pragma once
#include <cfloat>
#include "fd_internal.cuh"

namespace fd {

constexpr int EST_LANES = 16;   // lanes per face: lane k < niters evaluates LMedS iteration k

struct EstConst {
    float tmpl[10];               // destination points when none are given (ArcFace template, config.rs:46-52)
    int niters;                   // <= EST_LANES
    int8_t pair0[16], pair1[16];  // LMedS sample pairs per iteration (host-precomputed from OpenCV's RNG)
};
int make_est_const(const fd_ctx *ctx, EstConst *out);   // host

#ifdef __CUDACC__
// v[2 * i + o] for a runtime point index i < 5, by selects: indexing the caller's register arrays directly would move them
// to local memory
__device__ __forceinline__ float pick_pt(const float *v, int i, int o) {
    float r = v[o];
#pragma unroll
    for (int k = 1; k < 5; ++k) r = i == k ? v[2 * k + o] : r;
    return r;
}
__device__ __forceinline__ void fit2(const float *f, const float *t, int i0, int i1, double *M) {
    double x1 = pick_pt(f, i0, 0), y1 = pick_pt(f, i0, 1), x2 = pick_pt(f, i1, 0), y2 = pick_pt(f, i1, 1);
    double X1 = pick_pt(t, i0, 0), Y1 = pick_pt(t, i0, 1), X2 = pick_pt(t, i1, 0), Y2 = pick_pt(t, i1, 1);
    double d = 1. / ((x1 - x2) * (x1 - x2) + (y1 - y2) * (y1 - y2));
    double S0 = d * ((X1 - X2) * (x1 - x2) + (Y1 - Y2) * (y1 - y2));
    double S1 = d * ((Y1 - Y2) * (x1 - x2) - (X1 - X2) * (y1 - y2));
    double S2 = d * ((Y1 - Y2) * (x1 * y2 - x2 * y1) - (X1 * y2 - X2 * y1) * (y1 - y2) - (X1 * x2 - X2 * x1) * (x1 - x2));
    double S3 = d * (-(X1 - X2) * (x1 * y2 - x2 * y1) - (Y1 * x2 - Y2 * x1) * (x1 - x2) - (Y1 * y2 - Y2 * y1) * (y1 - y2));
    M[0] = S0; M[1] = -S1; M[2] = S2; M[3] = S1; M[4] = S0; M[5] = S3;
}
__device__ __forceinline__ void affine_err5(const float *f, const float *t, const double *M, float *err) {
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        double a = M[0] * f[2 * i] + M[1] * f[2 * i + 1] + M[2] - t[2 * i];
        double b = M[3] * f[2 * i] + M[4] * f[2 * i + 1] + M[5] - t[2 * i + 1];
        err[i] = (float)(a * a + b * b);
    }
}
__device__ __forceinline__ void invert_affine(const double *M, double *iM) {
    double D = M[0] * M[4] - M[1] * M[3];
    D = D != 0 ? 1. / D : 0;
    double A11 = M[4] * D, A22 = M[0] * D;
    iM[0] = A11; iM[1] = M[1] * (-D); iM[3] = M[3] * (-D); iM[4] = A22;
    iM[2] = -iM[0] * M[2] - iM[1] * M[5];
    iM[5] = -iM[3] * M[2] - iM[4] * M[5];
}

// One face per group of EST_LANES lanes; EVERY lane of the warp must call (shuffles).  live: this group has a face.
// sub = lane index inside the group.  Lane k < niters fits iteration k's 2-point model and takes the median of the 5
// float32 errors; a lexicographic (median, iteration) min over the group picks the model the sequential loop would have
// kept (first strictly smaller median wins).  The group's lane 0 (and only it) receives M, its inverse and ok.
__device__ __forceinline__ void estimate_group(const EstConst &ec, const float *from, const float *to, bool live, int sub,
                                               double *M, double *iM, bool &ok_out) {
    const int n = 5;
    double model[6] = {0, 0, 0, 0, 0, 0};
    double median = DBL_MAX;
    float err[5];
    if (live && sub < ec.niters) {
        fit2(from, to, ec.pair0[sub], ec.pair1[sub], model);
        bool finite = true;
#pragma unroll
        for (int k = 0; k < 6; ++k) finite &= isfinite(model[k]);
        if (finite) {
            affine_err5(from, to, model, err);
            // median of 5 by a min/max network (registers only; the errors are never NaN for a finite model)
            float e0 = err[0], e1 = err[1], e2 = err[2], e3 = err[3], e4 = err[4], t;
            t = fminf(e0, e1); e1 = fmaxf(e0, e1); e0 = t;
            t = fminf(e3, e4); e4 = fmaxf(e3, e4); e3 = t;
            t = fmaxf(e0, e3); e3 = fminf(e0, e3); e0 = t;          // e3 = overall min of the two pairs' minima: discard
            t = fminf(e1, e4); e4 = fmaxf(e1, e4); e1 = t;          // e4 = overall max of the two pairs' maxima: discard
            // median of {e0, e1, e2}
            t = fminf(e0, e1); e1 = fmaxf(e0, e1); e0 = t;
            const float med3 = fmaxf(e0, fminf(e1, e2));
            (void)e3; (void)e4;
            const double med = (double)med3;
            if (med < DBL_MAX) median = med;  // NaN / inf medians never win (median < minMedian is false)
        }
    }
    int win = sub;
    double best_med = median;
#pragma unroll
    for (int o = EST_LANES / 2; o > 0; o >>= 1) {
        const double om = __shfl_xor_sync(0xffffffffu, best_med, o);
        const int ow = __shfl_xor_sync(0xffffffffu, win, o);
        if (om < best_med || (om == best_med && ow < win)) { best_med = om; win = ow; }
    }
    const int base_lane = (threadIdx.x & 31) & ~(EST_LANES - 1);
    double best[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) best[k] = __shfl_sync(0xffffffffu, model[k], base_lane + win);
    ok_out = false;
#pragma unroll
    for (int k = 0; k < 6; ++k) M[k] = 0;
    if (live && sub == 0) {
        const double minMedian = best_med;
        bool ok = minMedian < DBL_MAX;
        if (ok) {
            double sigma = 2.5 * 1.4826 * (1 + 5. / (n - 2)) * sqrt(minMedian);
            if (sigma < 0.001) sigma = 0.001;
            affine_err5(from, to, best, err);
            const float thr = (float)(sigma * sigma);
            bool mask[5];
            int good = 0;
#pragma unroll
            for (int i = 0; i < 5; ++i) { mask[i] = err[i] <= thr; good += mask[i]; }
            ok = good >= 2;
            if (ok) {
                // least squares over the inliers (fixed operation order; the test oracle performs the identical sequence)
                double sx = 0, sy = 0, sX = 0, sY = 0;
#pragma unroll
                for (int i = 0; i < 5; ++i) if (mask[i]) { sx += from[2 * i]; sy += from[2 * i + 1]; sX += to[2 * i]; sY += to[2 * i + 1]; }
                double mx = sx / good, my = sy / good, mX = sX / good, mY = sY / good;
                double num_a = 0, num_b = 0, den = 0;
#pragma unroll
                for (int i = 0; i < 5; ++i) if (mask[i]) {
                    double dx = from[2 * i] - mx, dy = from[2 * i + 1] - my, dX = to[2 * i] - mX, dY = to[2 * i + 1] - mY;
                    num_a += dx * dX + dy * dY;
                    num_b += dx * dY - dy * dX;
                    den += dx * dx + dy * dy;
                }
                double sa = num_a / den, sb = num_b / den;
                M[0] = sa; M[1] = -sb; M[2] = mX - (sa * mx - sb * my);
                M[3] = sb; M[4] = sa;  M[5] = mY - (sb * mx + sa * my);
            }
        }
        ok_out = ok;
    }
    invert_affine(M, iM);
}
#endif  // __CUDACC__

}  // namespace fd
