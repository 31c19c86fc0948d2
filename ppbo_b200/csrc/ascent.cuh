// ppbo_b200 -- batched multi-start gradient ascent on [0,1]^D, one CTA per start (rff_maximize_kernel of acq.cu: sampled
// functions; mu_ascent_kernel of gram.cu: the GP posterior mean).  Only the evaluation differs between the two; the loop is here.
#pragma once
#include "common.cuh"

namespace ppbo {

constexpr int RM_THREADS = 128, RM_MAX_D = 32;

// Projected gradient ascent with Barzilai-Borwein step lengths and Armijo backtracking on the box.  eval(xv, gv) evaluates the
// objective and its gradient at xv (shared) together and leaves them in fval_s and gv (shared), every thread taking part.
// Stationarity is measured by the projected gradient |clip(x + grad) - x|_inf.  Coordinates with their bit set in `periodic` have
// period 1: a step reduces them modulo 1 instead of projecting them, the Armijo slope and the Barzilai-Borwein pair use the
// unwrapped step, and their full gradient counts in the stationarity measure.  periodic = 0 is plain projected ascent on the box.
// On return x, g hold the end point and its gradient, f its value; the result is the iteration count.
template <class Eval>
__device__ __forceinline__ int ascent_loop(const Eval& eval, int D, const double* __restrict__ x0, int max_iter, double gtol,
                                           unsigned periodic, double* x, double* g, double* xt, double* gt, double* sx,
                                           const double& fval_s, double& f_end) {
    const int tid = threadIdx.x;
    const bool wrap = (periodic >> (tid & 31)) & 1u;    // this thread's coordinate (tid < D) is periodic
    if (tid < D) x[tid] = wrap ? x0[tid] - floor(x0[tid]) : fmin(fmax(x0[tid], 0.0), 1.0);
    __syncthreads();
    eval(x, g);
    double f = fval_s;
    double gmax = 0.0;
    for (int d = 0; d < D; ++d) gmax = fmax(gmax, fabs(g[d]));
    double t = 0.05 / fmax(gmax, 1e-12);               // first step: at most 5 % of the box
    int it = 0;
    for (; it < max_iter; ++it) {
        double pg = 0.0;                                // projected-gradient stationarity measure
        for (int d = 0; d < D; ++d) pg = fmax(pg, ((periodic >> d) & 1u) ? fabs(g[d]) : fabs(fmin(fmax(x[d] + g[d], 0.0), 1.0) - x[d]));
        if (pg <= gtol) break;
        double ft = f, slope = 0.0;
        int tries = 0;
        for (;; ++tries) {
            __syncthreads();
            if (tid < D) {
                const double v = x[tid] + t * g[tid];
                if (wrap) {
                    xt[tid] = v - floor(v);
                    sx[tid] = v - x[tid];
                } else {
                    xt[tid] = fmin(fmax(v, 0.0), 1.0);
                    sx[tid] = xt[tid] - x[tid];
                }
            }
            __syncthreads();
            slope = 0.0;
            for (int d = 0; d < D; ++d) slope = fma(g[d], sx[d], slope);
            eval(xt, gt);
            ft = fval_s;
            if (ft >= f + 1e-4 * slope || tries >= 30) break;
            t *= 0.5;
        }
        if (!(ft >= f)) break;                          // no ascent possible at this resolution
        double ss = 0.0, sy = 0.0;
        for (int d = 0; d < D; ++d) {
            const double sd = sx[d], yd = gt[d] - g[d];
            ss = fma(sd, sd, ss);
            sy = fma(sd, yd, sy);
        }
        __syncthreads();
        if (tid < D) { x[tid] = xt[tid]; g[tid] = gt[tid]; }
        __syncthreads();
        f = ft;
        t = (sy < 0.0) ? fmin(fmax(-ss / sy, 1e-8), 1e4) : 2.0 * t;       // Barzilai-Borwein (concave along s), else expand
        if (ss == 0.0) break;
    }
    f_end = f;
    return it;
}

}  // namespace ppbo
