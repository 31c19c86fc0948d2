// ppbo_b200 -- K4 (prediction + exact-GP acquisition) and K3 (random Fourier features) on sm_100a.
// Replaces GPModel.mu_Sigma_pred (src/gp_model.py:441-452), the sampling loops of acquisition.EI / varmax
// (src/acquisition.py:72-81,170-178) and Hsampler.phiVec/phi/Dphi/S/S_grad/S_hessian and its function
// evaluations (src/random_fourier_sampler.py:45-53,106-122,166,170).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "../../include/ppbo_b200.h"
#include "ascent.cuh"
#include "common.cuh"
#include "gemm_f64.cuh"
#include "linalg.cuh"
#include "philox.cuh"

namespace ppbo {

extern int g_tuning[16];
int kernel_matvec(int kind, const double* X1, int n1, const double* X2, int n2, int D, const double* ls_h, double sigma_f,
                  const double* alpha, double* mu, double* partial, cudaStream_t st);
bool km_has_matvec(int kind);
int kernel_matrix_raw(int kind, const double* X1, int n1, const double* X2, int n2, int D, const double* ls_h,
                      double sigma_f, double scale, double diag_add, double* out, long long ld, cudaStream_t st);

// ---------------------------------------------------------------------------------------------- prediction helpers
// The two kernels below take one grid row per prediction point p < PT = P batch and walk the rows in steps of gridDim.y, which
// the launch caps at the hardware limit of 65535 (sampled_max_batch predicts P = 70 points for every (xi, x) pair).
constexpr int PRED_GRID_Y = 65535;
// Ut[p][u] = sa[u] * (Kc[p][r(u)] - Kc[p][w(u)]),  sa = sqrt(max(arrow,0))          (a+^1/2 B^T k*, one RHS per row)
__global__ void __launch_bounds__(256) pred_diff_kernel(const double* __restrict__ Kc, long long ldk, int PT, int Q, int m,
                                                        const double* __restrict__ arrow, double* __restrict__ Ut,
                                                        long long ldu) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= Q * m) return;
    const int q = u / m, j = u % m;
    const long long w = (long long)q * (m + 1);
    const double a = arrow[u];
    for (int p = blockIdx.y; p < PT; p += gridDim.y) {
        const double* k = Kc + (long long)p * ldk;
        Ut[(long long)p * ldu + u] = a > 0.0 ? sqrt(a) * (k[w + 1 + j] - k[w]) : 0.0;
    }
}
// Ud[p][i] = Kc[p][r(u_i)] - Kc[p][w(u_i)] for the negative-coefficient indices u_i
__global__ void pred_negdiff_kernel(const double* __restrict__ Kc, long long ldk, int PT, int m, const int* __restrict__ idx,
                                    int r, double* __restrict__ Ud, long long ldu) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= r) return;
    const int u = idx[i], q = u / m, j = u % m;
    const long long w = (long long)q * (m + 1);
    for (int p = blockIdx.y; p < PT; p += gridDim.y) {
        const double* k = Kc + (long long)p * ldk;
        Ud[(long long)p * ldu + i] = k[w + 1 + j] - k[w];
    }
}
// rows of  a+^1/2 G[:, J-]  (transposed: one row per negative index) and  R0 = diag(1/|a_j|) - G[J-, J-]
__global__ void neg_rows_kernel(const double* __restrict__ G, long long ldg, int M, const double* __restrict__ arrow,
                                const int* __restrict__ idx, int r, double* __restrict__ Ht, double* __restrict__ R,
                                long long ldr) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (u >= M) return;
    const int ui = idx[i];
    const double a = arrow[u];
    const double g = G[(long long)ui * ldg + u];          // G symmetric
    Ht[(long long)i * M + u] = a > 0.0 ? sqrt(a) * g : 0.0;
    if (u < r) {
        const int uj = idx[u];
        double v = -G[(long long)ui * ldg + uj];
        if (u == i) v += 1.0 / fabs(arrow[ui]);
        R[(long long)i * ldr + u] = v;
    }
}

// ---------------------------------------------------------------------------------------------- acquisition reductions
// out[b] = { sum max(fmax - mustar, 0), sum fmax, sum fmax^2 (centred on the first sample for stability is NOT used:
// plain sums in a fixed order, the host forms mean / variance) }
__global__ void __launch_bounds__(1024) acq_reduce_kernel(const double* __restrict__ fm, int S, double mustar,
                                                          const double* __restrict__ mustar_dev, double* __restrict__ out) {
    __shared__ double red[33];
    if (mustar_dev) mustar = mustar_dev[0];
    const double* x = fm + (long long)blockIdx.x * S;
    double s0 = 0, s1 = 0, s2 = 0;
    for (int i = threadIdx.x; i < S; i += 1024) {
        const double v = x[i];
        s0 += fmax(v - mustar, 0.0);
        s1 += v;
        s2 = fma(v, v, s2);
    }
    s0 = block_sum(s0, red);
    s1 = block_sum(s1, red);
    s2 = block_sum(s2, red);
    if (threadIdx.x == 0) {
        out[blockIdx.x * 3 + 0] = s0;
        out[blockIdx.x * 3 + 1] = s1;
        out[blockIdx.x * 3 + 2] = s2;
    }
}

// ---- greedy batch selection (q-EI over the shared draws) ----------------------------------------------------------------------
// gain[b] = sum_s max(max(cur[s], fm[b][s]) - mu*, 0) with cur = the per-sample max of the lines chosen so far (k == 0: none, cur
// is not read).  The strided order and block_sum of acq_reduce_kernel, so that step 0 equals its column 0 bit for bit.
// gain[batch] = S: the number of samples the gains sum over (summed with them over the ranks; the pick divides by it).
__global__ void __launch_bounds__(1024) acq_batch_gain_kernel(const double* __restrict__ fm, int S, int batch,
                                                              const double* __restrict__ mustar_dev, const double* __restrict__ cur,
                                                              int k, double* __restrict__ gain) {
    __shared__ double red[33];
    const double mustar = mustar_dev[0];
    const double* x = fm + (long long)blockIdx.x * S;
    double s0 = 0;
    for (int i = threadIdx.x; i < S; i += 1024) {
        double v = x[i];
        if (k > 0) v = fmax(cur[i], v);
        s0 += fmax(v - mustar, 0.0);
    }
    s0 = block_sum(s0, red);
    if (threadIdx.x == 0) {
        gain[blockIdx.x] = s0;
        if (blockIdx.x == 0) gain[batch] = (double)S;
    }
}

// Step k of the greedy selection: w = arg-max of gain over the candidates not in idx[0..k) (lowest index on ties), idx[k] = w,
// val[k] = gain[w] / gain[batch], cur[s] = max(cur[s], fm[w][s]) (k == 0: cur = fm[w]).  Every CTA recomputes the same arg-max
// over the B gains with its own chosen mask in shared memory, built from idx[0..k) (written by earlier launches: CTA 0 writing
// idx[k] races with nobody), and updates its own slice of cur.
constexpr int PICK_THREADS = 256;
__global__ void __launch_bounds__(PICK_THREADS) acq_batch_pick_kernel(const double* __restrict__ gain, int batch,
                                                                      const double* __restrict__ fm, int S, int k,
                                                                      int* __restrict__ idx, double* __restrict__ val,
                                                                      double* __restrict__ cur) {
    __shared__ unsigned chosen[(PPBO_ACQ_BATCH_MAX + 31) / 32];
    __shared__ double wv[PICK_THREADS / 32];
    __shared__ int wi[PICK_THREADS / 32];
    __shared__ int win_s;
    const int nwords = (batch + 31) >> 5, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < nwords; i += PICK_THREADS) chosen[i] = 0u;
    __syncthreads();
    for (int j = threadIdx.x; j < k; j += PICK_THREADS) {
        const int c = idx[j];
        atomicOr(&chosen[c >> 5], 1u << (c & 31));
    }
    __syncthreads();
    // bi < 0: nothing seen yet (the first unchosen candidate is taken whatever its gain, so a NaN cannot leave the pick empty)
    double bv = -INFINITY;
    int bi = -1;
    for (int c = threadIdx.x; c < batch; c += PICK_THREADS) {
        if ((chosen[c >> 5] >> (c & 31)) & 1u) continue;
        const double g = gain[c];
        if (bi < 0 || g > bv) { bv = g; bi = c; }           // increasing c: a tie keeps the lower index
    }
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if (lane == 0) { wv[warp] = bv; wi[warp] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < PICK_THREADS / 32; ++w)
            if (wi[w] >= 0 && (bi < 0 || wv[w] > bv || (wv[w] == bv && wi[w] < bi))) { bv = wv[w]; bi = wi[w]; }
        win_s = bi;
        if (blockIdx.x == 0) {
            idx[k] = bi;
            val[k] = bv / gain[batch];
        }
    }
    __syncthreads();
    const int w = win_s;
    const int s = blockIdx.x * PICK_THREADS + threadIdx.x;
    if (s < S) {
        const double v = fm[(long long)w * S + s];
        cur[s] = k > 0 ? fmax(cur[s], v) : v;
    }
}

// out[0] = max(init, max_i x[i]) with init = out[0] if `accumulate` (single CTA; used for mu* over candidate points)
__global__ void __launch_bounds__(1024) vec_max_kernel(const double* __restrict__ x, long long n, int accumulate,
                                                       double* __restrict__ out) {
    __shared__ double mx[32];
    double v = accumulate ? out[0] : -INFINITY;
    for (long long i = threadIdx.x; i < n; i += 1024) v = fmax(v, x[i]);
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) mx[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) v = fmax(v, mx[w]);
        out[0] = v;
    }
}

// ---------------------------------------------------------------------------------------------- random Fourier features
// point-major PhiT[i][f] (transposed == 0) or feature-major Phi[f][i] (transposed == 1, the reference's layout)
__global__ void __launch_bounds__(256) rff_features_kernel(const double* __restrict__ W, const double* __restrict__ b, int F,
                                                           int D, const double* __restrict__ X, int n, double amp,
                                                           double* __restrict__ out, long long ld, int feature_major) {
    extern __shared__ double xs[];          // the CTA's point (point-major) or feature row (feature-major)
    if (!feature_major) {
        const int i = blockIdx.y;
        for (int d = threadIdx.x; d < D; d += blockDim.x) xs[d] = X[(long long)i * D + d];
        __syncthreads();
        const int f = blockIdx.x * blockDim.x + threadIdx.x;
        if (f >= F) return;
        double s = b[f];
        for (int d = 0; d < D; ++d) s = fma(W[(long long)f * D + d], xs[d], s);
        out[(long long)i * ld + f] = amp * cos(s);
    } else {
        const int f = blockIdx.y;
        for (int d = threadIdx.x; d < D; d += blockDim.x) xs[d] = W[(long long)f * D + d];
        __syncthreads();
        const int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n) return;
        double s = b[f];
        for (int d = 0; d < D; ++d) s = fma(xs[d], X[(long long)i * D + d], s);
        out[(long long)f * ld + i] = amp * cos(s);
    }
}
__global__ void rff_jacobian_kernel(const double* __restrict__ W, const double* __restrict__ b, int F, int D,
                                    const double* __restrict__ x, double amp, double* __restrict__ J) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    double s = b[f];
    for (int d = 0; d < D; ++d) s = fma(W[(long long)f * D + d], x[d], s);
    const double c = -amp * sin(s);
    for (int d = 0; d < D; ++d) J[(long long)f * D + d] = c * W[(long long)f * D + d];
}
// out[0] = phi(x)' omega, out[1 + d] = d/dx_d (phi(x)' omega): the objective and gradient Hsampler.return_xstar hands to L-BFGS-B
// (src/random_fourier_sampler.py:166-167), fused so a host optimiser pays one launch per evaluation.  Single CTA, D <= 64.
__global__ void __launch_bounds__(256) rff_value_grad_kernel(const double* __restrict__ W, const double* __restrict__ b, int F,
                                                             int D, const double* __restrict__ omega, const double* __restrict__ x,
                                                             double amp, double* __restrict__ out) {
    __shared__ double xs[PPBO_MAX_D];
    __shared__ double red[33];
    for (int d = threadIdx.x; d < D; d += 256) xs[d] = x[d];
    __syncthreads();
    double val = 0.0, g[PPBO_MAX_D];
#pragma unroll 4
    for (int d = 0; d < PPBO_MAX_D; ++d) g[d] = 0.0;
    for (int f = threadIdx.x; f < F; f += 256) {
        const double* w = W + (long long)f * D;
        double s = b[f];
        for (int d = 0; d < D; ++d) s = fma(w[d], xs[d], s);
        double sn, cs;
        sincos(s, &sn, &cs);
        const double om = omega[f];
        val = fma(om, cs, val);
        const double c = -om * sn;
        for (int d = 0; d < D; ++d) g[d] = fma(c, w[d], g[d]);
    }
    val = block_sum(val, red);
    if (threadIdx.x == 0) out[0] = amp * val;
    for (int d = 0; d < D; ++d) {
        const double t = block_sum(g[d], red);
        if (threadIdx.x == 0) out[1 + d] = amp * t;
    }
}
// ---- batched maximiser of sampled functions --------------------------------------------------------------------------------
// Hsampler.return_xstar (src/random_fourier_sampler.py:143-178) maximises ONE sampled function g(x) = phi(x)' omega over [0,1]^D with
// 5-30 sequential scipy L-BFGS-B restarts, every objective / gradient evaluation a Python call.  Here every (sample s, restart r)
// pair is one CTA running ascent_loop (ascent.cuh), the objective and its gradient evaluated together (each thread owns F / 128
// features; one block reduction of D + 1 numbers per evaluation).  A second kernel keeps the best restart per sample.  The sampled
// functions of a periodic kernel's basis are exactly periodic on its periodic coordinates, which `periodic` names.
__global__ void __launch_bounds__(RM_THREADS) rff_maximize_kernel(const double* __restrict__ W, const double* __restrict__ b, int F, int D,
                                                                  double amp, const double* __restrict__ Omega, long long ldo,
                                                                  const double* __restrict__ X0, int R, int max_iter, double gtol,
                                                                  unsigned periodic, double* __restrict__ xout,
                                                                  double* __restrict__ fout, int* __restrict__ iters_out) {
    __shared__ double x[RM_MAX_D], g[RM_MAX_D], xt[RM_MAX_D], gt[RM_MAX_D], sx[RM_MAX_D];
    __shared__ double red[RM_THREADS / 32][RM_MAX_D + 1];
    __shared__ double fval_s;
    const int s = blockIdx.x / R, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* om = Omega + (long long)s * ldo;
    const double* x0 = X0 + (long long)blockIdx.x * D;
    // value and gradient of g at xv (shared) -> fval_s, gv (shared)
    auto eval = [&](const double* xv, double* gv) {
        double val = 0.0, gl[RM_MAX_D];
#pragma unroll
        for (int d = 0; d < RM_MAX_D; ++d) gl[d] = 0.0;
        for (int f = tid; f < F; f += RM_THREADS) {
            const double* w = W + (long long)f * D;
            double a = b[f];
            for (int d = 0; d < D; ++d) a = fma(w[d], xv[d], a);
            double sn, cs;
            sincos(a, &sn, &cs);
            const double o = om[f];
            val = fma(o, cs, val);
            const double c = -o * sn;
#pragma unroll
            for (int d = 0; d < RM_MAX_D; ++d)
                if (d < D) gl[d] = fma(c, w[d], gl[d]);
        }
        for (int o = 16; o > 0; o >>= 1) val += __shfl_xor_sync(0xffffffffu, val, o);
        if (lane == 0) red[warp][RM_MAX_D] = val;
#pragma unroll
        for (int d = 0; d < RM_MAX_D; ++d) {
            if (d < D) {
                double v = gl[d];
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) red[warp][d] = v;
            }
        }
        __syncthreads();
        if (tid <= D) {
            const int k = (tid == D) ? RM_MAX_D : tid;
            const double v = amp * ((red[0][k] + red[1][k]) + (red[2][k] + red[3][k]));
            if (tid == D) fval_s = v;
            else gv[tid] = v;
        }
        __syncthreads();
    };
    double f;
    const int it = ascent_loop(eval, D, x0, max_iter, gtol, periodic, x, g, xt, gt, sx, fval_s, f);
    if (tid < D) xout[(long long)blockIdx.x * D + tid] = x[tid];
    if (tid == 0) {
        fout[blockIdx.x] = f;
        if (iters_out) iters_out[blockIdx.x] = it;
    }
}
// best restart per sample (first maximum)
__global__ void rff_maximize_select_kernel(const double* __restrict__ xall, const double* __restrict__ fall, int S, int R, int D,
                                           double* __restrict__ xbest, double* __restrict__ fbest) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    int br = 0;
    double bf = fall[(long long)s * R];
    for (int r = 1; r < R; ++r) {
        const double v = fall[(long long)s * R + r];
        if (v > bf) { bf = v; br = r; }
    }
    fbest[s] = bf;
    for (int d = 0; d < D; ++d) xbest[(long long)s * D + d] = xall[((long long)s * R + br) * D + d];
}
// also the pick of the posterior-mean search (gram.cu, S = 1)
int maximize_select(const double* xall, const double* fall, int S, int R, int D, double* xbest, double* fbest, cudaStream_t st) {
    PPBO_CL rff_maximize_select_kernel<<<ceil_div(S, 128), 128, 0, st>>>(xall, fall, S, R, D, xbest, fbest);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

// y[i] = sum_f Phi[f][i] omega[f]   (feature-major Phi: coalesced over i).  HBM-bound (8 F N bytes): the feature range is cut
// into FV_SLICES slices so that ~8 x N/128 CTAs stream concurrently; slice partials are combined in a fixed order by the last CTA
// of each column block to finish (count[blockIdx.x] counts the finished slices and is back at 0 when the kernel ends).
constexpr int FV_SLICES = 8, FV_COLS = 128;
__global__ void __launch_bounds__(256) rff_fvals_kernel(const double* __restrict__ Phi, long long ld, int F, int N,
                                                        const double* __restrict__ omega, double* part, double* __restrict__ y,
                                                        unsigned* __restrict__ count, const double* __restrict__ skip) {
    __shared__ double red[FV_COLS];
    __shared__ bool last;
    if (skip && *skip != 0.0) return;          // queued chord step behind the one that stopped the batch (see ppbo_rff_fit)
    const int c = threadIdx.x & (FV_COLS - 1), half = threadIdx.x >> 7;          // 128 columns x 2 row phases
    const int i = blockIdx.x * FV_COLS + c;
    const int per = (F + FV_SLICES - 1) / FV_SLICES;
    const int f0 = blockIdx.y * per, f1 = min(F, f0 + per);
    double s0 = 0.0, s1 = 0.0;
    if (i < N) {
        int f = f0 + half;
        for (; f + 2 < f1; f += 4) {
            s0 = fma(Phi[(long long)f * ld + i], omega[f], s0);
            s1 = fma(Phi[(long long)(f + 2) * ld + i], omega[f + 2], s1);
        }
        for (; f < f1; f += 2) s0 = fma(Phi[(long long)f * ld + i], omega[f], s0);
    }
    if (half == 1) red[c] = s0 + s1;
    __syncthreads();
    if (half == 0 && i < N) part[(long long)blockIdx.y * N + i] = (s0 + s1) + red[c];
    __threadfence();                           // this slice's partials are visible before it is counted
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(count + blockIdx.x, 1u) == FV_SLICES - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (half == 0 && i < N) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < FV_SLICES; ++k) s += __ldcg(part + (long long)k * N + i);
        y[i] = s;
    }
    if (threadIdx.x == 0) count[blockIdx.x] = 0u;
}
// part: FV_SLICES * N doubles of scratch; count: fvals_count_words(N) zeroed words (left zeroed)
static int fvals_count_words(int N) { return ceil_div(N, FV_COLS); }
static int launch_rff_fvals(const double* Phi, long long ld, int F, int N, const double* omega, double* part, double* y,
                            unsigned* count, cudaStream_t st, const double* skip = nullptr) {
    PPBO_CL rff_fvals_kernel<<<dim3(ceil_div(N, FV_COLS), FV_SLICES), 256, 0, st>>>(Phi, ld, F, N, omega, part, y, count, skip);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}
// one warp per feature: grad[f] = -omega[f] + sum_rows beta[row] Phi[f][row]
//                       hdiag[f] = -1 - sum_u arrow[u] (Phi[f][r(u)] - Phi[f][w(u)])^2
__global__ void __launch_bounds__(256) rff_grad_hess_kernel(const double* __restrict__ Phi, long long ld, int F, int Q, int m,
                                                            const double* __restrict__ omega, const double* __restrict__ beta,
                                                            const double* __restrict__ arrow, double* __restrict__ grad,
                                                            double* __restrict__ hdiag, const double* __restrict__ skip) {
    if (skip && *skip != 0.0) return;
    const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f >= F) return;
    const double* ph = Phi + (long long)f * ld;
    const int N = Q * (m + 1), M = Q * m;
    double g = 0.0, h = 0.0;
    if (grad) for (int i = lane; i < N; i += 32) g = fma(beta[i], ph[i], g);
    if (hdiag)
        for (int u = lane; u < M; u += 32) {
            const int q = u / m, j = u % m;
            const double d = ph[(long long)q * (m + 1) + 1 + j] - ph[(long long)q * (m + 1)];
            h = fma(arrow[u], d * d, h);
        }
    for (int o = 16; o > 0; o >>= 1) {
        g += __shfl_xor_sync(0xffffffffu, g, o);
        h += __shfl_xor_sync(0xffffffffu, h, o);
    }
    if (lane == 0) {
        if (grad) grad[f] = -omega[f] + g;
        if (hdiag) hdiag[f] = -1.0 - h;
    }
}
// grad[f] = -omega[f] + sum_rows beta[row] Phi[f][row]: four warps per feature (a quarter of the row each), two features per CTA.
// One warp per feature (rff_grad_hess_kernel) leaves 125 CTAs of 8 long-running warps for F = 1000: 26-80 us per call in the chord
// steps of the fit, latency-bound; this shape streams the same 8 F N bytes with 4x the loads in flight.
__global__ void __launch_bounds__(256) rff_grad_kernel(const double* __restrict__ Phi, long long ld, int F, int N,
                                                       const double* __restrict__ omega, const double* __restrict__ beta,
                                                       double* __restrict__ grad, const double* __restrict__ skip) {
    __shared__ double part[8];
    if (skip && *skip != 0.0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int f = blockIdx.x * 2 + (warp >> 2), qtr = warp & 3;
    double g0 = 0.0, g1 = 0.0;
    if (f < F) {
        const double* ph = Phi + (long long)f * ld;
        const int per = ((N + 3) / 4 + 31) / 32 * 32, i0 = qtr * per, i1 = min(N, i0 + per);
        int i = i0 + lane;
        for (; i + 32 < i1; i += 64) {
            g0 = fma(beta[i], ph[i], g0);
            g1 = fma(beta[i + 32], ph[i + 32], g1);
        }
        if (i < i1) g0 = fma(beta[i], ph[i], g0);
    }
    double g = g0 + g1;
    for (int o = 16; o > 0; o >>= 1) g += __shfl_xor_sync(0xffffffffu, g, o);
    if (lane == 0) part[warp] = g;
    __syncthreads();
    if (threadIdx.x < 2) {
        const int ff = blockIdx.x * 2 + threadIdx.x;
        if (ff < F) grad[ff] = -omega[ff] + ((part[4 * threadIdx.x] + part[4 * threadIdx.x + 1]) + (part[4 * threadIdx.x + 2] + part[4 * threadIdx.x + 3]));
    }
}
// PsiT[f][u] = sa[u] (Phi[f][r(u)] - Phi[f][w(u)])     (F x M, K-contiguous operand of the weight-space Hessian GEMM)
__global__ void __launch_bounds__(256) rff_psi_kernel(const double* __restrict__ Phi, long long ld, int Q, int m,
                                                      const double* __restrict__ arrow, double* __restrict__ PsiT, long long ldp) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
    if (u >= Q * m) return;
    const int q = u / m, j = u % m;
    const double* ph = Phi + (long long)f * ld;
    const double a = arrow[u];
    PsiT[(long long)f * ldp + u] = a > 0.0 ? sqrt(a) * (ph[(long long)q * (m + 1) + 1 + j] - ph[(long long)q * (m + 1)]) : 0.0;
}
// Signed form for the exact Hessian I + Psi' diag(a) Psi (ppbo_rff_hessian_factor): PsiA[f][u] = sqrt|a_u| d_u(f) and
// PsiB[f][u] = sign(a_u) sqrt|a_u| d_u(f), d_u = Phi[f][r(u)] - Phi[f][w(u)], so that PsiA . PsiB^T = sum_u a_u d_u d_u'.
__global__ void __launch_bounds__(256) rff_psi_signed_kernel(const double* __restrict__ Phi, long long ld, int Q, int m,
                                                             const double* __restrict__ arrow, double* __restrict__ PsiA,
                                                             double* __restrict__ PsiB, long long ldp) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
    if (u >= Q * m) return;
    const int q = u / m, j = u % m;
    const double* ph = Phi + (long long)f * ld;
    const double a = arrow[u];
    const double v = sqrt(fabs(a)) * (ph[(long long)q * (m + 1) + 1 + j] - ph[(long long)q * (m + 1)]);
    PsiA[(long long)f * ldp + u] = v;
    PsiB[(long long)f * ldp + u] = a < 0.0 ? -v : v;
}
__global__ void add_identity_kernel(double* __restrict__ A, long long ld, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[(long long)i * ld + i] += 1.0;
}
// scal[0] = -0.5 |omega|^2 ; scal[1] = max|x| ; scal[2] = max|omega|
__global__ void __launch_bounds__(1024) rff_scalars_kernel(const double* __restrict__ omega, const double* __restrict__ x, int F,
                                                           double* __restrict__ scal) {
    __shared__ double red[33];
    __shared__ double mx[2][32];
    double s = 0, m0 = 0, m1 = 0;
    for (int i = threadIdx.x; i < F; i += 1024) {
        s = fma(omega[i], omega[i], s);
        if (x) m0 = fmax(m0, fabs(x[i]));
        m1 = fmax(m1, fabs(omega[i]));
    }
    s = block_sum(s, red);
    for (int o = 16; o > 0; o >>= 1) {
        m0 = fmax(m0, __shfl_xor_sync(0xffffffffu, m0, o));
        m1 = fmax(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    }
    if ((threadIdx.x & 31) == 0) { mx[0][threadIdx.x >> 5] = m0; mx[1][threadIdx.x >> 5] = m1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) { m0 = fmax(m0, mx[0][w]); m1 = fmax(m1, mx[1][w]); }
        scal[0] = -0.5 * s; scal[1] = m0; scal[2] = m1;
    }
}
__global__ void axpy_kernel(double* __restrict__ y, const double* __restrict__ x, double a, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] += a * x[i];
}
__global__ void axpy_out_kernel(double* __restrict__ out, const double* __restrict__ y, const double* __restrict__ x, double a, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = y[i] + a * x[i];
}

// defined in laplace.cu
int launch_lik_terms(const double* f, int Q, int m, double sigma, double* set_lik, double* beta, double* arrow, double* sa,
                     double* bvec, cudaStream_t st);
int launch_sum(const double* x, int n, double* out, cudaStream_t st);
int launch_linesearch_lik(const double* f, const double* df, int Q, int m, double sigma, double* part, cudaStream_t st);
constexpr int LS_STEPS = 8;      // == NSTEP of laplace.cu: step sizes 1, 1/2, ..., 2^-7

// scal[0..2] = omega.omega, omega.step, step.step ; scal[3] = max|step| ; scal[4] = max|omega| ; scal[8 + c] = sum_q part[c][q]
// (1024 threads)
// (rff_chord_tail_kernel writes omega and scal later on: no __restrict__ on them, so that no read goes through the non-coherent
// read-only path)
__device__ __forceinline__ void rff_ls_scalars(const double* omega, const double* __restrict__ step, int F,
                                               const double* __restrict__ part, int Q, double* scal) {
    __shared__ double red_multi[32 * (3 + LS_STEPS)];
    __shared__ double mx[2][32];
    double m0 = 0, m1 = 0;
    double sums[3 + LS_STEPS];
#pragma unroll
    for (int c = 0; c < 3 + LS_STEPS; ++c) sums[c] = 0.0;
    for (int i = threadIdx.x; i < F; i += 1024) {
        const double o = omega[i], d = step[i];
        sums[0] = fma(o, o, sums[0]);
        sums[1] = fma(o, d, sums[1]);
        sums[2] = fma(d, d, sums[2]);
        m0 = fmax(m0, fabs(d));
        m1 = fmax(m1, fabs(o));
    }
    for (int q = threadIdx.x; q < Q; q += 1024) {
#pragma unroll
        for (int c = 0; c < LS_STEPS; ++c) sums[3 + c] += part[(long long)c * Q + q];
    }
    block_sum_multi<3 + LS_STEPS>(sums, red_multi);          // one pair of barriers for all eleven sums
    for (int o = 16; o > 0; o >>= 1) {
        m0 = fmax(m0, __shfl_xor_sync(0xffffffffu, m0, o));
        m1 = fmax(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    }
    if ((threadIdx.x & 31) == 0) { mx[0][threadIdx.x >> 5] = m0; mx[1][threadIdx.x >> 5] = m1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) { m0 = fmax(m0, mx[0][w]); m1 = fmax(m1, mx[1][w]); }
        scal[0] = sums[0]; scal[1] = sums[1]; scal[2] = sums[2]; scal[3] = m0; scal[4] = m1;
        for (int c = 0; c < LS_STEPS; ++c) scal[8 + c] = sums[3 + c];
    }
}
__global__ void __launch_bounds__(1024) rff_ls_scalars_kernel(const double* __restrict__ omega, const double* __restrict__ step,
                                                              int F, const double* __restrict__ part, int Q,
                                                              double* __restrict__ scal) {
    rff_ls_scalars(omega, step, F, part, Q, scal);
}

// Device-side acceptance test of one weight-space chord step (same scheme as chord_decide_kernel of laplace.cu): the full step is
// taken when S does not fall, convergence and contraction are tested here, and the host synchronises once per batch.
//   state[0] S after the last accepted step  state[1] relative size of the last step  state[2] the one before  state[3] the one before that
//   state[4] 0 = keep going, 1 = converged, 2 = contraction too slow (refactor), 3 = full step rejected (refactor)
//   state[5] chord steps taken in this batch   state[6] tolerance    state[7] 1 = this call took the full step (rff_anderson_kernel)
//   hist[2i], hist[2i+1] = (rel, S) of step i
// scal: output of rff_ls_scalars_kernel for this step; scal[24] the likelihood sum at the current iterate (rff_eval), from which S at
// the current iterate is recomputed every step (the iterate may have been mixed since the last accepted step).
// The steps are mixed (rff_anderson); mixed steps are not monotone step by step, so the contraction is judged over three steps (a
// chord step costs ~1/10 of a refactorisation: three steps must gain a factor 5).
// Returns whether the step was taken (the same value in every thread).
__device__ __forceinline__ bool rff_chord_decide(double* omega, const double* __restrict__ step, int F, const double* scal, int m,
                                                 double* state, double* hist) {
    __shared__ int accept_s;
    if (threadIdx.x == 0) {
        const double oo = scal[0], od = scal[1], dd = scal[2], max_step = scal[3], max_om = fmax(scal[4], 1e-300);
        const double S_cur = -0.5 * oo - scal[24] / m;
        const double S1 = -0.5 * (oo + 2.0 * od + dd) - scal[8] / m;
        const int accept = S1 >= S_cur - 1e-13 * fabs(S_cur);
        accept_s = accept;
        state[7] = accept ? 1.0 : 0.0;
        if (!accept) {
            state[4] = 3.0;
        } else {
            const double rel = max_step / max_om, prev = state[1], rel3 = state[3];
            const int n = (int)state[5];
            state[0] = S1;
            state[3] = state[2];
            state[2] = prev;
            state[1] = rel;
            state[5] = n + 1;
            hist[2 * n] = rel;
            hist[2 * n + 1] = S1;
            if (rel <= state[6]) state[4] = 1.0;
            else if (rel3 < 1e300 && !(rel <= 0.2 * rel3)) state[4] = 2.0;
        }
    }
    __syncthreads();
    if (!accept_s) return false;
    for (int i = threadIdx.x; i < F; i += blockDim.x) omega[i] += step[i];
    return true;
}

// Anderson acceleration of the weight-space chord iteration omega <- g(omega) = omega + (-H0)^-1 grad S(omega) (depth RAA_M; same
// scheme as chord_anderson_kernel of laplace.cu).  With the clamped Hessian the iteration matrix differs from the true Hessian by the
// negative curvature coefficients, so even a factor built next to the optimum contracts only linearly (0.3 .. 0.45 per step on the
// bench problem, 0.55 for the factor of the previous PPBO iteration); mixing the last residual differences gains about
// rho / (1 + sqrt(1 - rho^2)) per step instead.  Called after rff_chord_decide has taken a full step: omega = g(omega_k),
// residual r_k = step still in memory.  The history is dropped when a step was rejected or the residual grew.  One CTA of 1024
// threads, fixed order.
//   aa: [0] history length, [1] next slot, [2] residual norm seen by the previous call, [3] 1 = (prev r, prev g) valid
//   Hh: [2 RAA_M + 2][F]: dR[RAA_M], dG[RAA_M], prev r, prev g
constexpr int RAA_M = 5;
__device__ __forceinline__ void rff_anderson(double* omega, const double* __restrict__ step, int F, const double* state, double* aa,
                                             double* Hh) {
    __shared__ double gam[RAA_M];
    __shared__ int nh_s;
    if (state[4] != 0.0) return;                                         // converged, rejected or about to refactor: nothing to mix
    double* dR = Hh;
    double* dG = Hh + (long long)RAA_M * F;
    double* pr = Hh + 2LL * RAA_M * F;
    double* pg = pr + F;
    const bool plain = state[7] == 1.0;
    const double rel = state[1];
    int nh = (int)aa[0], slot = (int)aa[1];
    const double rel_prev = aa[2];
    bool have_prev = aa[3] == 1.0;
    __syncthreads();                                                     // everybody has read the state
    if (!plain || (have_prev && rel > 1.5 * rel_prev)) {
        if (threadIdx.x == 0) { aa[0] = 0.0; aa[1] = 0.0; aa[2] = rel; aa[3] = 0.0; }
        if (!plain) return;
        nh = 0;
        slot = 0;
        have_prev = false;
    }
    if (have_prev) {
        for (int i = threadIdx.x; i < F; i += 1024) {
            dR[(long long)slot * F + i] = step[i] - pr[i];
            dG[(long long)slot * F + i] = omega[i] - pg[i];
        }
        nh = min(nh + 1, RAA_M);
        slot = (slot + 1) % RAA_M;
    }
    for (int i = threadIdx.x; i < F; i += 1024) {
        pr[i] = step[i];
        pg[i] = omega[i];
    }
    __syncthreads();
    // all products of the normal equations in one pass and one multi-value reduction
    constexpr int NPAIR = RAA_M * (RAA_M + 1) / 2;
    __shared__ double red_multi[32 * (NPAIR + RAA_M)];
    double acc[NPAIR + RAA_M];
#pragma unroll
    for (int i = 0; i < NPAIR + RAA_M; ++i) acc[i] = 0.0;
    for (int k = threadIdx.x; k < F; k += 1024) {
        double dv[RAA_M];
#pragma unroll
        for (int i = 0; i < RAA_M; ++i) dv[i] = (i < nh) ? dR[(long long)i * F + k] : 0.0;
        const double rk = step[k];
        int idx = 0;
#pragma unroll
        for (int i = 0; i < RAA_M; ++i) {
#pragma unroll
            for (int j = 0; j <= i; ++j) { acc[idx] = fma(dv[i], dv[j], acc[idx]); ++idx; }
            acc[NPAIR + i] = fma(dv[i], rk, acc[NPAIR + i]);
        }
    }
    block_sum_multi<NPAIR + RAA_M>(acc, red_multi);
    double A[RAA_M][RAA_M], bb[RAA_M];
    {
        int idx = 0;
#pragma unroll
        for (int i = 0; i < RAA_M; ++i) {
#pragma unroll
            for (int j = 0; j <= i; ++j) { A[i][j] = A[j][i] = acc[idx]; ++idx; }
            bb[i] = acc[NPAIR + i];
        }
    }
    if (threadIdx.x == 0) {
        double tr = 0.0;
        for (int i = 0; i < nh; ++i) tr += A[i][i];
        for (int i = 0; i < nh; ++i) A[i][i] += 1e-10 * tr + 1e-300;     // damping: nearly collinear differences
        bool ok = true;
        for (int c = 0; c < nh && ok; ++c) {                             // Gaussian elimination with partial pivoting
            int pv = c;
            for (int r2 = c + 1; r2 < nh; ++r2) if (fabs(A[r2][c]) > fabs(A[pv][c])) pv = r2;
            if (A[pv][c] == 0.0) { ok = false; break; }
            for (int k = 0; k < nh; ++k) { const double t = A[c][k]; A[c][k] = A[pv][k]; A[pv][k] = t; }
            { const double t = bb[c]; bb[c] = bb[pv]; bb[pv] = t; }
            for (int r2 = c + 1; r2 < nh; ++r2) {
                const double l = A[r2][c] / A[c][c];
                for (int k = c; k < nh; ++k) A[r2][k] -= l * A[c][k];
                bb[r2] -= l * bb[c];
            }
        }
        for (int i = nh - 1; i >= 0 && ok; --i) {
            double v = bb[i];
            for (int k = i + 1; k < nh; ++k) v -= A[i][k] * gam[k];
            gam[i] = v / A[i][i];
            if (!(fabs(gam[i]) < 1e3)) ok = false;
        }
        nh_s = ok ? nh : 0;
        aa[0] = ok ? nh : 0;
        aa[1] = ok ? slot : 0;
        aa[2] = rel;
        aa[3] = 1.0;
    }
    __syncthreads();
    const int nm = nh_s;
    if (nm == 0) return;
    for (int i = threadIdx.x; i < F; i += 1024) {
        double c = 0.0;
        for (int j = 0; j < nm; ++j) c = fma(gam[j], dG[(long long)j * F + i], c);
        omega[i] -= c;
    }
}

// End of one weight-space chord step in one CTA: the likelihood sum at the current iterate (scal[24], the reduction of sum_kernel),
// the line-search scalars, the acceptance test and the Anderson mixing, each with the reductions of its former kernel.  What one
// part writes the next reads after a barrier, through plain (coherent) loads: only step, setlik and part are read-only here.
__global__ void __launch_bounds__(1024) rff_chord_tail_kernel(double* omega, const double* __restrict__ step, int F,
                                                              const double* __restrict__ setlik, const double* __restrict__ part,
                                                              int Q, int m, double* scal, double* state, double* hist, double* aa,
                                                              double* Hh) {
    __shared__ double red[33];
    if (state[4] != 0.0) return;               // queued step behind the one that stopped the batch
    double s = 0.0;
    for (int i = threadIdx.x; i < Q; i += 1024) s += setlik[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) scal[24] = s;
    rff_ls_scalars(omega, step, F, part, Q, scal);
    __syncthreads();
    if (!rff_chord_decide(omega, step, F, scal, m, state, hist)) return;
    __syncthreads();
    rff_anderson(omega, step, F, state, aa, Hh);
}

}  // namespace ppbo

using namespace ppbo;

extern "C" long long ppbo_factor_doubles(int n) { return (long long)n * n + potrf_dinv_doubles(n) ; }

// ------------------------------------------------------------------------------------------------ negative-coefficient correction
/* number of negative arrow coefficients and their indices (host sync).  idx_h may be NULL. */
extern "C" int ppbo_neg_count(const double* arrow, int M, int* idx_h, int idx_capacity, void* stream) {
    std::vector<double> a((size_t)M);
    if (readback().add(a.data(), arrow, sizeof(double) * M, (cudaStream_t)stream) != cudaSuccess ||
        readback().finish((cudaStream_t)stream) != cudaSuccess) {
        set_error("ppbo_neg_count: copy failed");
        return PPBO_ERR_CUDA;
    }
    int r = 0;
    for (int u = 0; u < M; ++u)
        if (a[u] < 0.0) {
            if (idx_h && r < idx_capacity) idx_h[r] = u;
            ++r;
        }
    return r;
}
/* neg_corr layout (doubles): [idx as int32, padded to 2*ceil(r/2) ints][Ht r x M][R factor object (r)] */
extern "C" long long ppbo_neg_corr_doubles(int M, int r) {
    return (long long)((r + 1) / 2) + (long long)r * M + ppbo_factor_doubles(r) + 2;
}
extern "C" int ppbo_neg_corr_build(const double* G, long long ldg, int M, const double* arrow, const double* Lfac, int cap,
                                   const int* idx_h, int r, double* neg_corr, void* stream) {
    if (r <= 0) return PPBO_OK;
    PPBO_REQUIRE(cap >= M && ldg >= M, "capacity / leading dimension below M");
    cudaStream_t st = (cudaStream_t)stream;
    int* idx = reinterpret_cast<int*>(neg_corr);
    double* Ht = neg_corr + (r + 1) / 2;
    double* R = Ht + (long long)r * M;
    double* Rdinv = R + (long long)r * r;
    int* info_d = reinterpret_cast<int*>(neg_corr + ppbo_neg_corr_doubles(M, r) - 1);
    PPBO_CUDA_CHECK(cudaMemcpyAsync(idx, idx_h, sizeof(int) * r, cudaMemcpyHostToDevice, st));
    PPBO_CL neg_rows_kernel<<<dim3(ceil_div(M, 256), r), 256, 0, st>>>(G, ldg, M, arrow, idx, r, Ht, R, r);
    PPBO_LAUNCH_CHECK();
    int rc = trsm_right_lower_t(Lfac, cap, M, Lfac + (long long)cap * cap, Ht, M, r, st);   // Ht <- Ht L^-T
    if (rc) return rc;
    GemmOperands g{Ht, M, 0, Ht, M, 0, r, r, M};
    StoreEpilogue ep{R, r, 0, 1.0, 1.0, 0, 0, 0};                                      // R += Ht Ht^T
    if ((rc = launch_gemm_nt(g, ep, 1, st))) return rc;
    if ((rc = potrf_lower(R, r, r, Rdinv, info_d, st))) return rc;
    int info = 0;
    PPBO_CUDA_CHECK(readback().add(&info, info_d, sizeof(int), st));
    PPBO_CUDA_CHECK(readback().finish(st));
    if (info) { set_error("posterior precision is not positive definite (negative-coefficient block, pivot %d)", info); return info; }
    return PPBO_OK;
}

// ------------------------------------------------------------------------------------------------ prediction
extern "C" long long ppbo_predict_workspace_bytes(int N, int Q, int m, int P, int batch) {
    const long long PT = (long long)P * batch, M = (long long)Q * m;
    return (PT * N + PT * M + PT * M + 64) * 8;     // Kc, Ut, (Ud | Zs up to r <= M columns)
}

/* workspace of a mean-only call (Sigma_p == NULL): the mat-vec mode of the SE / RQ / Matern / camphor kernels never materialises
   the cross-covariance */
static long long predict_mean_bytes(bool streams, int N, long long PT) { return (PT * (streams ? (N + 63) / 64 : N) + 64) * 8; }
extern "C" long long ppbo_predict_mean_workspace_bytes(int kind, int N, int P, int batch) {
    return predict_mean_bytes(km_has_matvec(kind), N, (long long)P * batch);
}

extern "C" int ppbo_predict(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f,
                            double shrinkage, int Q, int m, const double* alpha, const double* arrow, const double* Lfac, int cap,
                            const double* neg_corr, int n_neg, const double* Xp, int P, int batch, double* mu,
                            double* Sigma_p, void* workspace, long long workspace_bytes, void* stream) {
    PPBO_REQUIRE(N == Q * (m + 1), "N must equal Q (m+1)");
    PPBO_REQUIRE(Sigma_p == nullptr || cap >= Q * m, "factor capacity below Q m");
    PPBO_REQUIRE(P >= 1 && batch >= 1, "empty grid");
    // the mean alone streams through kernel_matvec unless tuning key 11 selects the materialising path (cross-covariance + GEMV)
    const bool streams = g_tuning[11] == 0 && km_has_matvec(kind);
    PPBO_REQUIRE(workspace_bytes >= (Sigma_p ? ppbo_predict_workspace_bytes(N, Q, m, P, batch)
                                             : predict_mean_bytes(streams, N, (long long)P * batch)),
                 "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int PT = P * batch, M = Q * m;
    double* Kc = (double*)workspace;                 // [PT x N]   k(x*_p, X_i)
    double* Ut = Kc + (long long)PT * N;             // [PT x M]
    double* Ud = Ut + (long long)PT * M;             // [PT x r]
    int rc;
    if (!Sigma_p) {                                  // mean only: no need for the PT x N cross-covariance in memory
        if (!mu) return PPBO_OK;
        rc = kernel_matvec(kind, Xp, PT, X, N, D, lengthscales_h, sigma_f, alpha, mu, Kc, st);
        if (rc < 0) return rc;
        if (rc == 1) return PPBO_OK;
    }
    if ((rc = kernel_matrix_raw(kind, Xp, PT, X, N, D, lengthscales_h, sigma_f, 1.0, 0.0, Kc, N, st))) return rc;
    if (mu && (rc = gemv(Kc, N, PT, N, alpha, mu, st))) return rc;
    if (!Sigma_p) return PPBO_OK;
    PPBO_CL pred_diff_kernel<<<dim3(ceil_div(M, 256), std::min(PT, PRED_GRID_Y)), 256, 0, st>>>(Kc, N, PT, Q, m, arrow, Ut, M);
    PPBO_LAUNCH_CHECK();
    if ((rc = trsm_right_lower_t(Lfac, cap, M, Lfac + (long long)cap * cap, Ut, M, PT, st))) return rc;   // Yt = Ut L^-T
    for (int b = 0; b < batch; ++b) {     // reg(K**) per grid (diagonal shrinkage needs the square form)
        const double* xb = Xp + (long long)b * P * D;
        if ((rc = kernel_matrix_raw(kind, xb, P, xb, P, D, lengthscales_h, sigma_f, 1.0 - shrinkage,
                                    shrinkage * sigma_f * sigma_f, Sigma_p + (long long)b * P * P, P, st)))
            return rc;
    }
    {
        GemmOperands g{Ut, M, (long long)P * M, Ut, M, (long long)P * M, P, P, M};
        StoreEpilogue ep{Sigma_p, P, (long long)P * P, -1.0, 1.0, 0, 0, 0};
        if ((rc = launch_gemm_nt(g, ep, batch, st))) return rc;                                     // -= Yt Yt^T
    }
    if (n_neg > 0) {
        PPBO_REQUIRE(neg_corr != nullptr, "neg_corr missing");
        const int r = n_neg;
        const int* idx = reinterpret_cast<const int*>(neg_corr);
        const double* Ht = neg_corr + (r + 1) / 2;
        const double* R = Ht + (long long)r * M;
        PPBO_CL pred_negdiff_kernel<<<dim3(ceil_div(r, 128), std::min(PT, PRED_GRID_Y)), 128, 0, st>>>(Kc, N, PT, m, idx, r, Ud, r);
        PPBO_LAUNCH_CHECK();
        GemmOperands g1{Ut, M, 0, Ht, M, 0, PT, r, M};
        StoreEpilogue e1{Ud, r, 0, -1.0, 1.0, 0, 0, 0};                                             // z = Ud - Yt Ht^T
        if ((rc = launch_gemm_nt(g1, e1, 1, st))) return rc;
        if ((rc = trsm_right_lower_t(R, r, r, R + (long long)r * r, Ud, r, PT, st))) return rc;     // Zs = z LR^-T
        GemmOperands g2{Ud, r, (long long)P * r, Ud, r, (long long)P * r, P, P, r};
        StoreEpilogue e2{Sigma_p, P, (long long)P * P, 1.0, 1.0, 0, 0, 0};                          // += Zs Zs^T
        if ((rc = launch_gemm_nt(g2, e2, batch, st))) return rc;
    }
    return PPBO_OK;
}

extern "C" int ppbo_mvn_rowmax(const double* Z, long long ldz, long long strideZ, const double* Fac, long long ldf,
                               long long strideF, const double* mu, long long strideMu, int S, int P, int K, int batch,
                               double* fmax, int* arg, void* stream) {
    PPBO_REQUIRE(S >= 0 && P >= 1 && K >= 1 && batch >= 1, "shape");
    GemmOperands g{Z, ldz, strideZ, Fac, ldf, strideF, S, P, K};
    RowMaxEpilogue ep{mu, strideMu, fmax, arg, nullptr, 0, 0};
    return launch_gemm_nt_rowmax(g, ep, batch, (cudaStream_t)stream);
}

extern "C" int ppbo_acq_reduce(const double* fmax, int S, int batch, double mustar, double* out, void* stream) {
    PPBO_REQUIRE(S >= 1 && batch >= 1, "shape");
    PPBO_CL acq_reduce_kernel<<<batch, 1024, 0, (cudaStream_t)stream>>>(fmax, S, mustar, nullptr, out);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_acq_reduce_dev(const double* fmax, int S, int batch, const double* mustar_dev, double* out, void* stream) {
    PPBO_REQUIRE(S >= 1 && batch >= 1 && mustar_dev != nullptr, "shape");
    PPBO_CL acq_reduce_kernel<<<batch, 1024, 0, (cudaStream_t)stream>>>(fmax, S, 0.0, mustar_dev, out);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_acq_batch_gain(const double* fmax, int S, int batch, const double* mustar_dev, const double* cur, int k, int q,
                                   double* gain, void* stream) {
    PPBO_REQUIRE(S >= 1 && batch >= 1 && mustar_dev != nullptr, "shape");
    PPBO_REQUIRE(batch <= PPBO_ACQ_BATCH_MAX, "more candidates than one selection takes");
    PPBO_REQUIRE(q >= 1 && q <= batch && k >= 0 && k < q, "need 0 <= k < q <= batch");
    PPBO_REQUIRE(k == 0 || cur != nullptr, "cur missing");
    PPBO_CL acq_batch_gain_kernel<<<batch, 1024, 0, (cudaStream_t)stream>>>(fmax, S, batch, mustar_dev, cur, k, gain);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_acq_batch_pick(const double* gain, int batch, const double* fmax, int S, int k, int q, int* idx, double* val,
                                   double* cur, void* stream) {
    PPBO_REQUIRE(S >= 0 && batch >= 1 && (S == 0 || (fmax != nullptr && cur != nullptr)), "shape");
    PPBO_REQUIRE(batch <= PPBO_ACQ_BATCH_MAX, "more candidates than one selection takes");
    PPBO_REQUIRE(q >= 1 && q <= batch && k >= 0 && k < q, "need 0 <= k < q <= batch");
    PPBO_CL acq_batch_pick_kernel<<<std::max(1, ceil_div(S, PICK_THREADS)), PICK_THREADS, 0, (cudaStream_t)stream>>>(
        gain, batch, fmax, S, k, idx, val, cur);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_vec_max(const double* x, long long n, int accumulate, double* out, void* stream) {
    PPBO_REQUIRE(n >= 0 && out != nullptr, "shape");
    PPBO_CL vec_max_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(x, n, accumulate, out);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

// ------------------------------------------------------------------------------------------------ RFF
extern "C" int ppbo_rff_features(const double* W, const double* b, int F, int D, const double* X, int n, double sigma_f,
                                 double* Phi, long long ld, int feature_major, void* stream) {
    PPBO_REQUIRE(F >= 1 && D >= 1 && n >= 0, "shape");
    if (n == 0) return PPBO_OK;
    const double amp = sqrt(2.0 * sigma_f * sigma_f / F);      // src/random_fourier_sampler.py:46
    dim3 grid = feature_major ? dim3(ceil_div(n, 256), F) : dim3(ceil_div(F, 256), n);
    PPBO_REQUIRE(grid.y <= 65535, "too many rows for one launch");
    PPBO_CL rff_features_kernel<<<grid, 256, sizeof(double) * D, (cudaStream_t)stream>>>(W, b, F, D, X, n, amp, Phi, ld, feature_major);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_rff_jacobian(const double* W, const double* b, int F, int D, const double* x, double sigma_f, double* J,
                                 void* stream) {
    const double amp = sqrt(2.0 * sigma_f * sigma_f / F);
    PPBO_CL rff_jacobian_kernel<<<ceil_div(F, 128), 128, 0, (cudaStream_t)stream>>>(W, b, F, D, x, amp, J);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_rff_value_grad(const double* W, const double* b, int F, int D, const double* omega, const double* x,
                                   double sigma_f, double* out, void* stream) {
    PPBO_REQUIRE(F >= 1 && D >= 1 && D <= PPBO_MAX_D, "shape");
    const double amp = sqrt(2.0 * sigma_f * sigma_f / F);
    PPBO_CL rff_value_grad_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(W, b, F, D, omega, x, amp, out);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_rff_maximize(const double* W, const double* b, int F, int D, double sigma_f, const double* Omega, long long ldo,
                                 int S, const double* X0, int R, int max_iter, double gtol, int periodic_mask, double* xbest,
                                 double* fbest, double* work, void* stream) {
    PPBO_REQUIRE(F >= 1 && D >= 1 && D <= RM_MAX_D, "D must be in [1, 32]");
    PPBO_REQUIRE(S >= 0 && R >= 1 && max_iter >= 0 && gtol >= 0 && work != nullptr, "arguments");
    PPBO_REQUIRE(periodic_mask >= 0 && (D == 32 || (periodic_mask >> D) == 0), "periodic_mask names a coordinate beyond D");
    if (S == 0) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const double amp = sqrt(2.0 * sigma_f * sigma_f / F);
    double* xall = work;                                  // [S][R][D]
    double* fall = work + (long long)S * R * D;          // [S][R]
    PPBO_CL rff_maximize_kernel<<<S * R, RM_THREADS, 0, st>>>(W, b, F, D, amp, Omega, ldo, X0, R, max_iter, gtol, (unsigned)periodic_mask, xall, fall,
                                                                  nullptr);
    return maximize_select(xall, fall, S, R, D, xbest, fbest, st);
}

extern "C" long long ppbo_rff_workspace_bytes(int F, int Q, int m) {
    const long long N = (long long)Q * (m + 1), M = (long long)Q * m;
    return ((3 + FV_SLICES) * N + 2 * M + Q * 9 + 64 + (long long)F * M + ppbo_factor_doubles(F) + 3 * (long long)F + 2 * CHOL_NB +
            blockinv_doubles(F) + (2LL * RAA_M + 2) * F + 8 + (fvals_count_words((int)N) + 1) / 2) * 8;
}

struct RffWs {
    double *fvals, *dfv, *fpart, *beta, *arrow, *setlik, *scal, *PsiT, *H, *step, *trial, *tmp, *binv, *aaH, *aa;
    unsigned* fv_count;        // slice counters of rff_fvals_kernel: zero them once per call (zero_counters)
    int nfv_count;
    void carve(double* p, int F, int Q, int m) {
        const long long N = (long long)Q * (m + 1), M = (long long)Q * m;
        fvals = p; p += N;
        dfv = p; p += N;
        fpart = p; p += (long long)FV_SLICES * N;
        beta = p; p += N;
        arrow = p; p += 2 * M;
        setlik = p; p += 9LL * Q;
        scal = p; p += 64;
        PsiT = p; p += (long long)F * M;
        H = p; p += ppbo_factor_doubles(F);
        step = p; p += F + CHOL_NB;
        trial = p; p += F;
        tmp = p; p += F;
        aaH = p; p += (2LL * RAA_M + 2) * F;
        aa = p; p += 8;
        binv = p; p += blockinv_doubles(F);
        fv_count = reinterpret_cast<unsigned*>(p);
        nfv_count = fvals_count_words((int)N);
    }
    cudaError_t zero_counters(cudaStream_t st) { return cudaMemsetAsync(fv_count, 0, sizeof(unsigned) * nfv_count, st); }
};

// lik_sum_dev == nullptr: the likelihood sum is left to the caller (the chord steps take it in rff_chord_tail_kernel)
static int rff_eval(const double* Phi, long long ld, int F, int Q, int m, double sigma, const double* omega, RffWs& ws,
                    double* grad, double* hdiag, bool want_arrow, double* lik_sum_dev, cudaStream_t st, const double* skip = nullptr) {
    const int N = Q * (m + 1);
    launch_rff_fvals(Phi, ld, F, N, omega, ws.fpart, ws.fvals, ws.fv_count, st, skip);
    launch_lik_terms(ws.fvals, Q, m, sigma, ws.setlik, ws.beta, want_arrow ? ws.arrow : nullptr, nullptr, nullptr, st);
    if (lik_sum_dev) launch_sum(ws.setlik, Q, lik_sum_dev, st);
    if (grad && !hdiag)
        PPBO_CL rff_grad_kernel<<<ceil_div(F, 2), 256, 0, st>>>(Phi, ld, F, N, omega, ws.beta, grad, skip);
    else if (grad || hdiag)
        PPBO_CL rff_grad_hess_kernel<<<ceil_div(F, 8), 256, 0, st>>>(Phi, ld, F, Q, m, omega, ws.beta, ws.arrow, grad, hdiag, skip);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

/* S, gradient and diagonal Hessian at omega (Phi_X feature-major [F x N]). */
extern "C" int ppbo_rff_objective(const double* Phi_X, long long ld, int F, int Q, int m, double sigma, const double* omega,
                                  double* S_out, double* grad, double* hess_diag, void* workspace, long long workspace_bytes,
                                  void* stream) {
    PPBO_REQUIRE(workspace_bytes >= ppbo_rff_workspace_bytes(F, Q, m), "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    RffWs ws;
    ws.carve((double*)workspace, F, Q, m);
    PPBO_CUDA_CHECK(ws.zero_counters(st));
    int rc = rff_eval(Phi_X, ld, F, Q, m, sigma, omega, ws, grad, hess_diag, true, ws.scal + 8, st);
    if (rc) return rc;
    if (S_out) {
        PPBO_CL rff_scalars_kernel<<<1, 1024, 0, st>>>(omega, nullptr, F, ws.scal);
        double h[9];
        PPBO_CUDA_CHECK(readback().add(h, ws.scal, sizeof(h), st));
        PPBO_CUDA_CHECK(readback().finish(st));
        *S_out = h[0] - h[8] / m;
    }
    return PPBO_OK;
}

/* omega_MAP = argmax S(omega) (Hsampler.update_omega_MAP, src/random_fourier_sampler.py:124-132): full Newton in weight
 * space with the exact (clamped) Hessian I + Psi' a+ Psi and a backtracking line search; also returns the DIAGONAL Hessian at the
 * optimum, which is what the reference's Laplace covariance uses (src/random_fourier_sampler.py:118-122,134-137). */
extern "C" long long ppbo_rff_factor_cache_doubles(int F) { return ppbo_factor_doubles(F) + blockinv_doubles(F); }

extern "C" int ppbo_rff_fit(const double* Phi_X, long long ld, int F, int Q, int m, double sigma, const double* omega0,
                            int max_iter, double tol, double* factor_cache, int warm_factor, double* omega_map, double* hess_diag,
                            void* workspace, long long workspace_bytes, double* stats_h, void* stream) {
    PPBO_REQUIRE(workspace_bytes >= ppbo_rff_workspace_bytes(F, Q, m), "workspace too small");
    PPBO_REQUIRE(!warm_factor || (factor_cache != nullptr && omega0 != nullptr), "a warm factor needs the cache and omega0");
    cudaStream_t st = (cudaStream_t)stream;
    const int M = Q * m;
    RffWs ws;
    ws.carve((double*)workspace, F, Q, m);
    if (factor_cache) {          // the Hessian factor (and its block inverses) live in the caller's persistent buffer
        ws.H = factor_cache;
        ws.binv = factor_cache + ppbo_factor_doubles(F);
    }
    double* Hdinv = ws.H + (long long)F * F;
    int* info_d = reinterpret_cast<int*>(ws.scal + 32);
    PPBO_CUDA_CHECK(cudaMemsetAsync(info_d, 0, sizeof(int), st));       // (a warm fit may never factorise)
    PPBO_CUDA_CHECK(ws.zero_counters(st));
    if (omega0) PPBO_CUDA_CHECK(cudaMemcpyAsync(omega_map, omega0, sizeof(double) * F, cudaMemcpyDeviceToDevice, st));
    else PPBO_CUDA_CHECK(cudaMemsetAsync(omega_map, 0, sizeof(double) * F, st));
    int rc, it = 0, info = 0, n_factor = 0, n_chord = 0;
    double h[32], S_cur = NAN, last_rel = INFINITY;
    const int N = Q * (m + 1);
    double* part = ws.setlik + Q;                       // [LS_STEPS][Q]
    const double CHORD_REL = 0.25;
    const bool trace = getenv("PPBO_TRACE") != nullptr;
    // warm_factor: the cache holds the factor of the previous fit's Hessian (the design grew by a comparison set, omega0 is the
    // previous optimum): start with chord steps, factorise only when they are rejected or contract too slowly.  warm_factor = 2: the
    // 1024-block inverses of that factor are in the cache as well.
    bool refactor = !warm_factor, binv_valid = warm_factor == 2;
    constexpr int RFF_BATCH_MAX = 8;
    double* state_d = ws.scal + 40;                     // [8] batch state, [16] history (scal holds 64 doubles)
    double* hist_d = ws.scal + 48;
    double prev_rel_h = INFINITY, rel3_h = INFINITY;
    bool first_batch = true;
    PPBO_CUDA_CHECK(cudaMemsetAsync(ws.aa, 0, sizeof(double) * 8, st));
    for (it = 0; it < max_iter; ++it) {
        if (!refactor) {
            // ---- a batch of chord steps with the device-side acceptance test: one host synchronise per batch (a host decision per
            // step cost ~0.29 ms per step for ~0.1 ms of kernels)
            if (!binv_valid) {
                if ((rc = blockinv_build(ws.H, F, F, Hdinv, ws.binv, st))) return rc;
                binv_valid = true;
            }
            double rho = (std::isfinite(prev_rel_h) && last_rel < prev_rel_h) ? last_rel / prev_rel_h : 0.2;
            rho = std::fmin(std::fmax(rho, 0.02), 0.7);
            int kb = !std::isfinite(last_rel) ? 3 : (last_rel > tol) ? (int)std::ceil(std::log(tol / last_rel) / std::log(rho)) : 1;
            if (first_batch) kb = std::min(kb, 3);
            kb = std::max(1, std::min(kb, std::min(RFF_BATCH_MAX, max_iter - it)));
            first_batch = false;
            double state_h[8] = {S_cur, last_rel, prev_rel_h, rel3_h, 0.0, 0.0, tol, 0.0}, hist_h[2 * RFF_BATCH_MAX];
            PPBO_CUDA_CHECK(cudaMemcpyAsync(state_d, state_h, sizeof(state_h), cudaMemcpyHostToDevice, st));
            const double* skip = state_d + 4;
            for (int i = 0; i < kb; ++i) {     // the gradient goes straight into the step vector, which the solve overwrites
                if ((rc = rff_eval(Phi_X, ld, F, Q, m, sigma, omega_map, ws, ws.step, nullptr, false, nullptr, st, skip))) return rc;
                if ((rc = potrs_vec_blockinv(ws.H, F, F, ws.binv, ws.step, st, skip))) return rc;
                launch_rff_fvals(Phi_X, ld, F, N, ws.step, ws.fpart, ws.dfv, ws.fv_count, st, skip);
                if ((rc = launch_linesearch_lik(ws.fvals, ws.dfv, Q, m, sigma, part, st))) return rc;
                PPBO_CL rff_chord_tail_kernel<<<1, 1024, 0, st>>>(omega_map, ws.step, F, ws.setlik, part, Q, m, ws.scal, state_d, hist_d,
                                                                 ws.aa, ws.aaH);
            }
            PPBO_LAUNCH_CHECK();
            PPBO_CUDA_CHECK(readback().add(state_h, state_d, sizeof(state_h), st));
            PPBO_CUDA_CHECK(readback().add(hist_h, hist_d, sizeof(double) * 2 * kb, st));
            PPBO_CUDA_CHECK(readback().finish(st));
            const int taken = (int)state_h[5], stop = (int)state_h[4];
            if (trace)
                for (int i = 0; i < taken; ++i)
                    fprintf(stderr, "[ppbo_rff_fit] it %d chord  step 1 rel %.3e S %.12g (batch of %d)\n", it + i, hist_h[2 * i], hist_h[2 * i + 1], kb);
            n_chord += taken;
            if (taken > 0) {
                last_rel = state_h[1];
                prev_rel_h = state_h[2];
                rel3_h = state_h[3];
            }
            // S after the last accepted step; stale once that step's result has been mixed (every accepted step but a converging one)
            S_cur = stop == 1 ? (taken > 0 ? state_h[0] : S_cur) : NAN;
            it += taken;
            if (stop == 1) break;
            if (stop == 2 || stop == 3) refactor = true;
            --it;                                        // the loop header adds one
            continue;
        }
        // ---- Newton step: gradient and clamped Hessian at omega, fresh factor (chord steps with a kept factor all go through the
        // batches above).  A null omega0 starts at omega = 0: every difference is 0, so a+ = 0 and the Hessian I + Psi' a+ Psi is
        // the identity.  That first step is the gradient itself (the same bits the solve with the factor of I gives), and nothing is
        // factorised: the factor in ws.H stays invalid and the next step factorises.
        const bool identity_step = it == 0 && omega0 == nullptr;
        // the gradient goes straight into the step vector, which the solve overwrites
        if ((rc = rff_eval(Phi_X, ld, F, Q, m, sigma, omega_map, ws, ws.step, nullptr, !identity_step, ws.scal + 24, st))) return rc;
        if (!identity_step) {
            PPBO_CL rff_psi_kernel<<<dim3(ceil_div(M, 256), F), 256, 0, st>>>(Phi_X, ld, Q, m, ws.arrow, ws.PsiT, M);
            {
                GemmOperands g{ws.PsiT, M, 0, ws.PsiT, M, 0, F, F, M};
                StoreEpilogue ep{ws.H, F, 0, 1.0, 0.0, 2, 0, 0};        // lower tiles only: the factorisation reads no more
                if ((rc = launch_gemm_nt(g, ep, 1, st))) return rc;
            }
            PPBO_CL add_identity_kernel<<<ceil_div(F, 256), 256, 0, st>>>(ws.H, F, F);
            if ((rc = potrf_lower(ws.H, F, F, Hdinv, info_d, st))) return rc;
            ++n_factor;
            binv_valid = false;
            PPBO_CUDA_CHECK(cudaMemsetAsync(ws.aa, 0, sizeof(double) * 8, st));     // new iteration matrix: forget the mixing history
            rel3_h = INFINITY;
            // step = (-Hessian)^-1 grad  (ascent direction)
            if ((rc = potrs_vec(ws.H, F, F, Hdinv, ws.step, st))) return rc;
        }
        // line search, all LS_STEPS step sizes in one pass: f(omega + s step) = f0 + s df, |omega + s step|^2 in closed form
        launch_rff_fvals(Phi_X, ld, F, N, ws.step, ws.fpart, ws.dfv, ws.fv_count, st);
        if ((rc = launch_linesearch_lik(ws.fvals, ws.dfv, Q, m, sigma, part, st))) return rc;
        PPBO_CL rff_ls_scalars_kernel<<<1, 1024, 0, st>>>(omega_map, ws.step, F, part, Q, ws.scal);
        PPBO_LAUNCH_CHECK();
        PPBO_CUDA_CHECK(readback().add(h, ws.scal, sizeof(double) * 32, st));
        PPBO_CUDA_CHECK(readback().add(&info, info_d, sizeof(int), st));
        PPBO_CUDA_CHECK(readback().finish(st));
        if (info) { set_error("weight-space Hessian not positive definite (pivot %d)", info); return info; }
        const double oo = h[0], od = h[1], dd = h[2], max_step = h[3], max_om = fmax(h[4], 1e-300);
        if (std::isnan(S_cur)) S_cur = -0.5 * oo - h[24] / m;
        int c;
        double s = 1.0, S_new = S_cur;
        for (c = 0; c < LS_STEPS; ++c) {
            s = std::ldexp(1.0, -c);
            const double S_try = -0.5 * (oo + 2.0 * s * od + s * s * dd) - h[8 + c] / m;
            if (S_try >= S_cur - 1e-13 * fabs(S_cur)) { S_new = S_try; break; }
        }
        if (c == LS_STEPS) { s = std::ldexp(1.0, -(LS_STEPS - 1)); S_new = NAN; }
        PPBO_CL axpy_kernel<<<ceil_div(F, 256), 256, 0, st>>>(omega_map, ws.step, s, F);
        PPBO_LAUNCH_CHECK();
        S_cur = S_new;
        prev_rel_h = last_rel;
        last_rel = s * max_step / max_om;
        if (trace) fprintf(stderr, "[ppbo_rff_fit] it %d newton step %.3g rel %.3e S %.12g\n", it, s, last_rel, S_cur);
        if (c == 0 && last_rel <= tol) { ++it; break; }
        refactor = identity_step || !(c == 0 && last_rel <= CHORD_REL);   // chord steps once a full Newton step is in the contraction region
    }
    if (std::isnan(S_cur)) {                             // last step left S unevaluated: evaluate at the final point
        if ((rc = rff_eval(Phi_X, ld, F, Q, m, sigma, omega_map, ws, nullptr, nullptr, false, ws.scal + 24, st))) return rc;
        PPBO_CL rff_scalars_kernel<<<1, 1024, 0, st>>>(omega_map, nullptr, F, ws.scal);
        PPBO_CUDA_CHECK(readback().add(h, ws.scal, sizeof(double) * 32, st));
        PPBO_CUDA_CHECK(readback().finish(st));
        S_cur = h[0] - h[24] / m;
    }
    if (hess_diag) {
        if ((rc = rff_eval(Phi_X, ld, F, Q, m, sigma, omega_map, ws, nullptr, hess_diag, true, ws.scal + 24, st))) return rc;
    }
    PPBO_CUDA_CHECK(readback().finish(st));
    if (stats_h) {
        stats_h[0] = it; stats_h[1] = last_rel; stats_h[2] = S_cur; stats_h[3] = n_factor + 0.001 * n_chord;
        stats_h[4] = (binv_valid && factor_cache) ? 1.0 : 0.0;      // the cache's block inverses belong to the cache's factor
    }
    return PPBO_OK;
}

/* The exact weight-space Hessian -grad^2 S(omega) = I + Psi' diag(a) Psi with the SIGNED coefficients a (the fit factors the clamped
 * I + Psi' a+ Psi, which is the right chord matrix but not the Laplace precision), factorised into the caller's L: the full
 * covariance of the weight-space posterior is its inverse.  Nothing of the fit's factor cache is touched. */
extern "C" long long ppbo_rff_hessian_factor_workspace_bytes(int F, int Q, int m) {
    return ppbo_rff_workspace_bytes(F, Q, m) + (long long)F * Q * m * 8;
}
extern "C" long long ppbo_rff_hessian_factor_doubles(int F, long long ldl) {
    return (long long)F * ldl + potrf_dinv_doubles(F) + 2;
}

extern "C" int ppbo_rff_hessian_factor(const double* Phi_X, long long ld, int F, int Q, int m, double sigma, const double* omega,
                                       double* L, long long ldl, void* workspace, long long workspace_bytes, int* info_h,
                                       void* stream) {
    PPBO_REQUIRE(F >= 1 && Q >= 1 && m >= 1 && ldl >= F && L != nullptr, "shape");
    PPBO_REQUIRE(workspace_bytes >= ppbo_rff_hessian_factor_workspace_bytes(F, Q, m), "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int M = Q * m;
    RffWs ws;
    ws.carve((double*)workspace, F, Q, m);
    double* PsiB = (double*)workspace + ppbo_rff_workspace_bytes(F, Q, m) / 8;
    double* dinv = L + (long long)F * ldl;
    int* info_d = reinterpret_cast<int*>(dinv + potrf_dinv_doubles(F));
    PPBO_CUDA_CHECK(ws.zero_counters(st));
    int rc;
    if ((rc = rff_eval(Phi_X, ld, F, Q, m, sigma, omega, ws, nullptr, nullptr, true, ws.scal + 24, st))) return rc;
    PPBO_CL rff_psi_signed_kernel<<<dim3(ceil_div(M, 256), F), 256, 0, st>>>(Phi_X, ld, Q, m, ws.arrow, ws.PsiT, PsiB, M);
    GemmOperands g{ws.PsiT, M, 0, PsiB, M, 0, F, F, M};
    StoreEpilogue ep{L, ldl, 0, 1.0, 0.0, 2, 0, 0};                  // lower tiles only: the factorisation reads no more
    if ((rc = launch_gemm_nt(g, ep, 1, st))) return rc;
    PPBO_CL add_identity_kernel<<<ceil_div(F, 256), 256, 0, st>>>(L, ldl, F);
    PPBO_LAUNCH_CHECK();
    if ((rc = potrf_lower(L, ldl, F, dinv, info_d, st))) return rc;
    if (!info_h) return PPBO_OK;
    int info = 0;
    PPBO_CUDA_CHECK(readback().add(&info, info_d, sizeof(int), st));
    PPBO_CUDA_CHECK(readback().finish(st));
    *info_h = info;
    if (info) set_error("exact weight-space Hessian not positive definite (pivot %d)", info);
    return info;
}

extern "C" int ppbo_rff_eval_argmax(const double* Omega, long long ldo, int S, int F, const double* PhiT_grid, long long ldp,
                                    long long stridePhi, int P, int batch, double* fmax, int* arg, double* Fs_full,
                                    void* stream) {
    PPBO_REQUIRE(S >= 0 && F >= 1 && P >= 1 && batch >= 1, "shape");
    GemmOperands g{Omega, ldo, 0, PhiT_grid, ldp, stridePhi, S, P, F};
    RowMaxEpilogue ep{nullptr, 0, fmax, arg, Fs_full, P, (long long)S * P};
    return launch_gemm_nt_rowmax(g, ep, batch, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ posterior weight samples
namespace ppbo {

// out[i] = normal number (offset + i) of the stream; element e lives in counter e/2, slot e%2
__global__ void __launch_bounds__(256) normal_fill_kernel(unsigned long long seed, uint32_t stream, long long offset,
                                                          double* __restrict__ out, long long n) {
    const long long first = offset >> 1, last = (offset + n - 1) >> 1;          // counters touched
    for (long long c = first + (long long)blockIdx.x * blockDim.x + threadIdx.x; c <= last;
         c += (long long)gridDim.x * blockDim.x) {
        double z0, z1;
        philox_normal2(seed, (unsigned long long)c, stream, z0, z1);
        const long long e0 = 2 * c - offset, e1 = e0 + 1;
        if (e0 >= 0 && e0 < n) out[e0] = z0;
        if (e1 >= 0 && e1 < n) out[e1] = z1;
    }
}

// Omega[s][f] = omega_map[f] + z[s][f] / sqrt(-hess_diag[f])   (Hsampler.sample_omega with the diagonal Laplace covariance,
// src/random_fourier_sampler.py:134-137,207-213).  Z == nullptr: z is normal number ((sample0 + s) * F + f) of the Philox stream.
__global__ void __launch_bounds__(256) sample_omega_kernel(const double* __restrict__ omega_map,
                                                           const double* __restrict__ hess_diag,
                                                           const double* __restrict__ Z, long long ldz,
                                                           unsigned long long seed, uint32_t stream, long long sample0, int S,
                                                           int F, double* __restrict__ Omega, long long ldo) {
    const int s = blockIdx.y;
    const int fp = blockIdx.x * blockDim.x + threadIdx.x;        // pair index: features 2fp, 2fp+1
    const int f0 = 2 * fp;
    if (f0 >= F) return;
    double z0, z1 = 0.0;
    if (Z) {
        z0 = Z[(long long)s * ldz + f0];
        if (f0 + 1 < F) z1 = Z[(long long)s * ldz + f0 + 1];
    } else {
        const long long e = (sample0 + s) * (long long)F + f0;   // global normal index of (s, f0)
        if ((e & 1) == 0) {
            philox_normal2(seed, (unsigned long long)(e >> 1), stream, z0, z1);
        } else {                                                  // odd F: the pair straddles two counters
            double a, b;
            philox_normal2(seed, (unsigned long long)(e >> 1), stream, a, b);
            z0 = b;
            philox_normal2(seed, (unsigned long long)((e + 1) >> 1), stream, a, b);
            z1 = a;
        }
    }
    double* o = Omega + (long long)s * ldo;
    o[f0] = omega_map[f0] + z0 * rsqrt(-hess_diag[f0]);
    if (f0 + 1 < F) o[f0 + 1] = omega_map[f0 + 1] + z1 * rsqrt(-hess_diag[f0 + 1]);
}

// Omega[s][:] = omega_map (the mean the full-covariance draw adds to Z L^-1)
__global__ void __launch_bounds__(256) rows_fill_kernel(const double* __restrict__ v, int F, double* __restrict__ Out, long long ld) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < F) Out[(long long)blockIdx.y * ld + f] = v[f];
}

int set_identity(double* A, long long ld, int n, cudaStream_t st);   // gram.cu

}  // namespace ppbo

extern "C" int ppbo_normal_fill(unsigned long long seed, unsigned int stream_id, long long offset, double* out, long long n,
                                void* stream) {
    PPBO_REQUIRE(n >= 0 && offset >= 0, "shape");
    if (n == 0) return PPBO_OK;
    const long long counters = ((offset + n - 1) >> 1) - (offset >> 1) + 1;
    const int blocks = (int)std::min<long long>(ceil_div_ll(counters, 256), PPBO_SM_COUNT * 16);
    PPBO_CL normal_fill_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(seed, stream_id, offset, out, n);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_rff_sample_omega(const double* omega_map, const double* hess_diag, const double* Z, long long ldz,
                                     unsigned long long seed, unsigned int stream_id, long long sample0, int S, int F,
                                     double* Omega, long long ldo, void* stream) {
    PPBO_REQUIRE(S >= 0 && F >= 1 && ldo >= F, "shape");
    PPBO_REQUIRE(S <= 65535 * 1024, "too many samples for one launch");
    if (S == 0) return PPBO_OK;
    // grid.y is limited to 65535: split the launch over row blocks
    for (int s0 = 0; s0 < S; s0 += 65535) {
        const int rows = std::min(65535, S - s0);
        dim3 grid(ceil_div((F + 1) / 2, 256), rows);
        PPBO_CL sample_omega_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(omega_map, hess_diag, Z ? Z + (long long)s0 * ldz : nullptr,
                                                                    ldz, seed, stream_id, sample0 + s0, rows, F,
                                                                    Omega + (long long)s0 * ldo, ldo);
    }
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

/* Omega = 1 omega_map' + Z L^-1 with H = L L' the factor of ppbo_rff_hessian_factor: draws from N(omega_map, H^-1).  L^-1 is applied as
 * (L^-T)' with L^-T formed once (the triangular solve of the identity of ppbo_potri_lower), then one GEMM over the S rows. */
extern "C" long long ppbo_rff_sample_omega_full_workspace_bytes(int S, int F) {
    return ((long long)F * F + (long long)S * F) * 8;
}

extern "C" int ppbo_rff_sample_omega_full(const double* omega_map, const double* L, long long ldl, const double* Z, long long ldz,
                                          unsigned long long seed, unsigned int stream_id, long long sample0, int S, int F,
                                          double* Omega, long long ldo, void* workspace, long long workspace_bytes, void* stream) {
    PPBO_REQUIRE(S >= 0 && F >= 1 && ldl >= F && ldo >= F && (Z == nullptr || ldz >= F), "shape");
    PPBO_REQUIRE(S <= 65535, "at most 65535 samples per call");
    PPBO_REQUIRE(workspace_bytes >= ppbo_rff_sample_omega_full_workspace_bytes(S, F), "workspace too small");
    if (S == 0) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    double* LinvT = (double*)workspace;
    int rc;
    if ((rc = set_identity(LinvT, F, F, st))) return rc;
    if ((rc = trsm_right_lower_t(L, ldl, F, L + (long long)F * ldl, LinvT, F, F, st))) return rc;     // L^-T (upper)
    if (!Z) {
        double* Zw = LinvT + (long long)F * F;
        if ((rc = ppbo_normal_fill(seed, stream_id, sample0 * F, Zw, (long long)S * F, stream))) return rc;
        Z = Zw;
        ldz = F;
    }
    PPBO_CL rows_fill_kernel<<<dim3(ceil_div(F, 256), S), 256, 0, st>>>(omega_map, F, Omega, ldo);
    PPBO_LAUNCH_CHECK();
    GemmOperands g{Z, ldz, 0, LinvT, F, 0, S, F, F};
    StoreEpilogue ep{Omega, ldo, 0, 1.0, 1.0, 0, 0, 0};              // Omega = Z (L^-T)' + 1 omega'
    return launch_gemm_nt(g, ep, 1, st);
}
