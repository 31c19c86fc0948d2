// ppbo_b200 -- K2: preference-likelihood terms and the Laplace (MAP) fit on sm_100a.
// Replaces GPModel.sum_Phi / T / T_grad / create_Lambda (src/gp_model.py:176-274) and the scipy trust-exact
// driver of GPModel.update_fMAP (src/gp_model.py:354-389).
//
// Formulation (DESIGN.md "Laplace fit"): with B the N x Qm incidence matrix of the comparison sets
// (column (q,j): +1 at pseudo-observation row, -1 at the winner row), the negative likelihood Hessian is
// W = B diag(a) B^T with a_qj = -Delta phi~(Delta) / (2 m sigma^2).  A damped Newton step with a+ = max(a,0) is
//     alpha_new = b - B a+^1/2 (I + a+^1/2 G a+^1/2)^-1 a+^1/2 B^T Sigma b ,   b = B a+ B^T f + beta ,  f_new = Sigma alpha_new
// where G = B^T Sigma B (Qm x Qm) is fixed during the fit.  One Cholesky of size Qm per step, no Sigma^-1.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include <cooperative_groups.h>

#include "../../include/ppbo_b200.h"
#include "common.cuh"
#include "gemm_f64.cuh"
#include "linalg.cuh"

namespace ppbo {

int diffspace_gram(const double* S, long long lds, int Q, int m, double* G, long long ldg, cudaStream_t st);
int newton_matrix(const double* G, long long ldg, int M, const double* sa, double* out, long long ldo, cudaStream_t st);

__device__ __forceinline__ double phi_tilde(double x) {           // density of N(0,2), src/misc.py:134-135
    return 0.28209479177387814 * exp(-0.25 * x * x);             // 1/sqrt(4 pi)
}
__device__ __forceinline__ double Phi_tilde(double x) {           // Phi(x / sqrt2) == GH-200 quadrature of src/gp_model.py:192
    return 0.5 * erfc(-0.5 * x);
}

// One warp per comparison set.  Outputs are optional (nullptr to skip).
//   set_lik[q] = sum_j Phi~(Delta_qj)        beta[N]        arrow[Qm] (signed a)       sa[Qm] = sqrt(max(a,0))
//   bvec[N]    = B a+ B^T f + beta           (Newton right-hand side)      ap_out[Qm] = a+
//   ap_fixed  : when given, bvec is built with these a+ instead of the current ones.  No caller passes it, but without the
//               parameter ptxas spills 32 bytes in this kernel instead of 12.
__global__ void __launch_bounds__(256) lik_terms_kernel(const double* __restrict__ f, int Q, int m, double sigma,
                                                        double* __restrict__ set_lik, double* __restrict__ beta,
                                                        double* __restrict__ arrow, double* __restrict__ sa,
                                                        double* __restrict__ bvec, const double* __restrict__ ap_fixed = nullptr,
                                                        double* __restrict__ ap_out = nullptr) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= Q) return;
    const long long base = (long long)q * (m + 1);
    const double fw = f[base];
    const double inv_s = 1.0 / sigma, cg = 1.0 / (sigma * m), ca = 0.5 / (m * sigma * sigma);
    double s_lik = 0.0, s_phi = 0.0, s_ad = 0.0;
    for (int j = lane; j < m; j += 32) {
        const double diff = f[base + 1 + j] - fw;
        const double dl = diff * inv_s;
        const double ph = phi_tilde(dl);
        const double a = -ca * dl * ph;
        const double ap = ap_fixed ? ap_fixed[(long long)q * m + j] : (a > 0.0 ? a : 0.0);
        if (ap_out) ap_out[(long long)q * m + j] = ap;
        s_lik += Phi_tilde(dl);
        s_phi += ph;
        s_ad += ap * diff;
        if (beta) beta[base + 1 + j] = -ph * cg;
        if (arrow) arrow[(long long)q * m + j] = a;
        if (sa) sa[(long long)q * m + j] = sqrt(ap);
        if (bvec) bvec[base + 1 + j] = ap * diff - ph * cg;
    }
    for (int o = 16; o > 0; o >>= 1) {
        s_lik += __shfl_xor_sync(0xffffffffu, s_lik, o);
        s_phi += __shfl_xor_sync(0xffffffffu, s_phi, o);
        s_ad += __shfl_xor_sync(0xffffffffu, s_ad, o);
    }
    if (lane == 0) {
        if (set_lik) set_lik[q] = s_lik;
        if (beta) beta[base] = s_phi * cg;
        if (bvec) bvec[base] = -s_ad + s_phi * cg;
    }
}

// out[0] = sum_i x[i]  in a fixed order (single CTA) -> bit-reproducible
__global__ void __launch_bounds__(1024) sum_kernel(const double* __restrict__ x, int n, double* __restrict__ out) {
    __shared__ double red[33];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 1024) s += x[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[0] = s;
}

// out[0] = x . y in a fixed order (single CTA)
__global__ void __launch_bounds__(1024) dot_kernel(const double* __restrict__ x, const double* __restrict__ y, int n,
                                                   double* __restrict__ out) {
    __shared__ double red[33];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 1024) s = fma(x[i], y[i], s);
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[0] = s;
}

// t[u] = sa[u] * (v[r(u)] - v[w(u)])                       (a+^1/2 B^T v)
__global__ void diff_scale_kernel(const double* __restrict__ v, const double* __restrict__ sa, int Q, int m,
                                  double* __restrict__ t) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= Q * m) return;
    const int q = u / m, j = u % m;
    const long long w = (long long)q * (m + 1);
    t[u] = sa[u] * (v[w + 1 + j] - v[w]);
}

// alpha_new = b - B (sa .* y);  dalpha = alpha_new - alpha  (one warp per set)
__global__ void __launch_bounds__(256) alpha_update_kernel(const double* __restrict__ bvec, const double* __restrict__ sa,
                                                           const double* __restrict__ y, const double* __restrict__ alpha,
                                                           int Q, int m, double* __restrict__ dalpha) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= Q) return;
    const long long base = (long long)q * (m + 1);
    double s = 0.0;
    for (int j = lane; j < m; j += 32) {
        const double u = sa[(long long)q * m + j] * y[(long long)q * m + j];
        s += u;
        dalpha[base + 1 + j] = bvec[base + 1 + j] - u - alpha[base + 1 + j];
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) dalpha[base] = bvec[base] + s - alpha[base];
}

// Line search data: for step sizes s_c = 2^-c, c = 0..NSTEP-1 (blockIdx.y = c):
//   part[c][q] = sum_j Phi~(Delta_qj(f + s_c df))
constexpr int NSTEP = 8;
__global__ void __launch_bounds__(256) linesearch_lik_kernel(const double* __restrict__ f, const double* __restrict__ df,
                                                             int Q, int m, double sigma, double* __restrict__ part) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= Q) return;
    const double step = ldexp(1.0, -(int)blockIdx.y);
    const long long base = (long long)q * (m + 1);
    const double fw = f[base] + step * df[base];
    const double inv_s = 1.0 / sigma;
    double s = 0.0;
    for (int j = lane; j < m; j += 32) s += Phi_tilde((f[base + 1 + j] + step * df[base + 1 + j] - fw) * inv_s);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) part[(long long)blockIdx.y * Q + q] = s;
}

// scal[0..3] = alpha.f, alpha.df, dalpha.f, dalpha.df ; scal[4] = max|df| ; scal[5] = max|f| ;
// scal[8 + c] = sum_q part[c][q]     (single CTA, fixed order)
__global__ void __launch_bounds__(1024) newton_scalars_kernel(const double* __restrict__ alpha, const double* __restrict__ dalpha,
                                                              const double* __restrict__ f, const double* __restrict__ df,
                                                              int N, const double* __restrict__ part, int Q,
                                                              double* __restrict__ scal) {
    __shared__ double red[33];
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0, mdf = 0, mf = 0;
    for (int i = threadIdx.x; i < N; i += 1024) {
        const double a = alpha[i], da = dalpha[i], fi = f[i], dfi = df[i];
        s0 = fma(a, fi, s0);
        s1 = fma(a, dfi, s1);
        s2 = fma(da, fi, s2);
        s3 = fma(da, dfi, s3);
        mdf = fmax(mdf, fabs(dfi));
        mf = fmax(mf, fabs(fi));
    }
    s0 = block_sum(s0, red);
    s1 = block_sum(s1, red);
    s2 = block_sum(s2, red);
    s3 = block_sum(s3, red);
    for (int o = 16; o > 0; o >>= 1) {
        mdf = fmax(mdf, __shfl_xor_sync(0xffffffffu, mdf, o));
        mf = fmax(mf, __shfl_xor_sync(0xffffffffu, mf, o));
    }
    __shared__ double mx[2][32];
    if ((threadIdx.x & 31) == 0) { mx[0][threadIdx.x >> 5] = mdf; mx[1][threadIdx.x >> 5] = mf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) { mdf = fmax(mdf, mx[0][w]); mf = fmax(mf, mx[1][w]); }
        scal[0] = s0; scal[1] = s1; scal[2] = s2; scal[3] = s3; scal[4] = mdf; scal[5] = mf;
    }
    for (int c = 0; c < NSTEP; ++c) {
        double s = 0.0;
        for (int q = threadIdx.x; q < Q; q += 1024) s += part[(long long)c * Q + q];
        s = block_sum(s, red);
        if (threadIdx.x == 0) scal[8 + c] = s;
    }
}

__global__ void axpy2_kernel(double* __restrict__ alpha, const double* __restrict__ dalpha, double* __restrict__ f,
                             const double* __restrict__ df, double step, int N) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) {
        alpha[i] += step * dalpha[i];
        f[i] += step * df[i];
    }
}

// Device-side acceptance test of one chord step, so that a batch of chord steps runs without a host round trip (a host decision
// per step left the launch queue empty after every synchronise: ~0.5 ms per step against ~0.25 ms of kernel time).
//   state[0] T at the current iterate   state[1] relative size of the last residual   state[2] the one before   state[3] last |df|
//   state[4] 0 = keep going, 1 = converged, 2 = contraction too slow (refactor), 3 = full step rejected (refactor)
//   state[5] chord steps taken in this batch      state[6] tolerance         state[7] step length omega of the queued step
//   state[8] previous contraction ratio           state[9] steps to wait before the next extrapolation
//   state[10] slowest contraction per step that is still cheaper than a new factor (0.5 after a Newton step of this fit; 0.85 for
//             the factor of the previous PPBO iteration: a chord step costs ~1/12 of a factorisation there and a refactorisation
//             is followed by one or two more)
//   state[11] residual three accepted steps ago    state[13] 1 = the steps of this batch are mixed by chord_anderson_kernel
//   state[14] 1 = the last call took a plain full step
//   hist[2i], hist[2i+1] = (rel, T) of step i
// A chord step of length 1 is only taken when T(alpha + dalpha) does not fall below T (same rule as the host line search with
// c == 0).  When state[4] != 0 this kernel and every other kernel of a queued step return at once (skip flag).
//
// Extrapolation: the chord iteration is a linear fixed-point iteration near the mode; once two successive contraction ratios
// agree to 8 % a single eigen-direction dominates the error and the NEXT step is taken with omega = 1 / (1 - ratio) (Aitken's
// delta-squared written as a step length, capped at 2), which removes that direction in one step.  An extrapolated step that
// lowers T is not taken: the step is repeated with omega = 1.
__global__ void __launch_bounds__(1024) chord_decide_kernel(double* __restrict__ alpha, const double* __restrict__ dalpha,
                                                            double* __restrict__ f, const double* __restrict__ df, int N,
                                                            const double* __restrict__ part, int Q, int m,
                                                            double* __restrict__ state, double* __restrict__ hist, int extrapolate,
                                                            const double* __restrict__ part0) {
    __shared__ double mx[2][32];
    __shared__ double step_s;
    if (state[4] != 0.0) return;                    // uniform: state[4] is only written after the barriers below
    const double omega = state[7];
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0, mdf = 0, mf = 0, lik = 0, lik0 = 0;
#pragma unroll 4
    for (int i = threadIdx.x; i < N; i += 1024) {
        const double a = alpha[i], da = dalpha[i], fi = f[i], dfi = df[i];
        s0 = fma(a, fi, s0);
        s1 = fma(a, dfi, s1);
        s2 = fma(da, fi, s2);
        s3 = fma(da, dfi, s3);
        mdf = fmax(mdf, fabs(dfi));
        mf = fmax(mf, fabs(fi));
    }
    for (int q = threadIdx.x; q < Q; q += 1024) {
        lik += part[q];
        if (part0) lik0 += part0[q];
    }
    {
        __shared__ double red6[32 * 6];
        double sums[6] = {s0, s1, s2, s3, lik, lik0};
        block_sum_multi<6>(sums, red6);               // one pair of barriers for all six sums
        s0 = sums[0]; s1 = sums[1]; s2 = sums[2]; s3 = sums[3]; lik = sums[4]; lik0 = sums[5];
    }
    for (int o = 16; o > 0; o >>= 1) {
        mdf = fmax(mdf, __shfl_xor_sync(0xffffffffu, mdf, o));
        mf = fmax(mf, __shfl_xor_sync(0xffffffffu, mf, o));
    }
    if ((threadIdx.x & 31) == 0) { mx[0][threadIdx.x >> 5] = mdf; mx[1][threadIdx.x >> 5] = mf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) { mdf = fmax(mdf, mx[0][w]); mf = fmax(mf, mx[1][w]); }
        const double T_cur = part0 ? (-0.5 * s0 - lik0 / m) : state[0];
        const double T1 = -0.5 * (s0 + omega * (s1 + s2) + omega * omega * s3) - lik / m;
        const bool accept = T1 >= T_cur - 1e-13 * fabs(T_cur);
        double step = 0.0;
        state[14] = (accept && omega == 1.0) ? 1.0 : 0.0;               // a plain full step was taken (chord_anderson_kernel)
        if (!accept) {
            if (omega > 1.0) { state[7] = 1.0; state[9] = 4.0; }       // repeat this step at full length, no extrapolation for a while
            else if (omega > 0.2) { state[7] = 0.5 * omega; state[9] = 4.0; }   // backtrack along the same direction (appended rows start
                                                                        // where the likelihood curvature vanishes: their first
                                                                        // Newton step overshoots like the cold start's does)
            else state[4] = 3.0;
        } else {
            step = omega;
            const double rel = mdf / fmax(mf, 1e-300), prev = state[1];
            const int n = (int)state[5];
            const double rel3 = state[11];                                 // residual three accepted steps ago
            state[11] = state[2];
            state[0] = T1;
            state[2] = prev;
            state[1] = rel;
            state[3] = mdf;
            state[5] = n + 1;
            hist[2 * n] = rel;
            hist[2 * n + 1] = T1;
            const double ratio = rel / prev, ratio_prev = state[8];
            double wait = state[9], next_omega = 1.0;
            const bool after_extrapolation = omega != 1.0;
            if (rel <= state[6]) {
                state[4] = 1.0;
            } else if (state[13] == 1.0) {
                // mixed (Anderson) steps are not monotone step by step: judge them over three steps
                if (rel3 < 1e300 && !(rel <= 0.5 * rel3)) state[4] = 2.0;
            } else if (!after_extrapolation && wait <= 0.0 && !(rel <= state[10] * prev)) {
                state[4] = 2.0;                                        // plain steps contract too slowly: pay for a new factor
            } else if (wait > 0.0 && !(rel <= 4.0 * prev)) {
                state[4] = 2.0;                                        // residual grows after an extrapolation: give up on this factor
            } else if (extrapolate && !after_extrapolation && wait <= 0.0 && ratio > 0.02 && ratio < 0.4 &&
                       fabs(ratio - ratio_prev) <= 0.08 * ratio) {
                // (ratio < 0.4: with slower contraction the error is spread over many eigen-directions and the long step
                // overshoots the others -- measured on a factor that contracted at 0.45: the residual rose after every extrapolation)
                next_omega = fmin(1.0 / (1.0 - ratio), 2.0);
                wait = 3.0;                                            // the ratios right after an extrapolation say nothing
            }
            state[8] = after_extrapolation ? 0.0 : ratio;
            state[9] = fmax(wait - 1.0, 0.0);
            state[7] = next_omega;
        }
        step_s = step;
    }
    __syncthreads();
    const double step = step_s;
    if (step == 0.0) return;
#pragma unroll 4
    for (int i = threadIdx.x; i < N; i += 1024) {
        alpha[i] = fma(step, dalpha[i], alpha[i]);
        f[i] = fma(step, df[i], f[i]);
    }
}

// Anderson acceleration of the chord iteration (depth AA_M).  The chord iteration x <- g(x) is, near the mode, a linear fixed-point
// iteration whose matrix (Sigma^-1 + W0)^-1 (W0 - W) has a real spectrum of radius rho (0.2 .. 0.8 depending on how stale the
// coefficients W0 of the factor are); plain iteration gains a factor rho per step, mixing the last AA_M residual differences
// (a Krylov method on the linearised problem) about rho / (1 + sqrt(1 - rho^2)).  After chord_decide_kernel has taken a plain full
// step -- alpha = g_a(x_k), f = g_f(x_k), residual r_k = df still in memory -- this kernel
//   * appends the differences (r_k - r_{k-1}, g_k - g_{k-1}) to the history,
//   * solves min_gamma | r_k - dR gamma |_2 (normal equations of order <= AA_M, Tikhonov-damped) and
//   * replaces (alpha, f) by g_k - dG gamma   (f = Sigma alpha is preserved: both are the same combination).
// The history is dropped when a step was damped / extrapolated / rejected, or when the residual grew.  Fixed summation order.
constexpr int AA_M = 5;
constexpr int AA_CL = 8;       // fixed element slices per call: one per CTA
constexpr int AA_NPAIR = AA_M * (AA_M + 1) / 2, AA_NV = AA_NPAIR + AA_M;
constexpr int AA_STATE = 8 + AA_CL * AA_NV + AA_M + 3;      // aa: 8 doubles of state, then scratch of the three-launch variant
//   aa: [0] history length, [1] next slot, [2] residual norm (max |df| / max |f|) seen by the previous call, [3] 1 = (prev r, g) valid
//       [8 ..) partial sums [AA_CL][AA_NV], mixing coefficients [AA_M], their count (three-launch variant)
//   H: [3 * AA_M + 3][N]: dR[AA_M], dGf[AA_M], dGa[AA_M], prev r, prev g_f, prev g_a
// One call moves ~32 N doubles through dependent global round trips; a single CTA needs 41-83 us for that at N = 5200 (one SM's
// load path).  The elements are cut into AA_CL = 8 fixed slices, one per CTA; the partial sums of the normal equations are added
// in slice order and the 5 x 5 system is solved by the same code wherever it runs, so both variants below return the same bits:
//   * chord_anderson_kernel: ONE launch of a thread-block cluster of 8 CTAs, partial sums through distributed shared memory, every
//     CTA solves redundantly (17 us).  Used by fits on a foreground host thread.
//   * chord_anderson_{sums,solve,apply}_kernel: three ordinary launches (8 CTAs, 1 warp, 8 CTAs; partial sums through global
//     memory).  Used by fits on a background host thread -- the GP chain of the overlapped one-GPU pipeline, which lives on the
//     16-32 SMs the sampling contraction leaves free: eight co-scheduled 1024-thread CTAs rarely find room there (the chain stalled
//     for milliseconds waiting for a slot: +1.8 ms on the cold iteration), and a cluster of one took 46-83 us per call.
struct AaView {
    double *dR, *dGf, *dGa, *pr, *pgf, *pga;
    __device__ AaView(double* H, int N)
        : dR(H), dGf(H + (long long)AA_M * N), dGa(H + 2LL * AA_M * N), pr(H + 3LL * AA_M * N), pgf(pr + N), pga(pgf + N) {}
};
// what every CTA of a call derives from the state: false = leave (nothing to mix); nh / slot / have_prev describe the history the
// call works with BEFORE its own append
struct AaPlan { int nh, slot; bool have_prev, reset, run; };
__device__ __forceinline__ AaPlan aa_plan(const double* __restrict__ state, const double* __restrict__ aa) {
    AaPlan p;
    const double stop = state[4];
    const bool plain = state[14] == 1.0;
    const double rel = state[1], rel_prev = aa[2];
    p.nh = (int)aa[0];
    p.slot = (int)aa[1];
    p.have_prev = aa[3] == 1.0;
    p.reset = false;
    p.run = !(stop == 1.0 || stop == 3.0);            // converged or rejected for good: nothing to mix
    if (p.run && (!plain || (p.have_prev && rel > 1.5 * rel_prev))) {
        // a damped / extrapolated / rejected step, or a residual that grew: the history no longer describes one linear map
        p.reset = true;
        if (!plain) p.run = false;
        p.nh = 0;
        p.slot = 0;
        p.have_prev = false;
    }
    return p;
}
// slice v: append the newest differences (needs the previous (r, g)) and remember the current ones
__device__ __forceinline__ void aa_slice_append(const AaView& h, const double* __restrict__ df, const double* __restrict__ f,
                                                const double* __restrict__ alpha, int N, int v, int slot, bool have_prev) {
    const int per = (N + AA_CL - 1) / AA_CL, lo = v * per, hi = min(N, lo + per);
    double* dRs = h.dR + (long long)slot * N;
    double* dGfs = h.dGf + (long long)slot * N;
    double* dGas = h.dGa + (long long)slot * N;
    for (int i = lo + threadIdx.x; i < hi; i += 1024) {
        const double r = df[i], gf = f[i], ga = alpha[i];
        if (have_prev) {
            dRs[i] = r - h.pr[i];
            dGfs[i] = gf - h.pgf[i];
            dGas[i] = ga - h.pga[i];
        }
        h.pr[i] = r;
        h.pgf[i] = gf;
        h.pga[i] = ga;
    }
}
// slice v: all products of the normal equations A_ij = <dR_i, dR_j>, b_i = <dR_i, r> in one pass + one multi-value block reduction;
// every thread returns the slice totals in acc.  (A thread only re-reads elements it wrote itself in aa_slice_append.)
__device__ __forceinline__ void aa_slice_products(const AaView& h, const double* __restrict__ df, int N, int v, int nh,
                                                  double (&acc)[AA_NV], double* red_multi) {
    const int per = (N + AA_CL - 1) / AA_CL, lo = v * per, hi = min(N, lo + per);
#pragma unroll
    for (int i = 0; i < AA_NV; ++i) acc[i] = 0.0;
    for (int k = lo + threadIdx.x; k < hi; k += 1024) {
        double dv[AA_M];
#pragma unroll
        for (int i = 0; i < AA_M; ++i) dv[i] = (i < nh) ? h.dR[(long long)i * N + k] : 0.0;
        const double rk = df[k];
        int idx = 0;
#pragma unroll
        for (int i = 0; i < AA_M; ++i) {
#pragma unroll
            for (int j = 0; j <= i; ++j) { acc[idx] = fma(dv[i], dv[j], acc[idx]); ++idx; }
            acc[AA_NPAIR + i] = fma(dv[i], rk, acc[AA_NPAIR + i]);
        }
    }
    block_sum_multi<AA_NV>(acc, red_multi);
}
// one thread: min_gamma | r - dR gamma |_2 from the totals (normal equations of order nh, Tikhonov-damped, Gaussian elimination with
// partial pivoting); returns the number of coefficients to apply (0: none)
__device__ __forceinline__ int aa_solve(const double (&tot)[AA_NV], int nh, double* gam) {
    double A[AA_M][AA_M], bb[AA_M];
    int idx = 0;
#pragma unroll
    for (int i = 0; i < AA_M; ++i) {
#pragma unroll
        for (int j = 0; j <= i; ++j) { A[i][j] = A[j][i] = tot[idx]; ++idx; }
        bb[i] = tot[AA_NPAIR + i];
    }
    double tr = 0.0;
    for (int i = 0; i < nh; ++i) tr += A[i][i];
    for (int i = 0; i < nh; ++i) A[i][i] += 1e-10 * tr + 1e-300;     // damping: nearly collinear differences
    bool ok = true;
    for (int c = 0; c < nh && ok; ++c) {
        int p = c;
        for (int r2 = c + 1; r2 < nh; ++r2) if (fabs(A[r2][c]) > fabs(A[p][c])) p = r2;
        if (A[p][c] == 0.0) { ok = false; break; }
        for (int k = 0; k < nh; ++k) { const double t = A[c][k]; A[c][k] = A[p][k]; A[p][k] = t; }
        { const double t = bb[c]; bb[c] = bb[p]; bb[p] = t; }
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
    return ok ? nh : 0;
}
// slice v: (alpha, f) <- g_k - dG gamma
__device__ __forceinline__ void aa_slice_apply(const AaView& h, double* __restrict__ alpha, double* __restrict__ f, int N, int v,
                                               int nm, const double* gam) {
    const int per = (N + AA_CL - 1) / AA_CL, lo = v * per, hi = min(N, lo + per);
    for (int i = lo + threadIdx.x; i < hi; i += 1024) {
        double cf = 0.0, ca = 0.0;
        for (int j = 0; j < nm; ++j) {
            cf = fma(gam[j], h.dGf[(long long)j * N + i], cf);
            ca = fma(gam[j], h.dGa[(long long)j * N + i], ca);
        }
        f[i] -= cf;
        alpha[i] -= ca;
    }
}

__global__ void __launch_bounds__(1024)
chord_anderson_kernel(double* __restrict__ alpha, double* __restrict__ f, const double* __restrict__ df, int N,
                      const double* __restrict__ state, double* __restrict__ aa, double* __restrict__ H) {
    namespace cg = cooperative_groups;
    cg::cluster_group cl = cg::this_cluster();
    const int rank = (int)cl.block_rank();                               // cluster of AA_CL CTAs: CTA rank owns slice rank
    __shared__ double part_s[AA_NV];
    __shared__ double red_multi[32 * AA_NV];
    __shared__ double gam[AA_M];
    __shared__ int nm_s;
    const AaView h(H, N);
    AaPlan p = aa_plan(state, aa);
    const double rel = state[1];
    cl.sync();                                                           // every CTA has read the state (rank 0 writes aa below)
    if (p.reset && rank == 0 && threadIdx.x == 0) { aa[0] = 0.0; aa[1] = 0.0; aa[2] = rel; aa[3] = 0.0; }
    if (!p.run) return;
    aa_slice_append(h, df, f, alpha, N, rank, p.slot, p.have_prev);
    int nh = p.nh, slot = p.slot;
    if (p.have_prev) {
        nh = min(nh + 1, AA_M);
        slot = (slot + 1) % AA_M;
    }
    double acc[AA_NV];
    aa_slice_products(h, df, N, rank, nh, acc, red_multi);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < AA_NV; ++i) part_s[i] = acc[i];
    }
    cl.sync();                                                           // every CTA's partial sums are in its shared memory
    if (threadIdx.x == 0) {
        double tot[AA_NV];
#pragma unroll
        for (int i = 0; i < AA_NV; ++i) tot[i] = 0.0;
        for (int v = 0; v < AA_CL; ++v) {                                // fixed order (by slice): identical totals in every CTA
            const double* rp = cl.map_shared_rank(part_s, (unsigned)v);
#pragma unroll
            for (int i = 0; i < AA_NV; ++i) tot[i] += rp[i];
        }
        const int nm = aa_solve(tot, nh, gam);
        nm_s = nm;
        if (rank == 0) {
            aa[0] = nm;
            aa[1] = nm ? slot : 0;
            aa[2] = rel;
            aa[3] = 1.0;                                                  // (prev r, g) are valid from now on
        }
    }
    __syncthreads();
    aa_slice_apply(h, alpha, f, N, rank, nm_s, gam);
    cl.sync();                                  // nobody leaves while another CTA may still read its partial sums
}

// ---- the same call as three ordinary launches (see above)
__global__ void __launch_bounds__(1024)
chord_anderson_sums_kernel(const double* __restrict__ alpha, const double* __restrict__ f, const double* __restrict__ df, int N,
                           const double* __restrict__ state, double* __restrict__ aa, double* __restrict__ H) {
    __shared__ double red_multi[32 * AA_NV];
    const AaView h(H, N);
    const AaPlan p = aa_plan(state, aa);                                 // (aa is not written before the solve kernel)
    if (!p.run) return;
    aa_slice_append(h, df, f, alpha, N, blockIdx.x, p.slot, p.have_prev);
    const int nh = p.have_prev ? min(p.nh + 1, AA_M) : p.nh;
    double acc[AA_NV];
    aa_slice_products(h, df, N, blockIdx.x, nh, acc, red_multi);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < AA_NV; ++i) aa[8 + blockIdx.x * AA_NV + i] = acc[i];
    }
}
__global__ void chord_anderson_solve_kernel(const double* __restrict__ state, double* __restrict__ aa) {
    if (threadIdx.x != 0) return;
    double* gam_g = aa + 8 + AA_CL * AA_NV;
    const AaPlan p = aa_plan(state, aa);
    const double rel = state[1];
    gam_g[AA_M] = 0.0;                                                   // number of coefficients the apply kernel uses
    if (p.reset) { aa[0] = 0.0; aa[1] = 0.0; aa[2] = rel; aa[3] = 0.0; }
    if (!p.run) return;
    int nh = p.nh, slot = p.slot;
    if (p.have_prev) {
        nh = min(nh + 1, AA_M);
        slot = (slot + 1) % AA_M;
    }
    double tot[AA_NV];
#pragma unroll
    for (int i = 0; i < AA_NV; ++i) tot[i] = 0.0;
    for (int v = 0; v < AA_CL; ++v) {
#pragma unroll
        for (int i = 0; i < AA_NV; ++i) tot[i] += aa[8 + v * AA_NV + i];
    }
    double gam[AA_M];
    const int nm = aa_solve(tot, nh, gam);
    for (int i = 0; i < AA_M; ++i) gam_g[i] = i < nm ? gam[i] : 0.0;
    gam_g[AA_M] = nm;
    aa[0] = nm;
    aa[1] = nm ? slot : 0;
    aa[2] = rel;
    aa[3] = 1.0;
}
__global__ void __launch_bounds__(1024)
chord_anderson_apply_kernel(double* __restrict__ alpha, double* __restrict__ f, int N, const double* __restrict__ aa,
                            double* __restrict__ H) {
    __shared__ double gam[AA_M];
    const double* gam_g = aa + 8 + AA_CL * AA_NV;
    const int nm = (int)gam_g[AA_M];
    if (nm == 0) return;
    if (threadIdx.x < AA_M) gam[threadIdx.x] = gam_g[threadIdx.x];
    __syncthreads();
    const AaView h(H, N);
    aa_slice_apply(h, alpha, f, N, blockIdx.x, nm, gam);
}

// dense Lambda (public attr GPModel.Lambda_MAP): one thread per row of the output
__global__ void lambda_dense_kernel(const double* __restrict__ arrow, int Q, int m, double* __restrict__ out, long long ld) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int N = Q * (m + 1);
    if (idx >= (long long)N * N) return;
    const int i = (int)(idx / N), j = (int)(idx % N);
    const int qi = i / (m + 1), ri = i % (m + 1), qj = j / (m + 1), rj = j % (m + 1);
    double v = 0.0;
    if (qi == qj) {
        const double* a = arrow + (long long)qi * m;
        if (ri == 0 && rj == 0) { for (int t = 0; t < m; ++t) v -= a[t]; }
        else if (ri == 0) v = a[rj - 1];
        else if (rj == 0) v = a[ri - 1];
        else if (ri == rj) v = -a[ri - 1];
    }
    out[(long long)i * ld + j] = v;
}

// out = I + sign * Sigma W with W = B diag(a) B' = -Lambda (signed coefficients): the matrix whose determinant enters the
// Laplace evidence.  sign = +1: I + Sigma W (posterior precision times prior covariance); sign = -1: I + Sigma Lambda, the matrix
// the reference factors (src/gp_model.py:301-302).  Column c of set q:  winner:  sum_j a_j (S[i][w] - S[i][r_j]);  pseudo-observation
// j:  a_j (S[i][r_j] - S[i][w]).
__global__ void __launch_bounds__(256) evidence_matrix_kernel(const double* __restrict__ S, long long lds, int Q, int m,
                                                              const double* __restrict__ arrow, double sign, double* __restrict__ out,
                                                              long long ldo) {
    const int N = Q * (m + 1);
    const int c = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (c >= N) return;
    const int q = c / (m + 1), rc = c % (m + 1);
    const long long w = (long long)q * (m + 1);
    const double* si = S + (long long)i * lds;
    const double* a = arrow + (long long)q * m;
    double v = 0.0;
    if (rc == 0) {
        const double sw = si[w];
        for (int j = 0; j < m; ++j) v = fma(a[j], sw - si[w + 1 + j], v);
    } else {
        v = a[rc - 1] * (si[c] - si[w]);
    }
    out[(long long)i * ldo + c] = ((i == c) ? 1.0 : 0.0) + sign * v;
}

// ---- bordered warm start ---------------------------------------------------------------------------------------------------
// After comparison sets were appended the Newton matrix is  A = [[A11, A21'], [A21, A22]]  with A11 = I + s_o G_oo s_o the system
// the previous iteration factored (L11), A21 = s_n G_no s_o and A22 = I + s_n G_nn s_n for the nb new rows.  With
//     R = (G_no s_o) L11^-T   (nb x M_old, computed ONCE per append)      C = G_nn - R R'      (nb x nb)
// the Schur complement of the new rows is  S = I + s_n C s_n  for ANY current coefficients s_n, so a solve A y = t is
//     z = L11^-1 t_o ;   y_n = S^-1 (t_n - s_n R z) ;   y_o = L11^-T (z - R' (s_n y_n))
// i.e. the old factor's two sweeps plus nb-sized work.  The new rows therefore always carry their CURRENT coefficients (a Newton
// step for them -- they start at the prior mean, where a = 0, and move by O(sigma_f)) while the old rows keep the coefficients their
// factor was built with (chord step).  This is the O(M^2 m) iteration of SURVEY.md 8f rank 2.
constexpr int BORDER_MAX = 64;           // new rows handled as a border (2 comparison sets of m = 25; more -> plain refactorisation)

// T[u][v] = G[M_old + u][v] sa[v]   (u < nb, v < M_old)
__global__ void __launch_bounds__(256) border_rows_kernel(const double* __restrict__ G, long long ldg, const double* __restrict__ sa,
                                                          int M_old, int nb, double* __restrict__ T, long long ldt) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x, u = blockIdx.y;
    if (v < M_old) T[(long long)u * ldt + v] = G[(long long)(M_old + u) * ldg + v] * sa[v];
}
// Cb[u][w] = G[M_old + u][M_old + w]
__global__ void border_corner_kernel(const double* __restrict__ G, long long ldg, int M_old, int nb, double* __restrict__ Cb) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nb * nb) Cb[e] = G[(long long)(M_old + e / nb) * ldg + M_old + e % nb];
}
// Cb[e] -= sum_p part[p][e]  (partial products R R' of the K chunks, fixed order)
__global__ void border_corner_sum_kernel(const double* __restrict__ part, int nparts, int nb, double* __restrict__ Cb) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nb * nb) return;
    double s = 0.0;
    for (int p = 0; p < nparts; ++p) s += part[(long long)p * nb * nb + e];
    Cb[e] -= s;
}
// One CTA: r = t_n - s_n (R z);  S = I + s_n C s_n;  y_n = S^-1 r  (Cholesky in shared memory);  t_n <- y_n,  w <- s_n y_n
__global__ void __launch_bounds__(1024) border_solve_kernel(const double* __restrict__ R, long long ldr, const double* __restrict__ Cb,
                                                            const double* __restrict__ s_new, const double* __restrict__ z, int M_old,
                                                            int nb, double* __restrict__ t_new, double* __restrict__ w,
                                                            const double* __restrict__ skip) {
    __shared__ double S[BORDER_MAX][BORDER_MAX + 1];
    __shared__ double r[BORDER_MAX];
    __shared__ double red_multi[32 * 16];
    if (skip && *skip != 0.0) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (nb <= 32) {
        // R z for all rows in ONE pass: a thread keeps one accumulator per row over its columns (coalesced in v), one multi-value
        // block reduction follows.  (One warp per row: 157 dependent iterations of a single warp per row, ~25 of the kernel's 35 us.)
        // (16 rows per pass: 32 accumulators would not fit the 64-register budget of a 1024-thread CTA)
        for (int u0 = 0; u0 < nb; u0 += 16) {
            double acc[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) acc[u] = 0.0;
            for (int v = tid; v < M_old; v += 1024) {
                const double zv = z[v];
#pragma unroll
                for (int u = 0; u < 16; ++u)
                    if (u0 + u < nb) acc[u] = fma(R[(long long)(u0 + u) * ldr + v], zv, acc[u]);
            }
            block_sum_multi<16>(acc, red_multi);
#pragma unroll
            for (int u = 0; u < 16; ++u)
                if (tid == u && u0 + u < nb) r[u0 + u] = t_new[u0 + u] - s_new[u0 + u] * acc[u];
        }
    } else {
        for (int u = warp; u < nb; u += 32) {
            const double* Ru = R + (long long)u * ldr;
            double a = 0.0;
            for (int v = lane; v < M_old; v += 32) a = fma(Ru[v], z[v], a);
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) r[u] = t_new[u] - s_new[u] * a;
        }
    }
    for (int e = tid; e < nb * nb; e += 1024) {
        const int u = e / nb, v = e % nb;
        S[u][v] = ((u == v) ? 1.0 : 0.0) + s_new[u] * Cb[e] * s_new[v];
    }
    __syncthreads();
    for (int k = 0; k < nb; ++k) {                         // right-looking Cholesky, lower triangle
        if (tid == 0) S[k][k] = sqrt(S[k][k]);
        __syncthreads();
        const double d = S[k][k];
        for (int i = k + 1 + tid; i < nb; i += 1024) S[i][k] /= d;
        __syncthreads();
        const int rem = nb - k - 1;
        for (int e = tid; e < rem * rem; e += 1024) {
            const int i = k + 1 + e / rem, j = k + 1 + e % rem;
            if (j <= i) S[i][j] = fma(-S[i][k], S[j][k], S[i][j]);
        }
        __syncthreads();
    }
    if (warp == 0) {                                       // two triangular solves by one warp
        for (int i = 0; i < nb; ++i) {
            double a = 0.0;
            for (int k = lane; k < i; k += 32) a = fma(S[i][k], r[k], a);
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) r[i] = (r[i] - a) / S[i][i];
            __syncwarp();
        }
        for (int i = nb - 1; i >= 0; --i) {
            double a = 0.0;
            for (int k = i + 1 + lane; k < nb; k += 32) a = fma(S[k][i], r[k], a);
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) r[i] = (r[i] - a) / S[i][i];
            __syncwarp();
        }
        for (int u = lane; u < nb; u += 32) {
            t_new[u] = r[u];
            w[u] = s_new[u] * r[u];
        }
    }
}
// z[v] -= sum_u R[u][v] w[u]
__global__ void __launch_bounds__(256) border_update_kernel(const double* __restrict__ R, long long ldr, const double* __restrict__ w,
                                                            int M_old, int nb, double* __restrict__ z, const double* __restrict__ skip) {
    if (skip && *skip != 0.0) return;
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M_old) return;
    double a = 0.0;
    for (int u = 0; u < nb; ++u) a = fma(R[(long long)u * ldr + v], w[u], a);
    z[v] -= a;
}
// L[M_old + u][v] = s_new[u] R[u][v] for v < b0: the appended rows of the grown factor left of the last diagonal block
__global__ void __launch_bounds__(256) border_write_rows_kernel(const double* __restrict__ R, long long ldr, const double* __restrict__ s_new,
                                                                int M_old, int nb, int b0, double* __restrict__ L, long long ldl) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x, u = blockIdx.y;
    if (v < b0) L[(long long)(M_old + u) * ldl + v] = s_new[u] * R[(long long)u * ldr + v];
}

// ---- chord steps in difference space ------------------------------------------------------------------------------------
// The likelihood only sees the differences d = B'f (d_qj = f_j - f_winner), and alpha stays in the range of B (alpha = B gamma:
// beta is, and every step keeps it there), so the iteration can be carried by the M-vectors (gamma, d = G gamma):
//     c = a0+ d + g(d)            g_qj = -phi~(d_qj / sigma) / (sigma m)      (beta = B g)
//     (I + s G s) y = s G c       the same factor / border solve as before
//     gamma_new = c - s y         d_new = G gamma_new = y / s   on every entry with s > 0
// (from s G s y = s G c - y).  One mat-vec with G (M x M) per step instead of two with Sigma (N x N); the entries whose coefficient
// is (nearly) zero -- observations above their winner, 130 of 5000 at the mode of the bench problem, and appended rows before
// their first step -- take their row of G gamma_new directly.  T = -1/2 gamma.d - lik(d)/m, so the acceptance test, the Aitken
// step lengths and the Anderson mixing (which preserves d = G gamma like it preserved f = Sigma alpha) run on (gamma, d) with
// the kernels of the alpha-space iteration.  alpha = B gamma and f = Sigma alpha are restored once per batch.
__global__ void to_diff_kernel(const double* __restrict__ f, const double* __restrict__ alpha, int Q, int m,
                               double* __restrict__ d, double* __restrict__ gamma) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= Q * m) return;
    const int q = u / m, j = u % m;
    const long long w = (long long)q * (m + 1);
    d[u] = f[w + 1 + j] - f[w];
    gamma[u] = alpha[w + 1 + j];
}
// alpha = B gamma (one warp per set; skip: nothing was changed in this batch is not a case -- always runs)
__global__ void __launch_bounds__(256) from_diff_kernel(const double* __restrict__ gamma, int Q, int m, double* __restrict__ alpha) {
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= Q) return;
    const long long base = (long long)q * (m + 1);
    double s = 0.0;
    for (int j = lane; j < m; j += 32) {
        const double g = gamma[(long long)q * m + j];
        s += g;
        alpha[base + 1 + j] = g;
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) alpha[base] = -s;
}
// c[u] = ap[u] d[u] + g(d[u])
__global__ void dchord_rhs_kernel(const double* __restrict__ d, const double* __restrict__ ap, int M, double sigma, int m,
                                  double* __restrict__ c, const double* __restrict__ skip) {
    if (skip && *skip != 0.0) return;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= M) return;
    const double du = d[u];
    c[u] = fma(ap[u], du, -phi_tilde(du / sigma) / (sigma * m));
}
// coefficients of the border rows at the current iterate (their own Newton step inside every chord step)
__global__ void dborder_coeff_kernel(const double* __restrict__ d, int nb, double sigma, int m, double* __restrict__ sa,
                                     double* __restrict__ ap, const double* __restrict__ skip) {
    if (skip && *skip != 0.0) return;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nb) return;
    const double dl = d[u] / sigma;
    const double a = -(0.5 / (m * sigma * sigma)) * dl * phi_tilde(dl);
    const double a_pos = a > 0.0 ? a : 0.0;
    ap[u] = a_pos;
    sa[u] = sqrt(a_pos);
}
// t[u] *= sa[u]    (t holds G c on entry)
__global__ void dchord_scale_kernel(double* __restrict__ t, const double* __restrict__ sa, int M, const double* __restrict__ skip) {
    if (skip && *skip != 0.0) return;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < M) t[u] *= sa[u];
}
// dgamma = (c - sa y) - gamma;  dd = y / sa - d where ap >= thr (the other rows: dchord_rows_kernel)
__global__ void dchord_update_kernel(const double* __restrict__ c, const double* __restrict__ sa, const double* __restrict__ ap,
                                     const double* __restrict__ y, const double* __restrict__ gamma, const double* __restrict__ d,
                                     int M, double thr, double* __restrict__ dgamma, double* __restrict__ dd,
                                     const double* __restrict__ skip) {
    if (skip && *skip != 0.0) return;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= M) return;
    const double s = sa[u], yu = y[u];
    dgamma[u] = fma(-s, yu, c[u]) - gamma[u];
    if (ap[u] >= thr) dd[u] = yu / s - d[u];
}
// rows whose coefficient is below thr: dd[u] = G[u, :] . (gamma + dgamma) - d[u].  One CTA per row, the others leave at once (with
// one WARP per row the ~150 working warps each stream their 40 KB row alone: 43 us, latency-bound; 256 threads per row: 8 us)
__global__ void __launch_bounds__(256) dchord_rows_kernel(const double* __restrict__ G, long long ldg, const double* __restrict__ gamma,
                                                          const double* __restrict__ dgamma, const double* __restrict__ ap,
                                                          const double* __restrict__ d, int M, double thr, double* __restrict__ dd,
                                                          const double* __restrict__ skip) {
    __shared__ double red[33];
    if (skip && *skip != 0.0) return;
    const int u = blockIdx.x;
    if (ap[u] >= thr) return;                              // uniform per CTA
    const double* g = G + (long long)u * ldg;
    double s0 = 0.0, s1 = 0.0;
    int k = threadIdx.x;
    for (; k + 256 < M; k += 512) {
        s0 = fma(g[k], gamma[k] + dgamma[k], s0);
        s1 = fma(g[k + 256], gamma[k + 256] + dgamma[k + 256], s1);
    }
    if (k < M) s0 = fma(g[k], gamma[k] + dgamma[k], s0);
    const double s = block_sum(s0 + s1, red);
    if (threadIdx.x == 0) dd[u] = s - d[u];
}
// likelihood sums of a queued step at its step length omega = state[7] and (part0) at the current iterate, from the differences
__global__ void __launch_bounds__(256) dchord_lik_kernel(const double* __restrict__ d, const double* __restrict__ dd, int Q, int m,
                                                         double sigma, const double* __restrict__ state, double* __restrict__ part,
                                                         double* __restrict__ part0) {
    if (state[4] != 0.0) return;
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= Q) return;
    const double step = state[7], inv_s = 1.0 / sigma;
    double s = 0.0, s0 = 0.0;
    for (int j = lane; j < m; j += 32) {
        const double du = d[(long long)q * m + j];
        s += Phi_tilde(fma(step, dd[(long long)q * m + j], du) * inv_s);
        if (part0) s0 += Phi_tilde(du * inv_s);
    }
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    }
    if (lane == 0) {
        part[q] = s;
        if (part0) part0[q] = s0;
    }
}

bool thread_is_background();        // linalg.cu
static int launch_chord_anderson(double* alpha, double* f, const double* df, int N, const double* state, double* aa, double* H,
                                 cudaStream_t st) {
    if (thread_is_background()) {               // three ordinary launches (see chord_anderson_kernel)
        PPBO_CL chord_anderson_sums_kernel<<<AA_CL, 1024, 0, st>>>(alpha, f, df, N, state, aa, H);
        PPBO_CL chord_anderson_solve_kernel<<<1, 32, 0, st>>>(state, aa);
        PPBO_CL chord_anderson_apply_kernel<<<AA_CL, 1024, 0, st>>>(alpha, f, N, aa, H);
        PPBO_LAUNCH_CHECK();
        return PPBO_OK;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(AA_CL);
    cfg.blockDim = dim3(1024);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = AA_CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    ++g_launch_count;
    PPBO_CUDA_CHECK(cudaLaunchKernelEx(&cfg, chord_anderson_kernel, alpha, f, df, N, state, aa, H));
    return PPBO_OK;
}

int launch_lik_terms(const double* f, int Q, int m, double sigma, double* set_lik, double* beta, double* arrow, double* sa,
                     double* bvec, cudaStream_t st) {
    PPBO_CL lik_terms_kernel<<<ceil_div(Q, 8), 256, 0, st>>>(f, Q, m, sigma, set_lik, beta, arrow, sa, bvec);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}
int launch_linesearch_lik(const double* f, const double* df, int Q, int m, double sigma, double* part, cudaStream_t st) {
    PPBO_CL linesearch_lik_kernel<<<dim3(ceil_div(Q, 8), NSTEP), 256, 0, st>>>(f, df, Q, m, sigma, part);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}
int launch_sum(const double* x, int n, double* out, cudaStream_t st) {
    PPBO_CL sum_kernel<<<1, 1024, 0, st>>>(x, n, out);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

constexpr int CHORD_STATE = 16, CHORD_BATCH_MAX = 16;

// sa[u] = sqrt(max(arrow[u], 0))
__global__ void sqrt_clamp_kernel(const double* __restrict__ arrow, int M, double* __restrict__ sa) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < M) sa[u] = sqrt(fmax(arrow[u], 0.0));
}
// ap[u] = sa[u]^2 (the clamped coefficients a factor was built with)
__global__ void square_kernel(const double* __restrict__ sa, int M, double* __restrict__ ap) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < M) ap[u] = sa[u] * sa[u];
}
// scal[4] = max|f_new - f_old|, scal[5] = max|f_new|  (relative size of the first step from a warm start; single CTA)
__global__ void __launch_bounds__(1024) warm_step_size_kernel(const double* __restrict__ f_old, const double* __restrict__ f_new,
                                                              int N, double* __restrict__ scal) {
    __shared__ double mx[2][32];
    double md = 0.0, mf = 0.0;
    for (int i = threadIdx.x; i < N; i += 1024) {
        md = fmax(md, fabs(f_new[i] - f_old[i]));
        mf = fmax(mf, fabs(f_new[i]));
    }
    for (int o = 16; o > 0; o >>= 1) {
        md = fmax(md, __shfl_xor_sync(0xffffffffu, md, o));
        mf = fmax(mf, __shfl_xor_sync(0xffffffffu, mf, o));
    }
    if ((threadIdx.x & 31) == 0) { mx[0][threadIdx.x >> 5] = md; mx[1][threadIdx.x >> 5] = mf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 32; ++w) { md = fmax(md, mx[0][w]); mf = fmax(mf, mx[1][w]); }
        scal[4] = md;
        scal[5] = mf;
    }
}
// rows [r_lo, r_hi) of the Newton matrix I + sa G sa, columns [c_lo(row), row]: c_lo = c_old for rows < r_split (rows whose
// leading columns already hold factor entries that must survive), 0 for the appended rows
__global__ void __launch_bounds__(256) newton_rows_kernel(const double* __restrict__ G, long long ldg, const double* __restrict__ sa,
                                                          int r_lo, int r_hi, int r_split, int c_old, double* __restrict__ out,
                                                          long long ldo) {
    const int u = r_lo + blockIdx.y, v = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= r_hi || v > u) return;
    if (u < r_split && v < c_old) return;
    double x = sa[u] * G[(long long)u * ldg + v] * sa[v];
    if (u == v) x += 1.0;
    out[(long long)u * ldo + v] = x;
}

struct FitWorkspace {
    double *bvec, *sa, *ap, *t, *Sb, *dalpha, *df, *set_part, *scal, *arrow_tmp, *binv, *state, *hist;
    double *bR, *bT, *bC, *bw;           // bordered warm start: R [BORDER_MAX x M], scratch T [BORDER_MAX x M], C [BORDER_MAX^2], w
    double *aaH, *aa, *part0;            // Anderson history [(3 AA_M + 3) x N], its state [8], likelihood sums at the current iterate [Q]
    double* sym;                         // partials of the symmetric mat-vecs with Sigma (N) and G (M < N): symv_scratch_doubles(N)
    int* info;
    static long long doubles(int Q, int m) {
        const long long N = (long long)Q * (m + 1), M = (long long)Q * m;
        return 4 * N + 3 * M + (M + CHOL_NB) + (long long)NSTEP * Q + 32 + 8 + 64 + CHORD_STATE + 2 * CHORD_BATCH_MAX +
               blockinv_doubles((int)M) + 2LL * BORDER_MAX * (M + 2) + (long long)BORDER_MAX * BORDER_MAX + BORDER_MAX + 8 +
               (3LL * AA_M + 3) * N + AA_STATE + Q + symv_scratch_doubles((int)N);
    }
    void carve(double* base, int Q, int m) {
        const long long N = (long long)Q * (m + 1), M = (long long)Q * m;
        double* p = base;
        bvec = p; p += N;
        Sb = p; p += N;
        dalpha = p; p += N;
        df = p; p += N;
        sa = p; p += M;
        ap = p; p += M;
        arrow_tmp = p; p += M;
        t = p; p += M + CHOL_NB;
        set_part = p; p += (long long)NSTEP * Q;
        scal = p; p += 32;
        info = reinterpret_cast<int*>(p); p += 8;
        state = p; p += CHORD_STATE;
        hist = p; p += 2 * CHORD_BATCH_MAX;
        binv = p; p += blockinv_doubles((int)M);
        if ((reinterpret_cast<uintptr_t>(p) & 15) != 0) ++p;           // 16-byte alignment for the GEMM operands
        const long long Mp = (M + 1) / 2 * 2;
        bR = p; p += BORDER_MAX * Mp;
        bT = p; p += BORDER_MAX * Mp;
        bC = p; p += (long long)BORDER_MAX * BORDER_MAX;
        bw = p; p += BORDER_MAX;
        aaH = p; p += (3LL * AA_M + 3) * N;
        aa = p; p += AA_STATE;
        part0 = p; p += Q;
        sym = p;
    }
};

}  // namespace ppbo

using namespace ppbo;

extern "C" int ppbo_lik_terms(const double* f, int Q, int m, double sigma, double* lik_sum, double* beta,
                              double* arrow, void* stream) {
    PPBO_REQUIRE(Q >= 0 && m >= 1 && sigma > 0, "shape / sigma");
    if (Q == 0) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    double* part = nullptr;
    if (lik_sum) PPBO_CUDA_CHECK(malloc_async((void**)&part, sizeof(double) * Q, st));
    PPBO_CL lik_terms_kernel<<<ceil_div(Q, 8), 256, 0, st>>>(f, Q, m, sigma, part, beta, arrow, nullptr, nullptr);
    PPBO_LAUNCH_CHECK();
    if (lik_sum) {
        PPBO_CL sum_kernel<<<1, 1024, 0, st>>>(part, Q, lik_sum);
        PPBO_LAUNCH_CHECK();
        PPBO_CUDA_CHECK(cudaFreeAsync(part, st));
    }
    return PPBO_OK;
}

/* set_sums[q] = sum_j Phi(Delta_qj / sqrt 2): GPModel.sum_Phi_vec(0, ...) for all comparison sets in one launch (src/gp_model.py:206-218) */
extern "C" int ppbo_lik_set_sums(const double* f, int Q, int m, double sigma, double* set_sums, void* stream) {
    PPBO_REQUIRE(Q >= 0 && m >= 1 && sigma > 0 && set_sums != nullptr, "shape / sigma");
    if (Q == 0) return PPBO_OK;
    PPBO_CL lik_terms_kernel<<<ceil_div(Q, 8), 256, 0, (cudaStream_t)stream>>>(f, Q, m, sigma, set_sums, nullptr, nullptr, nullptr, nullptr);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_lambda_dense(const double* arrow, int Q, int m, double* out, long long ld, void* stream) {
    const long long N = (long long)Q * (m + 1);
    if (N == 0) return PPBO_OK;
    PPBO_CL lambda_dense_kernel<<<(unsigned)ceil_div_ll(N * N, 256), 256, 0, (cudaStream_t)stream>>>(arrow, Q, m, out, ld);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_evidence_matrix(const double* Sigma, long long lds, int Q, int m, const double* arrow, int reference_sign,
                                    double* out, long long ldo, void* stream) {
    PPBO_REQUIRE(Q >= 1 && m >= 1 && ldo >= (long long)Q * (m + 1), "shape");
    PPBO_REQUIRE((long long)Q * (m + 1) <= 65535, "Q (m+1) above 65535 (one grid row per row of the output)");
    const int N = Q * (m + 1);
    PPBO_CL evidence_matrix_kernel<<<dim3(ceil_div(N, 256), N), 256, 0, (cudaStream_t)stream>>>(Sigma, lds, Q, m, arrow,
                                                                                                reference_sign ? -1.0 : 1.0, out, ldo);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" long long ppbo_laplace_workspace_bytes(int Q, int m) { return FitWorkspace::doubles(Q, m) * 8; }

namespace ppbo {
int diffspace_gram_append(const double* S, long long lds, int Q_old, int Q_new, int m, double* G, long long ldg, cudaStream_t st);
}

extern "C" int ppbo_diffspace_gram_append(const double* Sigma, long long lds, int Q_old, int Q_new, int m, double* G,
                                          long long ldg, void* stream) {
    PPBO_REQUIRE(Q_old >= 0 && Q_new >= Q_old && m >= 1 && ldg >= (long long)Q_new * m, "shape");
    return diffspace_gram_append(Sigma, lds, Q_old, Q_new, m, G, ldg, (cudaStream_t)stream);
}

/* Factor at the mode on demand (ppbo_laplace_fit without PPBO_FIT_FACTOR_AT_MODE leaves the last Newton factor behind):
 * sa_fac = sqrt(max(arrow, 0)), Lfac = chol(I + sa_fac G sa_fac).  Returns 0 / pivot index (host sync). */
extern "C" int ppbo_laplace_refactor(const double* G, long long ldg, int M, const double* arrow, double* Lfac, int cap,
                                     double* sa_fac, void* stream) {
    PPBO_REQUIRE(M >= 1 && cap >= M && ldg >= M, "shape");
    cudaStream_t st = (cudaStream_t)stream;
    double* dinv = Lfac + (long long)cap * cap;
    int* info_d = nullptr;
    PPBO_CUDA_CHECK(malloc_async((void**)&info_d, sizeof(int), st));
    PPBO_CL sqrt_clamp_kernel<<<ceil_div(M, 256), 256, 0, st>>>(arrow, M, sa_fac);
    int rc;
    if ((rc = newton_matrix(G, ldg, M, sa_fac, Lfac, cap, st))) return rc;
    if ((rc = potrf_lower(Lfac, cap, M, dinv, info_d, st))) return rc;
    int info = 0;
    PPBO_CUDA_CHECK(readback().add(&info, info_d, sizeof(int), st));
    PPBO_CUDA_CHECK(cudaFreeAsync(info_d, st));
    PPBO_CUDA_CHECK(readback().finish(st));
    if (info) set_error("mode system not positive definite at pivot %d", info);
    return info;
}

/* Grow a factor by the rows of appended comparison sets.  On entry Lfac holds chol(I + sa G sa) of size M_old for the first
 * M_old entries of sa_fac; sa_fac[M_old .. M_new) hold the coefficients chosen for the new rows (ppbo_lik_terms at the warm
 * start).  On return Lfac is the factor of the M_new system with those coefficients: the block rows from the last 128-boundary
 * b0 <= M_old on are recomputed (new rows: L21 = A21 L11^-T by a 25-row triangular solve; Schur complement of the <= 2 trailing
 * diagonal blocks; their Cholesky) -- O(M^2 m) instead of O(M^3 / 3).  (src/feedback_processing.py:133-154 appends one (m+1)-row
 * block per iteration; SURVEY.md 8f rank 2.) */
extern "C" int ppbo_factor_extend(const double* G, long long ldg, int M_old, int M_new, double* sa_fac, const double* f_new_sets,
                                  int m, double sigma, double* Lfac, int cap, void* stream) {
    PPBO_REQUIRE(M_old >= 0 && M_new >= M_old && cap >= M_new && ldg >= M_new, "shape");
    if (M_new == M_old) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (f_new_sets) {      // coefficients of the appended sets at the warm start: sa = sqrt(max(a(f), 0))
        PPBO_REQUIRE(m >= 1 && sigma > 0 && (M_new - M_old) % m == 0, "appended rows must be whole comparison sets");
        const int Qn = (M_new - M_old) / m;
        PPBO_CL lik_terms_kernel<<<ceil_div(Qn, 8), 256, 0, st>>>(f_new_sets, Qn, m, sigma, nullptr, nullptr, nullptr, sa_fac + M_old, nullptr);
        PPBO_LAUNCH_CHECK();
    }
    double* dinv = Lfac + (long long)cap * cap;
    const int b0 = (M_old / CHOL_NB) * CHOL_NB, nt = M_new - b0;
    int rc;
    int* info_d = nullptr;
    PPBO_CUDA_CHECK(malloc_async((void**)&info_d, sizeof(int), st));
    PPBO_CL newton_rows_kernel<<<dim3(ceil_div(M_new, 256), nt), 256, 0, st>>>(G, ldg, sa_fac, b0, M_new, M_old, b0, Lfac, cap);
    PPBO_LAUNCH_CHECK();
    if (b0 > 0) {
        double* Lnew = Lfac + (long long)M_old * cap;          // appended rows, columns [0, b0): A21 -> A21 L11^-T
        if ((rc = trsm_right_lower_t(Lfac, cap, b0, dinv, Lnew, cap, M_new - M_old, st))) return rc;
        double* Lt = Lfac + (long long)b0 * cap;               // rows [b0, M_new): S = A[b0:, b0:] - L[b0:, :b0] L[b0:, :b0]^T
        GemmOperands g{Lt, cap, 0, Lt, cap, 0, nt, nt, b0};
        StoreEpilogue ep{Lt + b0, cap, 0, -1.0, 1.0, 1, 0};
        if ((rc = launch_gemm_nt(g, ep, 1, st))) return rc;
    }
    if ((rc = potrf_lower(Lfac + (long long)b0 * cap + b0, cap, nt, dinv + (long long)(b0 / CHOL_NB) * CHOL_NB * CHOL_NB, info_d, st)))
        return rc;
    int info = 0;
    PPBO_CUDA_CHECK(readback().add(&info, info_d, sizeof(int), st));
    PPBO_CUDA_CHECK(cudaFreeAsync(info_d, st));
    PPBO_CUDA_CHECK(readback().finish(st));
    if (info) { info += b0; set_error("extended factor not positive definite at pivot %d", info); }
    return info;
}

extern "C" int ppbo_laplace_fit(const double* Sigma, long long lds, int Q, int m, double sigma, const double* f_init,
                                const double* alpha_init, int max_iter, double tol, int flags, double* G, long long ldg,
                                double* Lfac, int cap, double* sa_fac, int warm_rows, double* binv_cache, int* binv_state_h,
                                double* f_map, double* alpha, double* arrow, void* workspace, long long workspace_bytes,
                                double* stats_h, void* stream) {
    PPBO_REQUIRE(Q >= 1 && m >= 1 && sigma > 0, "shape / sigma");
    PPBO_REQUIRE(workspace_bytes >= ppbo_laplace_workspace_bytes(Q, m), "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int N = Q * (m + 1), M = Q * m;
    PPBO_REQUIRE(cap >= M && ldg >= M, "capacity / leading dimension below Q m");
    const bool g_ready = (flags & PPBO_FIT_G_READY) != 0, warm_factor = (flags & PPBO_FIT_FACTOR_WARM) != 0;
    const bool factor_at_mode = (flags & PPBO_FIT_FACTOR_AT_MODE) != 0;
    PPBO_REQUIRE(!warm_factor || (f_init != nullptr && alpha_init != nullptr && sa_fac != nullptr),
                 "a warm factor needs f_init, alpha_init = Sigma^-1 f_init and sa_fac");
    PPBO_REQUIRE(!warm_factor || (warm_rows >= 1 && warm_rows <= M), "warm_rows: size of the system the warm factor belongs to");
    PPBO_REQUIRE(alpha_init == nullptr || f_init != nullptr, "alpha_init without f_init");
    FitWorkspace ws;
    ws.carve((double*)workspace, Q, m);
    // block inverses of the factor: in the caller's persistent buffer when given (a factor that only grows at its end keeps its
    // leading 1024-blocks: binv_state_h = {leading rows unchanged since the build, ceil(rows / 1024) of that build})
    if (binv_cache) ws.binv = binv_cache;
    const long long ldl = cap;
    double* Mdinv = Lfac + (long long)cap * cap;  // factor object = [cap x cap lower factor | inverted diagonal blocks]
    int rc;
    if (!g_ready && (rc = diffspace_gram(Sigma, lds, Q, m, G, ldg, st))) return rc;

    const bool have_start = f_init != nullptr;
    if (have_start) PPBO_CUDA_CHECK(cudaMemcpyAsync(f_map, f_init, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
    else PPBO_CUDA_CHECK(cudaMemsetAsync(f_map, 0, sizeof(double) * N, st));
    if (alpha_init) PPBO_CUDA_CHECK(cudaMemcpyAsync(alpha, alpha_init, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
    else PPBO_CUDA_CHECK(cudaMemsetAsync(alpha, 0, sizeof(double) * N, st));

    const int set_blocks = ceil_div(Q, 8);
    double scal_h[32];
    int it = 0, info = 0, n_factor = 0, n_chord = 0;
    double last_step = 0.0, last_rel = INFINITY, T_cur = NAN, prev_rel_h = INFINITY;
    bool alpha_known = !have_start || alpha_init != nullptr;   // alpha = Sigma^-1 f is known for the zero start or when handed in
    int n_halvings_total = 0;
    // Newton steps refactor I + a+^1/2 G a+^1/2 at the current iterate; once the relative step is below CHORD_REL the factor
    // is kept and only the right-hand side is refreshed (chord steps: same fixed point Sigma^-1 f = beta(f), linear
    // convergence at the rate of the relative change of a+; a chord step costs ~1/6 of a factorisation at Qm = 5000, so it
    // is kept as long as it at least halves the step).
    constexpr double CHORD_REL = 0.25;
    const bool trace = getenv("PPBO_TRACE") != nullptr;
    bool refactor = true, converged = false;
    // Cold start f = 0: every difference is 0, so a = -Delta phi~(Delta) / (2 m sigma^2) = 0 and the Newton matrix
    // I + a+^1/2 G a+^1/2 is the identity: its factor is known, nothing to factorise and nothing to solve.
    bool identity_factor = false;
    // chord steps reuse one factor many times: its diagonal blocks are inverted at the first chord step (linalg.cu, block-inverse
    // solves), which makes every later solve with that factor ~3x cheaper than the 40-link chained solve
    bool binv_valid = false;
    bool first_chord_batch = true;
    double chord_omega = 1.0, chord_ratio = 0.0, chord_wait = 0.0;
    // Anderson acceleration of the chord iteration: a fit that starts without a usable factor enters the chord phase after its
    // FIRST factorisation (relative step <= 0.6 instead of 0.25) and mixes the chord steps there; if three mixed steps do not halve
    // the residual the fit pays for the second factorisation and continues exactly like the unaccelerated iteration.  Warm
    // (bordered) fits are not mixed: the border's Newton steps change the map from step to step and the Aitken step lengths do
    // better there (measured).
    bool aa_failed = false;
    double rel3_h = INFINITY;
    auto aa_now = [&]() { return !warm_factor && n_factor == 1 && !aa_failed; };
    PPBO_CUDA_CHECK(cudaMemsetAsync(ws.aa, 0, sizeof(double) * 8, st));
    bool factor_current = false;         // Lfac is the factor for the coefficients in ws.sa / ws.ap
    double warm_first_rel = NAN;
    // ---- warm start with the previous iteration's factor (bordered, see border_solve_kernel): chord steps from (f_init, alpha_init)
    int M_old = M, nb = 0;               // bordered: the factor in Lfac covers the first M_old rows, the last nb are the border
    bool bordered = false;
    if (warm_factor && M - warm_rows <= BORDER_MAX && (M - warm_rows) % m == 0) {
        M_old = warm_rows;
        nb = M - M_old;
        bordered = nb > 0;
        PPBO_CUDA_CHECK(cudaMemcpyAsync(ws.sa, sa_fac, sizeof(double) * M_old, cudaMemcpyDeviceToDevice, st));
        PPBO_CL square_kernel<<<ceil_div(M_old, 256), 256, 0, st>>>(ws.sa, M_old, ws.ap);
        int first_block = 0;
        if (binv_cache && binv_state_h && binv_state_h[1] == ceil_div(M_old, 1024)) first_block = std::min(binv_state_h[0], M_old) / 1024;
        if ((rc = blockinv_build(Lfac, ldl, M_old, Mdinv, ws.binv, st, first_block))) return rc;
        binv_valid = true;
        if (bordered) {
            const long long Mp = (M + 1) / 2 * 2;
            PPBO_CL border_rows_kernel<<<dim3(ceil_div(M_old, 256), nb), 256, 0, st>>>(G, ldg, ws.sa, M_old, nb, ws.bT, Mp);
            PPBO_CL border_corner_kernel<<<ceil_div(nb * nb, 256), 256, 0, st>>>(G, ldg, M_old, nb, ws.bC);
            PPBO_LAUNCH_CHECK();
            if ((rc = trsm_right_blockinv(Lfac, ldl, M_old, ws.binv, ws.bT, Mp, ws.bR, Mp, nb, st))) return rc;
            // C = G_nn - R R' (25 x 25, K = M_old): as ONE product the tiled GEMM walks all of K on a single CTA (270 us at
            // K = 5000); cut into 1024-column chunks it is a batched product of the same launch count whose partial results
            // (in the scratch T, which the solve above has consumed) are added in chunk order by border_corner_sum_kernel.
            // (One-warp-per-output-column kernels for these 25-row products, with and without a shared-memory stage for R, were
            // measured and were no faster than the tiled GEMM: 45-110 us / 120-470 us per call against 55-60 us.)
            const int KC = 1024, nfull = M_old / KC, krem = M_old - nfull * KC, nparts = nfull + (krem > 0 ? 1 : 0);
            if (nfull > 0) {
                GemmOperands g{ws.bR, Mp, KC, ws.bR, Mp, KC, nb, nb, KC};
                StoreEpilogue ep{ws.bT, nb, (long long)nb * nb, 1.0, 0.0, 0, 0, 0};
                if ((rc = launch_gemm_nt(g, ep, nfull, st))) return rc;
            }
            if (krem > 0) {
                GemmOperands g{ws.bR + (long long)nfull * KC, Mp, 0, ws.bR + (long long)nfull * KC, Mp, 0, nb, nb, krem};
                StoreEpilogue ep{ws.bT + (long long)nfull * nb * nb, nb, 0, 1.0, 0.0, 0, 0, 0};
                if ((rc = launch_gemm_nt(g, ep, 1, st))) return rc;
            }
            PPBO_CL border_corner_sum_kernel<<<ceil_div(nb * nb, 256), 256, 0, st>>>(ws.bT, nparts, nb, ws.bC);
            PPBO_LAUNCH_CHECK();
        }
        // T at the start (the chord acceptance test compares against it): -1/2 alpha.f - lik(f)/m
        PPBO_CL lik_terms_kernel<<<set_blocks, 256, 0, st>>>(f_map, Q, m, sigma, ws.arrow_tmp, nullptr, nullptr, nullptr, nullptr);
        PPBO_CL sum_kernel<<<1, 1024, 0, st>>>(ws.arrow_tmp, Q, ws.scal + 24);
        PPBO_CL dot_kernel<<<1, 1024, 0, st>>>(alpha, f_map, N, ws.scal);
        PPBO_LAUNCH_CHECK();
        PPBO_CUDA_CHECK(readback().add(scal_h, ws.scal, sizeof(double) * 32, st));
        PPBO_CUDA_CHECK(readback().finish(st));
        T_cur = -0.5 * scal_h[0] - scal_h[24] / m;
        last_rel = INFINITY;                 // unknown yet: the first batch (3 steps) measures the contraction
        factor_current = !bordered;          // a bordered factor is not a factor object of the whole system (finalised below)
        refactor = false;
        if (trace) fprintf(stderr, "[ppbo_laplace_fit] warm start: factor of %d rows, border %d, T %.12g\n", M_old, nb, T_cur);
    }
    // (I + s G s) y = t in place with the factor in Lfac (+ border)
    auto chord_solve = [&](const double* skip) -> int {
        int r_;
        if (!bordered) return potrs_vec_blockinv(Lfac, ldl, M, ws.binv, ws.t, st, skip);
        const long long Mp = (M + 1) / 2 * 2;
        double* z = blockinv_y(ws.binv, M_old);
        if ((r_ = potrs_fwd_blockinv(Lfac, ldl, M_old, ws.binv, ws.t, st, skip))) return r_;
        PPBO_CL border_solve_kernel<<<1, 1024, 0, st>>>(ws.bR, Mp, ws.bC, ws.sa + M_old, z, M_old, nb, ws.t + M_old, ws.bw, skip);
        PPBO_CL border_update_kernel<<<ceil_div(M_old, 256), 256, 0, st>>>(ws.bR, Mp, ws.bw, M_old, nb, z, skip);
        return potrs_bwd_blockinv(Lfac, ldl, M_old, ws.binv, ws.t, st, skip);
    };
    // chord batches in difference space keep (gamma, d) between batches; (alpha, f) are restored when the fit leaves the chord phase
    bool in_diff = false;
    auto leave_diff = [&]() -> int {
        if (!in_diff) return PPBO_OK;
        in_diff = false;
        PPBO_CL from_diff_kernel<<<set_blocks, 256, 0, st>>>(ws.bvec, Q, m, alpha);          // alpha = B gamma
        return symv_lower(Sigma, lds, N, alpha, f_map, ws.sym, st);                            // f = Sigma alpha
    };
    while (it < max_iter && !converged) {
        if (!refactor) {
            // ---- a batch of chord steps: the factor is kept, only the right-hand side is refreshed; acceptance, the convergence
            // test and the contraction test run on the device (chord_decide_kernel), one host synchronise per batch.  The batch
            // length is the number of steps the observed contraction rate predicts (the first batch is short: it measures the rate).
            if (!binv_valid) {
                if ((rc = blockinv_build(Lfac, ldl, M, Mdinv, ws.binv, st))) return rc;
                binv_valid = true;
            }
            double rho = (std::isfinite(prev_rel_h) && last_rel < prev_rel_h) ? last_rel / prev_rel_h : 0.2;
            const bool anderson = aa_now();
            rho = std::fmin(std::fmax(rho, 0.02), (anderson || (warm_factor && n_factor == 0)) ? 0.85 : 0.5);
            int kb = !std::isfinite(last_rel) ? 3 : (last_rel > tol) ? (int)std::ceil(std::log(tol / last_rel) / std::log(rho)) : 1;
            if (first_chord_batch) kb = std::min(kb, 3);
            // warm (bordered) fits converge faster than their contraction predicts once an Aitken step lands; every queued step
            // behind the converging one still costs ~26 no-op launches (0.15 ms), a batch boundary one synchronise (0.03 ms)
            if (warm_factor && n_factor == 0) kb = std::min(kb, 4);
            kb = std::max(1, std::min(kb, std::min(CHORD_BATCH_MAX, max_iter - it)));
            first_chord_batch = false;
            const double slow = (warm_factor && n_factor == 0) ? 0.85 : 0.5;
            double state_h[CHORD_STATE] = {T_cur, last_rel, prev_rel_h, last_step, 0.0, 0.0, tol, chord_omega, chord_ratio, chord_wait, slow,
                                           rel3_h, 0.0, anderson ? 1.0 : 0.0};
            double hist_h[2 * CHORD_BATCH_MAX];
            PPBO_CUDA_CHECK(cudaMemcpyAsync(ws.state, state_h, sizeof(state_h), cudaMemcpyHostToDevice, st));
            const double* skip = ws.state + 4;               // non-zero once a step of the batch has stopped it
            // ---- the batch in difference space (see to_diff_kernel): gamma, d, c, dgamma, dd live in the N-vectors of the
            // alpha-space Newton step, which are idle here
            double *gam = ws.bvec, *dv = ws.Sb, *cv = ws.dalpha, *dgam = ws.df, *ddv = ws.arrow_tmp;
            const double thr = 1e-3 * 0.121 / (m * sigma * sigma);       // 1e-3 of the largest possible coefficient
            if (!in_diff) {              // (consecutive batches stay in difference space: nothing else touches these vectors)
                PPBO_CL to_diff_kernel<<<ceil_div(M, 256), 256, 0, st>>>(f_map, alpha, Q, m, dv, gam);
                in_diff = true;
            }
            for (int i = 0; i < kb; ++i) {
                if (bordered)
                    PPBO_CL dborder_coeff_kernel<<<ceil_div(nb, 64), 64, 0, st>>>(dv + M_old, nb, sigma, m, ws.sa + M_old, ws.ap + M_old, skip);
                PPBO_CL dchord_rhs_kernel<<<ceil_div(M, 256), 256, 0, st>>>(dv, ws.ap, M, sigma, m, cv, skip);
                if ((rc = symv_lower(G, ldg, M, cv, ws.t, ws.sym, st, skip))) return rc;
                PPBO_CL dchord_scale_kernel<<<ceil_div(M, 256), 256, 0, st>>>(ws.t, ws.sa, M, skip);
                if ((rc = chord_solve(skip))) return rc;
                PPBO_CL dchord_update_kernel<<<ceil_div(M, 256), 256, 0, st>>>(cv, ws.sa, ws.ap, ws.t, gam, dv, M, thr, dgam, ddv, skip);
                PPBO_CL dchord_rows_kernel<<<M, 256, 0, st>>>(G, ldg, gam, dgam, ws.ap, dv, M, thr, ddv, skip);
                PPBO_CL dchord_lik_kernel<<<set_blocks, 256, 0, st>>>(dv, ddv, Q, m, sigma, ws.state, ws.set_part, anderson ? ws.part0 : nullptr);
                PPBO_CL chord_decide_kernel<<<1, 1024, 0, st>>>(gam, dgam, dv, ddv, M, ws.set_part, Q, m, ws.state, ws.hist,
                                                                  !anderson, anderson ? ws.part0 : nullptr);
                if (anderson && (rc = launch_chord_anderson(gam, dv, ddv, M, ws.state, ws.aa, ws.aaH, st))) return rc;
            }
            PPBO_LAUNCH_CHECK();
            PPBO_CUDA_CHECK(readback().add(state_h, ws.state, sizeof(state_h), st));
            PPBO_CUDA_CHECK(readback().add(hist_h, ws.hist, sizeof(double) * 2 * kb, st));
            PPBO_CUDA_CHECK(readback().finish(st));
            const int taken = (int)state_h[5], stop = (int)state_h[4];
            if (trace)
                for (int i = 0; i < taken; ++i)
                    fprintf(stderr, "[ppbo_laplace_fit] it %d chord  step 1 rel %.3e T %.12g (batch of %d)\n", it + i, hist_h[2 * i], hist_h[2 * i + 1], kb);
            it += taken;
            n_chord += taken;
            if (warm_factor && std::isnan(warm_first_rel) && taken > 0) warm_first_rel = hist_h[0];
            if (taken > 0) {
                T_cur = state_h[0];
                last_rel = state_h[1];
                prev_rel_h = state_h[2];
                last_step = state_h[3];
            }
            chord_omega = state_h[7];
            chord_ratio = state_h[8];
            chord_wait = state_h[9];
            rel3_h = state_h[11];
            if (anderson && (stop == 2 || stop == 3)) aa_failed = true;      // mixing did not pay: the rest of the fit runs unaccelerated
            if (stop == 1) { converged = true; break; }
            if (stop == 2 || stop == 3) refactor = true;      // contraction too slow / step rejected: pay for a new factor
            continue;
        }
        // ---- Newton step: refactor I + a+^1/2 G a+^1/2 at the current iterate
        if ((rc = leave_diff())) return rc;
        PPBO_CL lik_terms_kernel<<<set_blocks, 256, 0, st>>>(f_map, Q, m, sigma, nullptr, nullptr, nullptr, ws.sa, ws.bvec, nullptr, ws.ap);
        identity_factor = (it == 0 && !have_start);
        if (identity_factor) {
            PPBO_CUDA_CHECK(cudaMemsetAsync(ws.info, 0, sizeof(int), st));
        } else {
            if ((rc = newton_matrix(G, ldg, M, ws.sa, Lfac, ldl, st))) return rc;
            if ((rc = potrf_lower(Lfac, ldl, M, Mdinv, ws.info, st))) return rc;
            ++n_factor;
            binv_valid = false;
            factor_current = true;
            bordered = false;                    // a full factor of the grown system replaces the bordered one
            chord_omega = 1.0;                   // a new factor: new iteration matrix, forget the contraction history
            chord_ratio = 0.0;
            chord_wait = 0.0;
            PPBO_CUDA_CHECK(cudaMemsetAsync(ws.aa, 0, sizeof(double) * 8, st));
            rel3_h = INFINITY;
        }
        if ((rc = symv_lower(Sigma, lds, N, ws.bvec, ws.Sb, ws.sym, st))) return rc;
        PPBO_CL diff_scale_kernel<<<ceil_div(M, 256), 256, 0, st>>>(ws.Sb, ws.sa, Q, m, ws.t);
        if (!identity_factor) {
            // From the second factorisation on -- and for the first one of a cold fit, which enters the Anderson-mixed chord phase
            // with it -- the factor is very likely reused by chord steps, which need the 1024-block inverses anyway: build them now
            // and let this solve use them too (0.13 ms against 0.48 ms for the chained solve).
            if ((n_factor >= 2 || (!warm_factor && !aa_failed)) && M >= 2048 && !binv_valid) {
                if ((rc = blockinv_build(Lfac, ldl, M, Mdinv, ws.binv, st))) return rc;
                binv_valid = true;
            }
            rc = binv_valid ? potrs_vec_blockinv(Lfac, ldl, M, ws.binv, ws.t, st) : potrs_vec(Lfac, ldl, M, Mdinv, ws.t, st);
            if (rc) return rc;
        }
        PPBO_CL alpha_update_kernel<<<set_blocks, 256, 0, st>>>(ws.bvec, ws.sa, ws.t, alpha, Q, m, ws.dalpha);
        if ((rc = symv_lower(Sigma, lds, N, ws.dalpha, ws.df, ws.sym, st))) return rc;
        PPBO_LAUNCH_CHECK();
        if (!alpha_known) {
            // arbitrary start: alpha_old is unknown (would need Sigma^-1 f); take the full Newton step, which
            // only depends on f:  alpha <- alpha_new (= dalpha, since alpha held 0), f <- Sigma alpha_new
            PPBO_CUDA_CHECK(cudaMemcpyAsync(alpha, ws.dalpha, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
            PPBO_CUDA_CHECK(cudaMemcpyAsync(f_map, ws.df, sizeof(double) * N, cudaMemcpyDeviceToDevice, st));
            alpha_known = true;
            PPBO_CUDA_CHECK(readback().add(&info, ws.info, sizeof(int), st));
            PPBO_CUDA_CHECK(readback().finish(st));
            if (info) { set_error("Newton system not positive definite at pivot %d (iteration %d)", info, it); return info; }
            ++it;
            continue;
        }
        // line search over s = 1, 1/2, ..., 2^-7 on T(alpha + s dalpha) = -1/2 (alpha+s dalpha).(f+s df) - lik(f+s df)/m
        PPBO_CL linesearch_lik_kernel<<<dim3(set_blocks, NSTEP), 256, 0, st>>>(f_map, ws.df, Q, m, sigma, ws.set_part);
        if (std::isnan(T_cur)) {   // need T at the current point once: evaluate via the same kernel at step 0
            PPBO_CL lik_terms_kernel<<<set_blocks, 256, 0, st>>>(f_map, Q, m, sigma, ws.arrow_tmp, nullptr, nullptr, nullptr, nullptr);
            PPBO_CL sum_kernel<<<1, 1024, 0, st>>>(ws.arrow_tmp, Q, ws.scal + 24);
        }
        PPBO_CL newton_scalars_kernel<<<1, 1024, 0, st>>>(alpha, ws.dalpha, f_map, ws.df, N, ws.set_part, Q, ws.scal);
        PPBO_LAUNCH_CHECK();
        PPBO_CUDA_CHECK(readback().add(scal_h, ws.scal, sizeof(double) * 32, st));
        PPBO_CUDA_CHECK(readback().add(&info, ws.info, sizeof(int), st));
        PPBO_CUDA_CHECK(readback().finish(st));
        if (info) { set_error("Newton system not positive definite at pivot %d (iteration %d)", info, it); return info; }
        const double af = scal_h[0], adf = scal_h[1], daf = scal_h[2], dadf = scal_h[3];
        if (std::isnan(T_cur)) T_cur = -0.5 * af - scal_h[24] / m;
        double step = 0.0, T_new = T_cur;
        int c;
        for (c = 0; c < NSTEP; ++c) {
            const double s = std::ldexp(1.0, -c);
            const double Ts = -0.5 * (af + s * (adf + daf) + s * s * dadf) - scal_h[8 + c] / m;
            if (Ts >= T_cur - 1e-13 * std::fabs(T_cur)) { step = s; T_new = Ts; break; }
        }
        const double fscale = std::fmax(scal_h[5], 1e-300);
        if (c == NSTEP) { step = std::ldexp(1.0, -(NSTEP - 1)); T_new = NAN; }   // keep moving; T re-evaluated next round
        n_halvings_total += (c == NSTEP) ? NSTEP : c;
        PPBO_CL axpy2_kernel<<<ceil_div(N, 256), 256, 0, st>>>(alpha, ws.dalpha, f_map, ws.df, step, N);
        PPBO_LAUNCH_CHECK();
        T_cur = T_new;
        prev_rel_h = last_rel;
        last_step = step * scal_h[4];
        last_rel = last_step / fscale;
        if (trace) fprintf(stderr, "[ppbo_laplace_fit] it %d newton step %.3g rel %.3e T %.12g\n", it, step, last_rel, T_cur);
        ++it;
        if (step == 1.0 && last_rel <= tol) { converged = true; break; }
        // chord steps once the Newton iteration is in its contraction region and a factor exists to reuse
        const double chord_rel = (!warm_factor && n_factor == 1 && !aa_failed) ? 0.6 : CHORD_REL;
        refactor = !(step == 1.0 && last_rel <= chord_rel) || identity_factor;
    }
    if ((rc = leave_diff())) return rc;
    // The factor a later warm fit can reuse is the one the last Newton step built (or the warm one it was handed): its
    // coefficients go to sa_fac.  (An identity "factor" -- cold start that converged at once -- is not a factor object.)
    if (bordered && !factor_at_mode) {
        // grow the factor object by the border rows with their final coefficients (the next iteration's "old" factor):
        // L[new, 0:b0] = s_n R[:, 0:b0]; the block rows from the last 128-boundary on are refactored from their Schur complement
        const long long Mp = (M + 1) / 2 * 2;
        const int b0 = (M_old / CHOL_NB) * CHOL_NB, nt = M - b0;
        if (b0 > 0) PPBO_CL border_write_rows_kernel<<<dim3(ceil_div(b0, 256), nb), 256, 0, st>>>(ws.bR, Mp, ws.sa + M_old, M_old, nb, b0, Lfac, ldl);
        PPBO_CL newton_rows_kernel<<<dim3(ceil_div(M, 256), nt), 256, 0, st>>>(G, ldg, ws.sa, b0, M, M, b0, Lfac, ldl);
        PPBO_LAUNCH_CHECK();
        if (b0 > 0) {
            double* Lt = Lfac + (long long)b0 * ldl;
            GemmOperands g{Lt, ldl, 0, Lt, ldl, 0, nt, nt, b0};
            StoreEpilogue ep{Lt + b0, ldl, 0, -1.0, 1.0, 1, 0};
            if ((rc = launch_gemm_nt(g, ep, 1, st))) return rc;
        }
        if ((rc = potrf_lower(Lfac + (long long)b0 * ldl + b0, ldl, nt, Mdinv + (long long)(b0 / CHOL_NB) * CHOL_NB * CHOL_NB, ws.info, st)))
            return rc;
        PPBO_CUDA_CHECK(readback().add(&info, ws.info, sizeof(int), st));
        PPBO_CUDA_CHECK(readback().finish(st));
        factor_current = info == 0;
        info = 0;
    }
    if (binv_state_h) {
        if (bordered && !factor_at_mode) {      // cache built for the old factor; the finalisation rewrote rows >= the last 128-boundary
            binv_state_h[0] = (M_old / CHOL_NB) * CHOL_NB;
            binv_state_h[1] = ceil_div(M_old, 1024);
        } else if (binv_valid && !factor_at_mode && !identity_factor) {
            binv_state_h[0] = M;
            binv_state_h[1] = ceil_div(M, 1024);
        } else {
            binv_state_h[0] = binv_state_h[1] = 0;
        }
    }
    bool have_factor = factor_current && !identity_factor;
    if (sa_fac && have_factor && !factor_at_mode)
        PPBO_CUDA_CHECK(cudaMemcpyAsync(sa_fac, ws.sa, sizeof(double) * M, cudaMemcpyDeviceToDevice, st));
    // consistent products at the mode: arrow (signed); with PPBO_FIT_FACTOR_AT_MODE also the factor of I + a+^1/2 G a+^1/2 there
    // (what prediction WITH covariance needs -- ppbo_laplace_refactor builds it later otherwise)
    PPBO_CL lik_terms_kernel<<<set_blocks, 256, 0, st>>>(f_map, Q, m, sigma, ws.arrow_tmp, nullptr, arrow, ws.sa, nullptr);
    PPBO_CL sum_kernel<<<1, 1024, 0, st>>>(ws.arrow_tmp, Q, ws.scal + 24);
    if (factor_at_mode) {
        if ((rc = newton_matrix(G, ldg, M, ws.sa, Lfac, ldl, st))) return rc;
        if ((rc = potrf_lower(Lfac, ldl, M, Mdinv, ws.info, st))) return rc;
        ++n_factor;
        have_factor = true;
        if (sa_fac) PPBO_CUDA_CHECK(cudaMemcpyAsync(sa_fac, ws.sa, sizeof(double) * M, cudaMemcpyDeviceToDevice, st));
        PPBO_CUDA_CHECK(readback().add(&info, ws.info, sizeof(int), st));
    }
    PPBO_CUDA_CHECK(readback().finish(st));
    if (stats_h) {
        stats_h[0] = it;
        stats_h[1] = last_step;
        stats_h[2] = last_rel;
        stats_h[3] = T_cur;
        stats_h[4] = n_halvings_total;
        stats_h[5] = info;
        stats_h[6] = n_factor;
        stats_h[7] = n_chord;
        stats_h[8] = factor_at_mode ? 2.0 : (have_factor ? 1.0 : 0.0);   // 2: factor at the mode, 1: last Newton / warm factor, 0: none
        stats_h[9] = converged ? 1.0 : 0.0;
        stats_h[10] = warm_first_rel;
        stats_h[11] = nb;
    }
    if (info) { set_error("mode system not positive definite at pivot %d", info); return info; }
    return PPBO_OK;
}
