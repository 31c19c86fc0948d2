// ppbo_b200 -- K1: FP64 covariance matrices on sm_100a.
// Replaces kernels.SE_kernel / RQ_kernel / camphor_copper_kernel (src/kernels.py:19-53), GPModel.create_Gramian
// (= kernel + misc.regularize_covariance, src/gp_model.py:147-151, src/misc.py:71-88) and
// GPModel.create_Gramian_nonsquare (src/gp_model.py:153-155).
//
// Roofline: 8 n1 n2 bytes written, 8 (n1+n2) D read -> HBM-write bound for small D; at D = 20 the FP64 pipe
// (2 D + exp) is within ~2x of the HBM floor (DESIGN.md K1).  Layout: CTA tile 64 rows x 128 columns, the two
// point tiles staged in shared memory pre-scaled by 1/l_d; thread = 2 adjacent columns x 16 rows, 16-byte
// coalesced stores.
#include "../../include/ppbo_b200.h"
#include "common.cuh"
#include "gemm_f64.cuh"

namespace ppbo {

extern int g_tuning[16];

struct KernelParams {
    int kind, D;
    double inv_ls[PPBO_MAX_D];   // 1 / l_d
    double sf2;                  // sigma_f^2
    double diag_scale, diag_add; // out = diag_scale * k (+ diag_add on i == j) : fused shrinkage
};

constexpr int KT_M = 64, KT_N = 128, KT_THREADS = 256;

__device__ __forceinline__ double kernel_from_sums(int kind, double r2, double sf2) {
    // r2: scaled squared distance (SE / RQ / Matern) or the summed exponent (camphor)
    if (kind == PPBO_KERNEL_SE) return sf2 * exp(-0.5 * r2);
    if (kind == PPBO_KERNEL_RQ) { const double t = 1.0 + 0.25 * r2; return sf2 / (t * t); }   // alpha = 2
    if (kind == PPBO_KERNEL_SQDIST) return r2;                                                // kernels.dist: the distance itself
    if (kind == PPBO_KERNEL_MATERN32) { const double a = sqrt(3.0 * r2); return sf2 * (1.0 + a) * exp(-a); }
    if (kind == PPBO_KERNEL_MATERN52) { const double a = sqrt(5.0 * r2); return sf2 * (1.0 + a + 5.0 * r2 / 3.0) * exp(-a); }
    return sf2 * exp(-r2);
}

template <int KIND>
__global__ void __launch_bounds__(KT_THREADS) kernel_matrix_kernel(const double* __restrict__ X1, int n1,
                                                                   const double* __restrict__ X2, int n2,
                                                                   KernelParams p, double* __restrict__ out,
                                                                   long long ld, int symmetric_diag) {
    extern __shared__ double sm[];
    const int D = p.D;
    double* s1 = sm;                    // [KT_M][D]   rows of X1 (scaled)
    double* s2 = sm + KT_M * D;         // [D][KT_N]   columns = points of X2 (scaled), d-major
    const int r0 = blockIdx.y * KT_M, c0 = blockIdx.x * KT_N;
    for (int e = threadIdx.x; e < KT_M * D; e += KT_THREADS) {
        const int r = e / D, d = e % D;
        const int gr = r0 + r;
        const double v = gr < n1 ? X1[(long long)gr * D + d] : 0.0;
        s1[e] = (KIND == PPBO_KERNEL_CAMPHOR) ? v : v * p.inv_ls[d];
    }
    for (int e = threadIdx.x; e < KT_N * D; e += KT_THREADS) {
        const int c = e / D, d = e % D;
        const int gc = c0 + c;
        const double v = gc < n2 ? X2[(long long)gc * D + d] : 0.0;
        s2[d * KT_N + c] = (KIND == PPBO_KERNEL_CAMPHOR) ? v : v * p.inv_ls[d];
    }
    __syncthreads();
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;     // 64 column pairs x 4 row groups of 16
    const int c = c0 + 2 * tx;
    const bool vec_ok = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
#pragma unroll 4
    for (int rr = 0; rr < 16; ++rr) {
        const int rl = ty * 16 + rr, r = r0 + rl;
        if (r >= n1) break;
        double a0 = 0.0, a1 = 0.0;
        if (KIND == PPBO_KERNEL_CAMPHOR) {
            // periodic (period 1) on dims 0,1,3,4,5: 2 sin^2(pi |dx|) / l^2 ; SE on dim 2 with l + 0.05
            const double il = p.inv_ls[0], il2 = il * il, ilz = p.inv_ls[2];
#pragma unroll
            for (int d = 0; d < 6; ++d) {
                const double x = s1[rl * D + d];
                const double2 y = *reinterpret_cast<const double2*>(&s2[d * KT_N + 2 * tx]);
                const double d0 = fabs(x - y.x), d1 = fabs(x - y.y);
                if (d == 2) {
                    a0 += 0.5 * d0 * d0 * ilz * ilz;
                    a1 += 0.5 * d1 * d1 * ilz * ilz;
                } else {
                    const double q0 = sinpi(d0), q1 = sinpi(d1);
                    a0 += 2.0 * q0 * q0 * il2;
                    a1 += 2.0 * q1 * q1 * il2;
                }
            }
        } else {
            for (int d = 0; d < D; ++d) {
                const double x = s1[rl * D + d];
                const double2 y = *reinterpret_cast<const double2*>(&s2[d * KT_N + 2 * tx]);
                const double d0 = x - y.x, d1 = x - y.y;
                a0 = fma(d0, d0, a0);
                a1 = fma(d1, d1, a1);
            }
        }
        double k0 = p.diag_scale * kernel_from_sums(KIND, a0, p.sf2);
        double k1 = p.diag_scale * kernel_from_sums(KIND, a1, p.sf2);
        if (symmetric_diag) {
            if (r == c) k0 += p.diag_add;
            if (r == c + 1) k1 += p.diag_add;
        }
        double* o = out + (long long)r * ld + c;
        if (c + 1 < n2 && vec_ok) {
            *reinterpret_cast<double2*>(o) = make_double2(k0, k1);
        } else {
            if (c < n2) o[0] = k0;
            if (c + 1 < n2) o[1] = k1;
        }
    }
}


// SE / RQ / Matern kernels: register-tiled version.  Thread tile 8 rows x 4 columns; the 4 column points' coordinates are cached in
// registers 4 dimensions at a time, the row coordinates arrive as warp-broadcast shared-memory loads, so the inner loop
// issues 0.31 shared loads per FMA (the plain version above issues 1.0 and is LDS-bound at D = 20).  Stores: 32 B per thread,
// 1 KB contiguous per warp and row.
constexpr int KR_ROWS = 8, KR_COLS = 4, KR_DC = 4;
template <int KIND>
__global__ void __launch_bounds__(KT_THREADS, 2) kernel_matrix_tiled_kernel(const double* __restrict__ X1, int n1,
                                                                            const double* __restrict__ X2, int n2,
                                                                            KernelParams p, double* __restrict__ out,
                                                                            long long ld, int symmetric_diag) {
    extern __shared__ double sm[];
    const int D = p.D, Dp = (D + KR_DC - 1) / KR_DC * KR_DC;
    double* s1 = sm;                    // [KT_M][Dp]  rows of X1 (scaled), zero-padded dims
    double* s2 = sm + KT_M * Dp;        // [Dp][KT_N]  points of X2 (scaled), d-major
    const int r0 = blockIdx.y * KT_M, c0 = blockIdx.x * KT_N;
    for (int e = threadIdx.x; e < KT_M * Dp; e += KT_THREADS) {
        const int r = e / Dp, d = e % Dp, gr = r0 + r;
        s1[e] = (gr < n1 && d < D) ? X1[(long long)gr * D + d] * p.inv_ls[d] : 0.0;
    }
    for (int e = threadIdx.x; e < KT_N * Dp; e += KT_THREADS) {
        const int c = e / Dp, d = e % Dp, gc = c0 + c;
        s2[d * KT_N + c] = (gc < n2 && d < D) ? X2[(long long)gc * D + d] * p.inv_ls[d] : 0.0;
    }
    __syncthreads();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 column groups of 4 x 8 row groups of 8
    double acc[KR_ROWS][KR_COLS];
#pragma unroll
    for (int i = 0; i < KR_ROWS; ++i)
#pragma unroll
        for (int j = 0; j < KR_COLS; ++j) acc[i][j] = 0.0;
    for (int d0 = 0; d0 < Dp; d0 += KR_DC) {
        double y[KR_DC][KR_COLS];
#pragma unroll
        for (int dd = 0; dd < KR_DC; ++dd) {
            const double2 a = *reinterpret_cast<const double2*>(&s2[(d0 + dd) * KT_N + 4 * tx]);
            const double2 b = *reinterpret_cast<const double2*>(&s2[(d0 + dd) * KT_N + 4 * tx + 2]);
            y[dd][0] = a.x; y[dd][1] = a.y; y[dd][2] = b.x; y[dd][3] = b.y;
        }
#pragma unroll
        for (int i = 0; i < KR_ROWS; ++i) {
            const double* xr = &s1[(ty * KR_ROWS + i) * Dp + d0];
#pragma unroll
            for (int dd = 0; dd < KR_DC; ++dd) {
                const double x = xr[dd];
#pragma unroll
                for (int j = 0; j < KR_COLS; ++j) {
                    const double t = x - y[dd][j];
                    acc[i][j] = fma(t, t, acc[i][j]);
                }
            }
        }
    }
    const int c = c0 + 4 * tx;
    const bool vec_ok = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
#pragma unroll
    for (int i = 0; i < KR_ROWS; ++i) {
        const int r = r0 + ty * KR_ROWS + i;
        if (r >= n1) break;
        double k[KR_COLS];
#pragma unroll
        for (int j = 0; j < KR_COLS; ++j) {
            k[j] = p.diag_scale * kernel_from_sums(KIND, acc[i][j], p.sf2);
            if (symmetric_diag && r == c + j) k[j] += p.diag_add;
        }
        double* o = out + (long long)r * ld + c;
        if (c + 3 < n2 && vec_ok) {
            *reinterpret_cast<double2*>(o) = make_double2(k[0], k[1]);
            *reinterpret_cast<double2*>(o + 2) = make_double2(k[2], k[3]);
        } else {
#pragma unroll
            for (int j = 0; j < KR_COLS; ++j)
                if (c + j < n2) o[j] = k[j];
        }
    }
}

// ---- SE / RQ / Matern kernels on the FP64 tensor pipe -----------------------------------------------------------------------
// The scaled squared distance is formed the way the reference's kernels.dist does (src/kernels.py:3-11),
//   r2 = |x|^2 + |y|^2 - 2 x.y   clipped at 0,
// with the cross term as a DMMA product (D FMAs per pair instead of the 2 D of the difference form, 0.03 shared-memory loads per
// FMA).  Both point sets are shifted by the first point of X2 before scaling, which keeps |x|^2 (and with it the cancellation
// error 2.2e-16 (|x|^2 + |y|^2) of the expansion) at the squared diameter of the data in length-scale units.  Per entry: D FMAs of
// cross term on DMMA and 24 FP64 instructions of entry function (se_entry) share the FP64 pipe -- at D = 20 that is 1.45 entries
// per clock and SM (~410 G entries/s), which is what bounds the store and mat-vec modes (profiles/r02_ncu_gram.txt: FP64 41 % +
// DMMA 38 %); the symmetric mode computes half of the entries and is bound by its 8 N^2 bytes of stores.
// Modes:  KM_STORE     out[i][j] = k(x_i, y_j)                              (cross-covariances)
//         KM_SYMMETRIC X1 == X2: lower tiles only, every off-diagonal tile is also written transposed (+ fused shrinkage)
//         KM_MATVEC    partial[i][tile] = sum_{j in tile} k(x_i, y_j) alpha_j   (posterior mean without materialising the matrix)
constexpr int KM_B = 128, KM_BN = 64, KM_THREADS = 512;        // 128 x 64 tiles, 16 warps of 32 x 16, two CTAs per SM (32 warps
                                                                  // hide the 13-deep Horner chains of the entry function)
enum { KM_STORE = 0, KM_SYMMETRIC = 1, KM_MATVEC = 2 };
__host__ __device__ inline int km_ldx(int D) { const int Dp = (D + 3) / 4 * 4; return (Dp % 8 == 4) ? Dp : Dp + 4; }

// ---- streaming tensor-pipe kernel -------------------------------------------------------------------------------------------
// profiles/r01_ncu_gram.txt: the one-tile-per-CTA kernel of round 1 executed ~109 instructions per matrix entry, 22 of them FP64:
// every CTA re-derived its 192 rows of scaled coordinates (integer division per element, constant-bank reads of 1 / l_d), their norms
// and 64-bit store addresses for 16 entries per thread, at an IPC of 0.5 per scheduler.  Here
//   * a pre-pass writes every point once in "operand form": per tile of TR points one contiguous block [TR x LDX scaled, shifted
//     coordinates | TR squared norms | TR weights (alpha, mat-vec mode)], zero-padded to whole tiles;
//   * a CTA owns one 128-row tile and LOOPS over column tiles g, g + G, g + 2G, ... : the row block arrives once and every column
//     block as ONE cp.async.bulk (TMA 1-D copy) signalled on an mbarrier, double-buffered, so no thread instruction is spent on
//     loading, scaling or bounds;
//   * the epilogue is straight-line (branch-free exp, see exp_nonpos) with row pointers advanced by a constant per tile; tiles
//     that touch the diagonal or the matrix edge take a guarded path.
// The per-entry arithmetic (operand roles, DMMA k order, norms) does not depend on the tile or the launch shape, so appended rows
// (ppbo_gram_append) are bit-identical to a from-scratch build as before.
// Coefficients live in constant memory and enter the FMAs as constant-bank operands: FP64 literals have no immediate form, and
// under the 64-register budget of this kernel the compiler otherwise re-materialises every coefficient with two moves per use
// (253 IMAD.MOV next to 256 DFMA per 16 entries in the first version).  Horner form: one constant per FMA.
__constant__ double KM_EXP[23] = {
    1.4426950408889634,          // [0] log2(e)
    6755399441055744.0,          // [1] 2^52 + 2^51
    -6.93147180369123816490e-01, // [2] -ln2 (high part)
    -1.90821492927058770002e-10, // [3] -ln2 (low part)
    1.0, 1.0, 0.5, 1.6666666666666666e-01, 4.1666666666666664e-02, 8.3333333333333332e-03, 1.3888888888888889e-03,      // [4..] 1/k!
    1.9841269841269841e-04, 2.4801587301587302e-05, 2.7557319223985893e-06, 2.7557319223985888e-07, 2.5052108385441720e-08,
    2.0876756987868100e-09, 1.6059043836821613e-10,
    -708.0, -0.25,
    1.5, 2.5, 3.3333333333333331e-01};                                                                                // [20..22] Matern
// exp(x) for x in [-708, 0] (a little beyond -708 is fine: 2^n stays normal down to x = -708.39), straight-line:
//   x = n ln2 + r with |r| <= ln2 / 2 (rint by the 2^52 + 2^51 trick, ln2 in two pieces); exp(r) by its degree-13 Taylor polynomial
//   in Horner form (truncation 4e-18); 2^n by an integer add to the exponent field.  17 FP64 + 2 integer instructions.
__device__ __forceinline__ double km_exp(double x) {
    const double t = fma(x, KM_EXP[0], KM_EXP[1]);
    const int n = __double2loint(t);
    const double nf = t - KM_EXP[1];
    double r = fma(nf, KM_EXP[2], x);
    r = fma(nf, KM_EXP[3], r);
    double pv = KM_EXP[17];
#pragma unroll
    for (int k = 16; k >= 4; --k) pv = fma(pv, r, KM_EXP[k]);
    return __hiloint2double(__double2hiint(pv) + (n << 20), __double2loint(pv));
}
// SE entry from v = |x|^2 + |y|^2 - 2 x.y (may be slightly negative by cancellation):  sf2' exp(-max(v, 0) / 2), straight-line.
//   w = v + |v| = 2 max(v, 0) exactly (|.| is an operand modifier), its high word clamped at that of 2832 (exp(-708) = 3e-308: the
//   result stays a normal number whatever the inputs; one integer min instead of the ~8 instructions of a NaN-aware fmax);
//   then exp(-w / 4) by km_exp.  23 FP64 + 2 integer instructions.
__device__ __forceinline__ double se_entry(double v, double scale_c) {
    double w = v + fabs(v);
    w = __hiloint2double(min(__double2hiint(w), 0x40A62000), __double2loint(w));          // high word of 2832.0
    return scale_c * km_exp(w * KM_EXP[19]);
}
// Matern-nu entry (nu = 3/2, 5/2) from the same v, straight-line.  With a = sqrt(2 nu) r (r^2 = max(v, 0)):
//   q = nu (v + |v|) = a^2, its high word clamped to [that of 2^-1000, that of 708^2]: rsqrt_nr needs a normal operand, and
//   a <= 708 (+3e-7 relative: the low word is kept) keeps exp(-a) normal as in se_entry.  At v <= 0 the entry is sf2' exactly
//   (a = 2^-500 rounds away).  a = q rsqrt_nr(q) (one MUFU + 9 FP64); e = sf2' exp(-a) by km_exp;
//   nu = 3/2: (1 + a) e,  nu = 5/2: (1 + a + a^2 / 3) e, the prefactor folded into the last FMA(s).  The coefficients (nu, 1/3)
//   are constant-bank operands like the exp's.
template <int KIND>
__device__ __forceinline__ double matern_entry(double v, double scale_c) {
    double q = (v + fabs(v)) * KM_EXP[KIND == PPBO_KERNEL_MATERN32 ? 20 : 21];
    q = __hiloint2double(max(min(__double2hiint(q), 0x411E9840), 0x01700000), __double2loint(q));     // [2^-1000, 708^2]
    const double a = q * rsqrt_nr(q);
    const double pf = (KIND == PPBO_KERNEL_MATERN32) ? a : fma(q, KM_EXP[22], a);                        // prefactor - 1
    const double e = scale_c * km_exp(-a);
    return fma(pf, e, e);
}
template <int KIND>
__device__ __forceinline__ double km_entry(double v, double scale_c, double sf2, double diag_scale) {
    if (KIND == PPBO_KERNEL_SE) return se_entry(v, scale_c);
    if (KIND == PPBO_KERNEL_MATERN32 || KIND == PPBO_KERNEL_MATERN52) return matern_entry<KIND>(v, scale_c);
    return diag_scale * kernel_from_sums(KIND, fmax(v, 0.0), sf2);
}

__host__ __device__ inline long long km_block_doubles(int TR, int LDX) { return (long long)TR * LDX + 2 * TR; }

// operand form of n points (rows of X, row stride D): tile t = rows [t TR, (t+1) TR), zero beyond n
__global__ void __launch_bounds__(128) km_prepare_kernel(const double* __restrict__ X, int n, int TR, KernelParams p,
                                                         const double* __restrict__ shift, const double* __restrict__ alpha,
                                                         double* __restrict__ out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int D = p.D, Dp = (D + 3) / 4 * 4, LDX = km_ldx(D);
    const int tiles = (n + TR - 1) / TR;
    if (r >= tiles * TR) return;
    double* blk = out + (long long)(r / TR) * km_block_doubles(TR, LDX);
    double* row = blk + (long long)(r % TR) * LDX;
    double s = 0.0;
    for (int d = 0; d < LDX; ++d) {
        const double v = (r < n && d < D) ? (X[(long long)r * D + d] - shift[d]) * p.inv_ls[d] : 0.0;
        row[d] = v;
        if (d < Dp) s = fma(v, v, s);
    }
    blk[(long long)TR * LDX + (r % TR)] = s;
    blk[(long long)TR * LDX + TR + (r % TR)] = (alpha != nullptr && r < n) ? alpha[r] : 0.0;
}

__device__ __forceinline__ uint32_t km_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void km_bulk_load(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(km_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(km_smem_u32(dst_smem)),
                 "l"(src), "r"(bytes), "r"(km_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void km_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(km_smem_u32(bar)), "r"(parity)
            : "memory");
    }
}

// P1: operand form of X1 in tiles of 128, P2: of X2 in tiles of 64.  grid = (G column groups, row tiles); CTA (g, ti) takes the
// column tiles tj = g, g + G, ... below nt_of(ti) (all tn tiles, or 2 ti + 2 in symmetric mode: the lower triangle).
// MATVEC: out[row][g] = sum over the CTA's column tiles of k(x_row, y_j) alpha_j (ld = G).
template <int KIND, int MODE>
__global__ void __launch_bounds__(KM_THREADS, 2) kernel_matrix_stream_kernel(const double* __restrict__ P1, int n1,
                                                                          const double* __restrict__ P2, int n2, int D, double sf2,
                                                                          double diag_scale, double diag_add, double* __restrict__ out,
                                                                          long long ld, int tn) {
    extern __shared__ __align__(16) double sm[];
    const int LDX = km_ldx(D), Dp = (D + 3) / 4 * 4;
    const long long blk1 = km_block_doubles(KM_B, LDX), blk2 = km_block_doubles(KM_BN, LDX);
    double* Xs = sm;                                   // [128 x LDX | 128 norms | 128 unused]
    double* Yb[2] = {sm + blk1, sm + blk1 + blk2};     // [64 x LDX | 64 norms | 64 weights] x 2
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + blk1 + 2 * blk2);      // [0]: row block, [1], [2]: column buffers
    const int ti = blockIdx.y, g = blockIdx.x, G = gridDim.x;
    const int nt = (MODE == KM_SYMMETRIC) ? min(tn, 2 * ti + 2) : tn;
    const int ntiles = (nt > g) ? (nt - g + G - 1) / G : 0;
    if (ntiles == 0) return;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int i = 0; i < 3; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(km_smem_u32(bars + i)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        km_bulk_load(Xs, P1 + (long long)ti * blk1, (uint32_t)(blk1 * 8), bars);
        km_bulk_load(Yb[0], P2 + (long long)g * blk2, (uint32_t)(blk2 * 8), bars + 1);
    }
    const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t4 = lane & 3;
    const int wm0 = (warp >> 2) * 32, wn0 = (warp & 3) * 16;       // 4 x 4 warps, 32 x 16 each
    const int m0 = ti * KM_B;
    const double scale_c = diag_scale * sf2;
    const double* nx = Xs + KM_B * LDX;
    const double* Ap = Xs + (wm0 + gq) * LDX + t4;
    double rowsum[4] = {0.0, 0.0, 0.0, 0.0};
    const bool vec_ok = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    const bool rows_full = m0 + KM_B <= n1;
    km_wait(bars, 0);
    const double* nxp = nx + wm0 + gq;                  // nxp[mi * 8]: squared norm of this thread's row mi
    for (int it = 0; it < ntiles; ++it) {
        const int buf = it & 1, tj = g + it * G, c0 = tj * KM_BN;
        if (tid == 0 && it + 1 < ntiles)               // (buffer buf ^ 1 was last read in iteration it - 1, behind its barrier)
            km_bulk_load(Yb[buf ^ 1], P2 + (long long)(tj + G) * blk2, (uint32_t)(blk2 * 8), bars + 1 + (buf ^ 1));
        km_wait(bars + 1 + buf, (uint32_t)((it >> 1) & 1));
        const double* Ys = Yb[buf];
        const double* ny = Ys + KM_BN * LDX;
        const double* al = ny + KM_BN;
        double acc[4][2][2];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 2; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
        const double* Bp = Ys + (wn0 + gq) * LDX + t4;
        for (int k = 0; k < Dp; k += 4) {
            double a[4], b[2];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) a[mi] = Ap[mi * 8 * LDX + k];
#pragma unroll
            for (int ni = 0; ni < 2; ++ni) b[ni] = Bp[ni * 8 * LDX + k];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 2; ++ni) dmma884(acc[mi][ni], a[mi], b[ni]);
        }
        const double* nyp = ny + wn0 + 2 * t4;             // nyp[nn * 8 + e], alp likewise (16-byte aligned pairs)
        const double* alp = al + wn0 + 2 * t4;
        if (MODE == KM_MATVEC) {
            // padded columns carry weight 0 and a finite kernel value: no bounds needed
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int nn = 0; nn < 2; ++nn)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const double r2 = fma(-2.0, acc[mi][nn][e], nxp[mi * 8] + nyp[nn * 8 + e]);      // clamped at 0 inside km_entry
                        rowsum[mi] = fma(km_entry<KIND>(r2, scale_c, sf2, diag_scale), alp[nn * 8 + e], rowsum[mi]);
                    }
        } else {
            const bool interior = rows_full && c0 + KM_BN <= n2 && vec_ok && !(MODE == KM_SYMMETRIC && c0 + KM_BN > m0);
            if (interior) {                            // full tile, strictly below the diagonal blocks in symmetric mode
                double* o = out + (long long)(m0 + wm0 + gq) * ld + c0 + wn0 + 2 * t4;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
#pragma unroll
                    for (int nn = 0; nn < 2; ++nn) {
                        double kv[2];
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const double r2 = fma(-2.0, acc[mi][nn][e], nxp[mi * 8] + nyp[nn * 8 + e]);      // clamped at 0 inside km_entry
                            kv[e] = km_entry<KIND>(r2, scale_c, sf2, diag_scale);
                        }
                        *reinterpret_cast<double2*>(o + (long long)mi * 8 * ld + nn * 8) = make_double2(kv[0], kv[1]);
                        if (MODE == KM_SYMMETRIC) {    // mirror (8 consecutive doubles per (t4, e) across gq)
                            double* om = out + (long long)(c0 + wn0 + nn * 8 + 2 * t4) * ld + m0 + wm0 + mi * 8 + gq;
                            om[0] = kv[0];
                            om[ld] = kv[1];
                        }
                    }
                }
            } else {
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
                    const int gr = m0 + wm0 + mi * 8 + gq;
#pragma unroll
                    for (int nn = 0; nn < 2; ++nn) {
                        const int gc = c0 + wn0 + nn * 8 + 2 * t4;
                        double kv[2];
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const double r2 = fma(-2.0, acc[mi][nn][e], nxp[mi * 8] + nyp[nn * 8 + e]);      // clamped at 0 inside km_entry
                            kv[e] = km_entry<KIND>(r2, scale_c, sf2, diag_scale);
                            if (MODE == KM_SYMMETRIC && gr == gc + e) kv[e] = fma(diag_scale, sf2, diag_add);  // exact diagonal: ONE rounding,
                        }                                                                                    // as in gram_mirror_kernel
                        if (gr < n1) {
                            double* o = out + (long long)gr * ld + gc;
                            if (gc + 1 < n2 && vec_ok) *reinterpret_cast<double2*>(o) = make_double2(kv[0], kv[1]);
                            else {
                                if (gc < n2) o[0] = kv[0];
                                if (gc + 1 < n2) o[1] = kv[1];
                            }
                            if (MODE == KM_SYMMETRIC && c0 + KM_BN <= m0) {
                                if (gc < n2) out[(long long)gc * ld + gr] = kv[0];
                                if (gc + 1 < n2) out[(long long)(gc + 1) * ld + gr] = kv[1];
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();                               // everybody is done with Yb[buf] before it is refilled
    }
    if (MODE == KM_MATVEC) {
        double* red = Yb[0];                           // [128][4] cross-warp buffer (all column blocks are consumed)
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
            double v = rowsum[mi];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            if (t4 == 0) red[(wm0 + mi * 8 + gq) * 4 + (warp & 3)] = v;
        }
        __syncthreads();
        if (tid < KM_B && m0 + tid < n1)
            out[(long long)(m0 + tid) * G + g] = (red[tid * 4] + red[tid * 4 + 1]) + (red[tid * 4 + 2] + red[tid * 4 + 3]);
    }
}

// mu[r] = sum_c partial[r][c] in a fixed order
__global__ void __launch_bounds__(256) km_rowsum_kernel(const double* __restrict__ partial, int n, int nc, double* __restrict__ mu) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double s = 0.0;
    for (int c = 0; c < nc; ++c) s += partial[(long long)r * nc + c];
    mu[r] = s;
}

// column groups per row tile: ~6 column tiles per CTA (the row block and the per-CTA setup are amortised over them) and enough
// CTAs for several waves of 2 x 148
static int km_column_groups(int tm, int tn) {
    int G = ceil_div(tn, 6);
    while (G < tn && (long long)G * tm < 4LL * 2 * PPBO_SM_COUNT) ++G;
    return G < 1 ? 1 : G;
}

template <int KIND>
static int launch_kernel_matrix_mma(const KernelParams& p, const double* X1, int n1, const double* X2, int n2, double* out,
                                    long long ld, int mode, const double* alpha, cudaStream_t st, int* groups_out = nullptr) {
    const int LDX = km_ldx(p.D);
    const long long blk1 = km_block_doubles(KM_B, LDX), blk2 = km_block_doubles(KM_BN, LDX);
    const size_t smem = (size_t)(blk1 + 2 * blk2) * sizeof(double) + 32;
    static bool attr_done = false;
    if (!attr_done) {
        const int LM = km_ldx(PPBO_MAX_D);
        const int max_smem = (int)((km_block_doubles(KM_B, LM) + 2 * km_block_doubles(KM_BN, LM)) * sizeof(double)) + 32;
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_stream_kernel<KIND, KM_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_stream_kernel<KIND, KM_SYMMETRIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_stream_kernel<KIND, KM_MATVEC>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        attr_done = true;
    }
    const int tm = ceil_div(n1, KM_B), tn = ceil_div(n2, KM_BN);
    // operand form of both point sets (stream-ordered scratch): tiles of 128 rows for X1, of 64 rows for X2
    double* P1 = nullptr;
    PPBO_CUDA_CHECK(malloc_async((void**)reinterpret_cast<void**>(&P1), sizeof(double) * (tm * blk1 + tn * blk2), st));
    double* P2 = P1 + tm * blk1;
    PPBO_CL km_prepare_kernel<<<ceil_div(tm * KM_B, 128), 128, 0, st>>>(X1, n1, KM_B, p, X2, nullptr, P1);
    PPBO_CL km_prepare_kernel<<<ceil_div(tn * KM_BN, 128), 128, 0, st>>>(X2, n2, KM_BN, p, X2, alpha, P2);
    const int G = km_column_groups(tm, tn);
    if (groups_out) *groups_out = G;
    const dim3 grid(G, tm);
    if (mode == KM_SYMMETRIC)
        PPBO_CL kernel_matrix_stream_kernel<KIND, KM_SYMMETRIC><<<grid, KM_THREADS, smem, st>>>(P1, n1, P2, n2, p.D, p.sf2, p.diag_scale, p.diag_add, out, ld, tn);
    else if (mode == KM_MATVEC)
        PPBO_CL kernel_matrix_stream_kernel<KIND, KM_MATVEC><<<grid, KM_THREADS, smem, st>>>(P1, n1, P2, n2, p.D, p.sf2, p.diag_scale, p.diag_add, out, G, tn);
    else
        PPBO_CL kernel_matrix_stream_kernel<KIND, KM_STORE><<<grid, KM_THREADS, smem, st>>>(P1, n1, P2, n2, p.D, p.sf2, p.diag_scale, p.diag_add, out, ld, tn);
    PPBO_LAUNCH_CHECK();
    PPBO_CUDA_CHECK(cudaFreeAsync(P1, st));
    return PPBO_OK;
}

static bool km_has_mma(int kind) {
    return kind == PPBO_KERNEL_SE || kind == PPBO_KERNEL_RQ || kind == PPBO_KERNEL_MATERN32 || kind == PPBO_KERNEL_MATERN52;
}
static int launch_kernel_matrix_mma_kind(const KernelParams& p, const double* X1, int n1, const double* X2, int n2, double* out,
                                         long long ld, int mode, const double* alpha, cudaStream_t st, int* groups_out = nullptr) {
    switch (p.kind) {
        case PPBO_KERNEL_SE: return launch_kernel_matrix_mma<PPBO_KERNEL_SE>(p, X1, n1, X2, n2, out, ld, mode, alpha, st, groups_out);
        case PPBO_KERNEL_RQ: return launch_kernel_matrix_mma<PPBO_KERNEL_RQ>(p, X1, n1, X2, n2, out, ld, mode, alpha, st, groups_out);
        case PPBO_KERNEL_MATERN32:
            return launch_kernel_matrix_mma<PPBO_KERNEL_MATERN32>(p, X1, n1, X2, n2, out, ld, mode, alpha, st, groups_out);
        case PPBO_KERNEL_MATERN52:
            return launch_kernel_matrix_mma<PPBO_KERNEL_MATERN52>(p, X1, n1, X2, n2, out, ld, mode, alpha, st, groups_out);
    }
    PPBO_REQUIRE(false, "kernel kind has no tensor-pipe version");
}

static int fill_params(KernelParams& p, int kind, int D, const double* ls_h, double sigma_f) {
    PPBO_REQUIRE(kind >= 0 && kind <= PPBO_KERNEL_MATERN52, "unknown kernel kind");
    PPBO_REQUIRE(D >= 1 && D <= PPBO_MAX_D, "D must be in [1, 64]");
    PPBO_REQUIRE(kind != PPBO_KERNEL_CAMPHOR || D == 6, "camphor_copper_kernel is defined for D = 6 only");
    PPBO_REQUIRE(ls_h != nullptr && sigma_f > 0, "hyper-parameters");
    p.kind = kind;
    p.D = D;
    for (int d = 0; d < PPBO_MAX_D; ++d) p.inv_ls[d] = 0.0;
    for (int d = 0; d < D; ++d) {
        PPBO_REQUIRE(ls_h[d] > 0, "length-scales must be positive");
        p.inv_ls[d] = 1.0 / ls_h[d];
    }
    if (kind == PPBO_KERNEL_CAMPHOR) p.inv_ls[2] = 1.0 / (ls_h[2] + 0.05);   // src/kernels.py:48
    p.sf2 = sigma_f * sigma_f;
    p.diag_scale = 1.0;
    p.diag_add = 0.0;
    return PPBO_OK;
}

int kernel_matrix(const KernelParams& p, const double* X1, int n1, const double* X2, int n2, double* out,
                  long long ld, int symmetric_diag, cudaStream_t st) {
    if (n1 <= 0 || n2 <= 0) return PPBO_OK;
    dim3 grid(ceil_div(n2, KT_N), ceil_div(n1, KT_M));
    const size_t smem = (size_t)(KT_M + KT_N) * p.D * sizeof(double);
    static bool attr_done = false;
    if (!attr_done) {   // D up to 64 needs 96 KB of dynamic shared memory
        const int max_smem = (KT_M + KT_N) * PPBO_MAX_D * (int)sizeof(double);
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_kernel<PPBO_KERNEL_SE>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_kernel<PPBO_KERNEL_RQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_kernel<PPBO_KERNEL_CAMPHOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_tiled_kernel<PPBO_KERNEL_SE>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_tiled_kernel<PPBO_KERNEL_RQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_tiled_kernel<PPBO_KERNEL_SQDIST>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_tiled_kernel<PPBO_KERNEL_MATERN32>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        PPBO_CUDA_CHECK(cudaFuncSetAttribute(kernel_matrix_tiled_kernel<PPBO_KERNEL_MATERN52>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        attr_done = true;
    }
    if (p.kind == PPBO_KERNEL_SQDIST) {         // squared distances: difference form (no cancellation), no tensor-pipe variant
        const int Dp = (p.D + KR_DC - 1) / KR_DC * KR_DC;
        PPBO_CL kernel_matrix_tiled_kernel<PPBO_KERNEL_SQDIST><<<grid, KT_THREADS, (size_t)(KT_M + KT_N) * Dp * sizeof(double), st>>>(
            X1, n1, X2, n2, p, out, ld, 0);
        PPBO_LAUNCH_CHECK();
        return PPBO_OK;
    }
    if (g_tuning[11] == 0 && km_has_mma(p.kind)) {     // tuning key 11 = 1: difference-form kernels
        const int mode = (symmetric_diag && X1 == X2 && n1 == n2) ? KM_SYMMETRIC : KM_STORE;
        KernelParams q = p;
        if (mode != KM_SYMMETRIC) q.diag_add = 0.0;
        if (symmetric_diag && mode != KM_SYMMETRIC) goto general;       // diagonal term on a non-aliased pair: keep the old path
        return launch_kernel_matrix_mma_kind(q, X1, n1, X2, n2, out, ld, mode, nullptr, st);
    }
general:
    const int Dp = (p.D + KR_DC - 1) / KR_DC * KR_DC;
    const size_t smem_t = (size_t)(KT_M + KT_N) * Dp * sizeof(double);
    switch (p.kind) {
        case PPBO_KERNEL_SE:
            PPBO_CL kernel_matrix_tiled_kernel<PPBO_KERNEL_SE><<<grid, KT_THREADS, smem_t, st>>>(X1, n1, X2, n2, p, out, ld, symmetric_diag);
            break;
        case PPBO_KERNEL_RQ:
            PPBO_CL kernel_matrix_tiled_kernel<PPBO_KERNEL_RQ><<<grid, KT_THREADS, smem_t, st>>>(X1, n1, X2, n2, p, out, ld, symmetric_diag);
            break;
        case PPBO_KERNEL_MATERN32:
            PPBO_CL kernel_matrix_tiled_kernel<PPBO_KERNEL_MATERN32><<<grid, KT_THREADS, smem_t, st>>>(X1, n1, X2, n2, p, out, ld, symmetric_diag);
            break;
        case PPBO_KERNEL_MATERN52:
            PPBO_CL kernel_matrix_tiled_kernel<PPBO_KERNEL_MATERN52><<<grid, KT_THREADS, smem_t, st>>>(X1, n1, X2, n2, p, out, ld, symmetric_diag);
            break;
        case PPBO_KERNEL_CAMPHOR:
            PPBO_CL kernel_matrix_kernel<PPBO_KERNEL_CAMPHOR><<<grid, KT_THREADS, smem, st>>>(X1, n1, X2, n2, p, out, ld, symmetric_diag);
            break;
        default:
            PPBO_REQUIRE(false, "unknown kernel kind");
    }
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

// internal entry used by predict (acq.cu)
int kernel_matrix_raw(int kind, const double* X1, int n1, const double* X2, int n2, int D, const double* ls_h,
                      double sigma_f, double scale, double diag_add, double* out, long long ld, cudaStream_t st) {
    KernelParams p;
    int rc = fill_params(p, kind, D, ls_h, sigma_f);
    if (rc) return rc;
    p.diag_scale = scale;
    p.diag_add = diag_add;
    return kernel_matrix(p, X1, n1, X2, n2, out, ld, diag_add != 0.0, st);
}

// mu[i] = sum_j k(X1_i, X2_j) alpha_j without materialising the n1 x n2 matrix (GPModel.mu_pred batched, src/gp_model.py:454-458);
// partial: n1 * ceil(n2 / 64) doubles of scratch.  Returns 1 when done, 0 when the kernel kind has no tensor-pipe version.
int kernel_matvec(int kind, const double* X1, int n1, const double* X2, int n2, int D, const double* ls_h, double sigma_f,
                  const double* alpha, double* mu, double* partial, cudaStream_t st) {
    if (g_tuning[11] != 0 || !km_has_mma(kind)) return 0;
    KernelParams p;
    int rc = fill_params(p, kind, D, ls_h, sigma_f);
    if (rc) return rc;
    if (n1 <= 0) return 1;
    int G = 1;
    rc = launch_kernel_matrix_mma_kind(p, X1, n1, X2, n2, partial, 0, KM_MATVEC, alpha, st, &G);
    if (rc) return rc;
    PPBO_CL km_rowsum_kernel<<<ceil_div(n1, 256), 256, 0, st>>>(partial, n1, G, mu);
    PPBO_LAUNCH_CHECK();
    return 1;
}

// ---- posterior mean at ONE point with host-resident argument and result ------------------------------------------------------
// GPModel.mu_star (src/gp_model.py:415-437) drives ~10^4 SEQUENTIAL evaluations of mu_pred (src/gp_model.py:454-458) from scipy's
// differential evolution ('immediate' updating: every trial depends on the previous accept / reject, so the evaluations cannot be
// batched without changing the reference's RNG trajectory).  Per evaluation the general path paid a tensor allocation, a pageable
// H2D copy, two launches and a D2H copy.  Here the point and the result live in mapped pinned host memory (one small buffer per
// host thread): the host writes x, one single-CTA launch reads it over PCIe, accumulates sum_i k(x, X_i) alpha_i in a fixed order
// (difference form, like kernel_matrix_kernel) and writes the mean back; the host waits on the stream.
template <int KIND>
__global__ void __launch_bounds__(1024) mu_pred_point_kernel(const double* __restrict__ X, int N, KernelParams p,
                                                             const double* __restrict__ alpha, const double* __restrict__ x_in,
                                                             double* __restrict__ out) {
    __shared__ double xs[PPBO_MAX_D];
    __shared__ double red[33];
    const int D = p.D;
    for (int d = threadIdx.x; d < D; d += 1024) xs[d] = x_in[(long long)blockIdx.x * D + d];     // one point per CTA
    __syncthreads();
    double s = 0.0;
    for (int i = threadIdx.x; i < N; i += 1024) {
        const double* xi = X + (long long)i * D;
        double a = 0.0;
        if (KIND == PPBO_KERNEL_CAMPHOR) {
            const double il = p.inv_ls[0], il2 = il * il, ilz = p.inv_ls[2];
#pragma unroll
            for (int d = 0; d < 6; ++d) {
                const double d0 = fabs(xs[d] - xi[d]);
                if (d == 2) a += 0.5 * d0 * d0 * ilz * ilz;
                else { const double q0 = sinpi(d0); a += 2.0 * q0 * q0 * il2; }
            }
        } else {
            for (int d = 0; d < D; ++d) {
                const double t = (xs[d] - xi[d]) * p.inv_ls[d];
                a = fma(t, t, a);
            }
        }
        s = fma(kernel_from_sums(KIND, a, p.sf2), alpha[i], s);
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[blockIdx.x] = s;
}

struct PinnedPoint {
    double* host = nullptr;
    double* dev = nullptr;
    int init() {
        if (host) return PPBO_OK;
        PPBO_CUDA_CHECK(cudaHostAlloc(&host, sizeof(double) * (PPBO_MAX_D + 8), cudaHostAllocMapped));
        PPBO_CUDA_CHECK(cudaHostGetDevicePointer(&dev, host, 0));
        return PPBO_OK;
    }
};
static thread_local PinnedPoint g_point;
// B points per launch (ppbo_mu_pred_points: the speculative windows of the differential evolution in de.cu)
struct PinnedBatch {
    double* host = nullptr;
    double* dev = nullptr;
    int init() {
        if (host) return PPBO_OK;
        PPBO_CUDA_CHECK(cudaHostAlloc(&host, sizeof(double) * (PPBO_MAX_D + 1) * PPBO_MAX_POINTS, cudaHostAllocMapped));
        PPBO_CUDA_CHECK(cudaHostGetDevicePointer(&dev, host, 0));
        return PPBO_OK;
    }
};
static thread_local PinnedBatch g_batch;

// ---- SE kernel gradients w.r.t. log length-scales and log sigma_f --------------------------------------
__global__ void __launch_bounds__(256) se_grad_kernel(const double* __restrict__ X1, int n1, const double* __restrict__ X2,
                                                      int n2, KernelParams p, double* __restrict__ dK, long long ld,
                                                      long long stride) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n1 * n2) return;
    const int i = (int)(idx / n2), j = (int)(idx % n2);
    double r2 = 0.0;
    for (int d = 0; d < p.D; ++d) {
        const double t = (X1[(long long)i * p.D + d] - X2[(long long)j * p.D + d]) * p.inv_ls[d];
        r2 = fma(t, t, r2);
    }
    const double k = p.sf2 * exp(-0.5 * r2);
    for (int d = 0; d < p.D; ++d) {
        const double t = (X1[(long long)i * p.D + d] - X2[(long long)j * p.D + d]) * p.inv_ls[d];
        dK[d * stride + (long long)i * ld + j] = k * t * t;          // dK / dlog l_d
    }
    dK[p.D * stride + (long long)i * ld + j] = 2.0 * k;               // dK / dlog sigma_f
}

// ---- difference-space Gram matrix and the Newton system matrix -----------------------------------------
// G[u][v] = S[r(u)][r(v)] - S[r(u)][w(v)] - S[w(u)][r(v)] + S[w(u)][w(v)],  u = (q, j): r = q(m+1)+1+j, w = q(m+1)
__global__ void __launch_bounds__(256) diffspace_gram_kernel(const double* __restrict__ S, long long lds, int Q, int m,
                                                             double* __restrict__ G, long long ldg) {
    const int M = Q * m;
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    const int u = blockIdx.y;
    if (v >= M) return;
    const int qu = u / m, ju = u % m, qv = v / m, jv = v % m;
    const long long ru = (long long)qu * (m + 1) + 1 + ju, wu = (long long)qu * (m + 1);
    const long long rv = (long long)qv * (m + 1) + 1 + jv, wv = (long long)qv * (m + 1);
    G[(long long)u * ldg + v] = (S[ru * lds + rv] - S[ru * lds + wv]) - (S[wu * lds + rv] - S[wu * lds + wv]);
}

// Mmat[u][v] = delta_uv + sa[u] G[u][v] sa[v] on the lower triangle (v <= u), the part the Cholesky reads
__global__ void __launch_bounds__(256) newton_matrix_kernel(const double* __restrict__ G, long long ldg, int M,
                                                            const double* __restrict__ sa, double* __restrict__ out,
                                                            long long ldo) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    const int u = blockIdx.y;
    if (v >= M || (int)(blockIdx.x * blockDim.x) > u) return;
    if (v > u) return;
    double x = sa[u] * G[(long long)u * ldg + v] * sa[v];
    if (u == v) x += 1.0;
    out[(long long)u * ldo + v] = x;
}

// K <- (1 - s) K + s (tr K / n) I in place: the closed form of sklearn's shrunk_covariance used by misc.regularize_covariance
// (src/misc.py:85).  Single CTA computes the trace in a fixed order, then the grid scales.
__global__ void __launch_bounds__(1024) trace_kernel(const double* __restrict__ K, long long ld, int n, double* __restrict__ out) {
    __shared__ double red[33];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 1024) s += K[(long long)i * ld + i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[0] = s / n;
}
__global__ void __launch_bounds__(256) shrink_kernel(double* __restrict__ K, long long ld, int n, double s,
                                                     const double* __restrict__ mu) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= n) return;
    double v = (1.0 - s) * K[(long long)i * ld + j];
    if (i == j) v += s * mu[0];
    K[(long long)i * ld + j] = v;
}
__global__ void __launch_bounds__(256) set_identity_kernel(double* __restrict__ A, long long ld, int n) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j < n) A[(long long)i * ld + j] = (i == j) ? 1.0 : 0.0;
}
int set_identity(double* A, long long ld, int n, cudaStream_t st) {
    if (n <= 0) return PPBO_OK;
    PPBO_CL set_identity_kernel<<<dim3(ceil_div(n, 256), n), 256, 0, st>>>(A, ld, n);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

int diffspace_gram(const double* S, long long lds, int Q, int m, double* G, long long ldg, cudaStream_t st) {
    const int M = Q * m;
    if (M <= 0) return PPBO_OK;
    dim3 grid(ceil_div(M, 256), M);
    PPBO_CL diffspace_gram_kernel<<<grid, 256, 0, st>>>(S, lds, Q, m, G, ldg);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

// Appended comparison sets: every entry of G with a row or a column in [M_old, M_new), by the expression of
// diffspace_gram_kernel (so the grown matrix is bit-identical to a from-scratch one).  blockIdx.y enumerates the new rows first
// (full rows), then the old rows (new columns only).
__global__ void __launch_bounds__(256) diffspace_gram_append_kernel(const double* __restrict__ S, long long lds, int M_old, int M_new,
                                                                    int m, double* __restrict__ G, long long ldg) {
    const int nn = M_new - M_old;
    int u, v;
    if ((int)blockIdx.y < nn) {
        u = M_old + blockIdx.y;
        v = blockIdx.x * blockDim.x + threadIdx.x;
        if (v >= M_new) return;
    } else {
        u = blockIdx.y - nn;
        v = M_old + blockIdx.x * blockDim.x + threadIdx.x;
        if (v >= M_new) return;
    }
    const int qu = u / m, ju = u % m, qv = v / m, jv = v % m;
    const long long ru = (long long)qu * (m + 1) + 1 + ju, wu = (long long)qu * (m + 1);
    const long long rv = (long long)qv * (m + 1) + 1 + jv, wv = (long long)qv * (m + 1);
    G[(long long)u * ldg + v] = (S[ru * lds + rv] - S[ru * lds + wv]) - (S[wu * lds + rv] - S[wu * lds + wv]);
}

int diffspace_gram_append(const double* S, long long lds, int Q_old, int Q_new, int m, double* G, long long ldg, cudaStream_t st) {
    const int M_old = Q_old * m, M_new = Q_new * m;
    if (M_new <= M_old) return PPBO_OK;
    PPBO_CL diffspace_gram_append_kernel<<<dim3(ceil_div(M_new, 256), M_new), 256, 0, st>>>(S, lds, M_old, M_new, m, G, ldg);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

// out[j][i] = out[i][j] for the appended rows i in [n_old, n_new) and all j < i; the diagonal of the appended rows is set to the
// exact value every from-scratch kernel stores there
__global__ void __launch_bounds__(256) gram_mirror_kernel(double* __restrict__ out, long long ld, int n_old, int n_new,
                                                          double diag_scale, double sf2, double diag_add) {
    const int i = n_old + blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_new || j > i) return;
    if (j == i) out[(long long)i * ld + i] = fma(diag_scale, sf2, diag_add);    // same value as the from-scratch kernels (one rounding)
    else out[(long long)j * ld + i] = out[(long long)i * ld + j];
}

int newton_matrix(const double* G, long long ldg, int M, const double* sa, double* out, long long ldo, cudaStream_t st) {
    if (M <= 0) return PPBO_OK;
    dim3 grid(ceil_div(M, 256), M);
    PPBO_CL newton_matrix_kernel<<<grid, 256, 0, st>>>(G, ldg, M, sa, out, ldo);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

}  // namespace ppbo

using namespace ppbo;

extern "C" int ppbo_kernel_matrix(int kind, const double* X1, int n1, const double* X2, int n2, int D,
                                  const double* lengthscales_h, double sigma_f, double* out, long long ld, void* stream) {
    PPBO_REQUIRE(n1 >= 0 && n2 >= 0 && ld >= n2, "shape");
    return kernel_matrix_raw(kind, X1, n1, X2, n2, D, lengthscales_h, sigma_f, 1.0, 0.0, out, ld, (cudaStream_t)stream);
}

/* out[n1 x n2] = |X1_i - X2_j|^2 (kernels.dist, src/kernels.py:3-11: the reference expands |x|^2 + |y|^2 - 2 x.y and clips at 0; the
 * difference form used here has no cancellation, so the clip never acts) */
extern "C" int ppbo_sqdist(const double* X1, int n1, const double* X2, int n2, int D, double* out, long long ld, void* stream) {
    PPBO_REQUIRE(n1 >= 0 && n2 >= 0 && ld >= n2 && D >= 1 && D <= PPBO_MAX_D, "shape");
    double ones[PPBO_MAX_D];
    for (int d = 0; d < PPBO_MAX_D; ++d) ones[d] = 1.0;
    return kernel_matrix_raw(PPBO_KERNEL_SQDIST, X1, n1, X2, n2, D, ones, 1.0, 1.0, 0.0, out, ld, (cudaStream_t)stream);
}

extern "C" int ppbo_gram_regularized(int kind, const double* X, int n, int D, const double* lengthscales_h,
                                     double sigma_f, double shrinkage, double* out, long long ld, void* stream) {
    PPBO_REQUIRE(n >= 0 && ld >= n, "shape");
    PPBO_REQUIRE(shrinkage >= 0.0 && shrinkage < 1.0, "shrinkage in [0,1)");
    // (1-s) K + s (tr K / n) I with tr K / n = sigma_f^2 (stationary kernels, k(x,x) = sigma_f^2)
    return kernel_matrix_raw(kind, X, n, X, n, D, lengthscales_h, sigma_f, 1.0 - shrinkage,
                             shrinkage * sigma_f * sigma_f, out, ld, (cudaStream_t)stream);
}

/* Rows / columns [n_old, n_new) of the regularised covariance of X[0:n_new] in place (leading dimension ld >= n_new): the
 * leading n_old x n_old block is untouched -- the shrinkage is N-independent for these stationary kernels (SURVEY.md 7-8), so
 * Sigma_old is the leading principal block of Sigma_new.  One (m+1)-row block is appended per PPBO iteration
 * (src/feedback_processing.py:133-154, src/gp_model.py:157 rebuilds everything).  Bit-identical to ppbo_gram_regularized. */
extern "C" int ppbo_gram_append(int kind, const double* X, int n_old, int n_new, int D, const double* lengthscales_h,
                                double sigma_f, double shrinkage, double* out, long long ld, void* stream) {
    PPBO_REQUIRE(n_old >= 0 && n_new >= n_old && ld >= n_new, "shape");
    PPBO_REQUIRE(shrinkage >= 0.0 && shrinkage < 1.0, "shrinkage in [0,1)");
    if (n_new == n_old) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    // appended rows against all points: same per-entry arithmetic as the symmetric kernel (same shift point X[0], same scaling)
    int rc = kernel_matrix_raw(kind, X + (long long)n_old * D, n_new - n_old, X, n_new, D, lengthscales_h, sigma_f, 1.0 - shrinkage, 0.0,
                               out + (long long)n_old * ld, ld, st);
    if (rc) return rc;
    PPBO_CL gram_mirror_kernel<<<dim3(ceil_div(n_new, 256), n_new - n_old), 256, 0, st>>>(out, ld, n_old, n_new, 1.0 - shrinkage,
                                                                                             sigma_f * sigma_f, shrinkage * sigma_f * sigma_f);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_mu_pred_point(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f,
                                   const double* alpha, const double* x_h, double* mu_h, void* stream) {
    KernelParams p;
    int rc = fill_params(p, kind, D, lengthscales_h, sigma_f);
    if (rc) return rc;
    PPBO_REQUIRE(N >= 0 && x_h != nullptr && mu_h != nullptr, "arguments");
    if ((rc = g_point.init())) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    for (int d = 0; d < D; ++d) g_point.host[d] = x_h[d];
    double* out = g_point.dev + PPBO_MAX_D;
    switch (kind) {
        case PPBO_KERNEL_SE: PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_SE><<<1, 1024, 0, st>>>(X, N, p, alpha, g_point.dev, out); break;
        case PPBO_KERNEL_RQ: PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_RQ><<<1, 1024, 0, st>>>(X, N, p, alpha, g_point.dev, out); break;
        case PPBO_KERNEL_MATERN32:
            PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_MATERN32><<<1, 1024, 0, st>>>(X, N, p, alpha, g_point.dev, out);
            break;
        case PPBO_KERNEL_MATERN52:
            PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_MATERN52><<<1, 1024, 0, st>>>(X, N, p, alpha, g_point.dev, out);
            break;
        case PPBO_KERNEL_CAMPHOR: PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_CAMPHOR><<<1, 1024, 0, st>>>(X, N, p, alpha, g_point.dev, out); break;
        default: PPBO_REQUIRE(false, "kernel kind has no posterior-mean kernel");
    }
    PPBO_LAUNCH_CHECK();
    PPBO_CUDA_CHECK(cudaStreamSynchronize(st));
    *mu_h = g_point.host[PPBO_MAX_D];
    return PPBO_OK;
}

extern "C" int ppbo_mu_pred_points(int kind, const double* X, int N, int D, const double* lengthscales_h, double sigma_f,
                                    const double* alpha, const double* x_h, int B, double* mu_h, void* stream) {
    KernelParams p;
    int rc = fill_params(p, kind, D, lengthscales_h, sigma_f);
    if (rc) return rc;
    PPBO_REQUIRE(N >= 0 && B >= 0 && B <= PPBO_MAX_POINTS && (B == 0 || (x_h != nullptr && mu_h != nullptr)), "arguments");
    if (B == 0) return PPBO_OK;
    if ((rc = g_batch.init())) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    memcpy(g_batch.host, x_h, sizeof(double) * (size_t)B * D);
    double* out_h = g_batch.host + (size_t)PPBO_MAX_D * PPBO_MAX_POINTS;
    double* out = g_batch.dev + (size_t)PPBO_MAX_D * PPBO_MAX_POINTS;
    switch (kind) {
        case PPBO_KERNEL_SE: PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_SE><<<B, 1024, 0, st>>>(X, N, p, alpha, g_batch.dev, out); break;
        case PPBO_KERNEL_RQ: PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_RQ><<<B, 1024, 0, st>>>(X, N, p, alpha, g_batch.dev, out); break;
        case PPBO_KERNEL_MATERN32:
            PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_MATERN32><<<B, 1024, 0, st>>>(X, N, p, alpha, g_batch.dev, out);
            break;
        case PPBO_KERNEL_MATERN52:
            PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_MATERN52><<<B, 1024, 0, st>>>(X, N, p, alpha, g_batch.dev, out);
            break;
        case PPBO_KERNEL_CAMPHOR: PPBO_CL mu_pred_point_kernel<PPBO_KERNEL_CAMPHOR><<<B, 1024, 0, st>>>(X, N, p, alpha, g_batch.dev, out); break;
        default: PPBO_REQUIRE(false, "kernel kind has no posterior-mean kernel");
    }
    PPBO_LAUNCH_CHECK();
    PPBO_CUDA_CHECK(cudaStreamSynchronize(st));
    memcpy(mu_h, out_h, sizeof(double) * (size_t)B);
    return PPBO_OK;
}

extern "C" int ppbo_kernel_se_grad(const double* X1, int n1, const double* X2, int n2, int D,
                                   const double* lengthscales_h, double sigma_f, double* dK, long long ld,
                                   long long stride, void* stream) {
    KernelParams p;
    int rc = fill_params(p, PPBO_KERNEL_SE, D, lengthscales_h, sigma_f);
    if (rc) return rc;
    if (n1 <= 0 || n2 <= 0) return PPBO_OK;
    const long long total = (long long)n1 * n2;
    PPBO_CL se_grad_kernel<<<(unsigned)ceil_div_ll(total, 256), 256, 0, (cudaStream_t)stream>>>(X1, n1, X2, n2, p, dK, ld, stride);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_shrink_inplace(double* K, long long ld, int n, double shrinkage, double* scratch1, void* stream) {
    PPBO_REQUIRE(n >= 0 && ld >= n && scratch1 != nullptr, "shape");
    if (n == 0) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    PPBO_CL trace_kernel<<<1, 1024, 0, st>>>(K, ld, n, scratch1);
    PPBO_CL shrink_kernel<<<dim3(ceil_div(n, 256), n), 256, 0, st>>>(K, ld, n, shrinkage, scratch1);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

extern "C" int ppbo_diffspace_gram(const double* Sigma, long long lds, int Q, int m, double* G, long long ldg, void* stream) {
    PPBO_REQUIRE(Q >= 0 && m >= 1, "shape");
    return diffspace_gram(Sigma, lds, Q, m, G, ldg, (cudaStream_t)stream);
}
