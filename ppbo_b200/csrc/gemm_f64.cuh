// ppbo_b200 -- FP64 "NT" GEMM building block for sm_100a:  acc[M x N] = A[M x K] . B[N x K]^T
//
// Both operands are row-major with K contiguous, which is what every dense contraction on the PPBO
// hot path looks like once the data layout is chosen for it (DESIGN.md "GEMM shapes"):
//   * Cholesky panel / trailing update      L21 = A21 . inv(L11)^T ,  A22 -= L21 . L21^T
//   * blocked triangular solves             X[:,J] -= X[:,K] . L[J,K]^T
//   * RFF posterior sampling                Fs[S x P] = Omega[S x F] . PhiT[P x F]^T   (+ row max / arg-max)
//   * exact-GP sampling                     Xs[S x P] = Z[S x P] . Lfac[P x P]^T + mu  (+ row max)
//   * predictive covariance                 Sigma_p = K** - Yt[P x M] . Yt[P x M]^T
//
// Math pipe: FP64 tensor op `mma.sync.aligned.m8n8k4.f64` (SASS DMMA.8x8x4).  tcgen05 has no f64 kind, so
// the Blackwell UMMA/TMEM path does not apply to this arithmetic; measured on B200 the DMMA pipe peaks at
// 37.1 TFLOP/s (== the DFMA pipe, profiles/r01_fp64_peaks_ubench.txt) and cuBLAS DGEMM reaches 35.5.
// Data path: cp.async (LDGSTS) 16-byte copies into a 4-stage shared-memory ring, rows padded to
// BK+4 doubles so the 8-byte fragment loads of a half-warp hit 16 distinct bank pairs.
#pragma once
#include "common.cuh"

namespace ppbo {

struct GemmOperands {
    const double* A; long long lda; long long strideA;   // A: M x K, row-major, batch stride
    const double* B; long long ldb; long long strideB;   // B: N x K, row-major, batch stride
    int M, N, K;
    // optional two-level batching: batch entry z = zo * zinner + zi sits at zi * stride + zo * stride2 (zinner == 0: one level)
    int zinner = 0; long long strideA2 = 0, strideB2 = 0;
};

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

template <int BYTES>
__device__ __forceinline__ void cp_async_zfill(double* smem_dst, const double* gsrc, int src_bytes) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;\n" ::"r"(s), "l"(gsrc), "n"(BYTES), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

template <int BM_, int BN_, int WARPS_M_, int WARPS_N_, int STAGES_, int VEC_, int MINB_ = 1>
struct GemmCfg {
    static constexpr int MINB = MINB_;        // CTAs per SM the register allocation must allow
    static constexpr int BM = BM_, BN = BN_, BK = 16, LDS = BK + 4;
    static constexpr int WARPS_M = WARPS_M_, WARPS_N = WARPS_N_, STAGES = STAGES_, VEC = VEC_;
    static constexpr int THREADS = 32 * WARPS_M * WARPS_N;
    static constexpr int WM = BM / WARPS_M, WN = BN / WARPS_N;
    static constexpr int MI = WM / 8, NI = WN / 8;
    static constexpr int STAGE_DOUBLES = (BM + BN) * LDS;
    static constexpr int SMEM_BYTES = STAGES * STAGE_DOUBLES * 8;
    static_assert(WM % 8 == 0 && WN % 8 == 0, "warp tile must be a multiple of the 8x8 DMMA tile");
};

// one k-tile (BK columns) of A and B rows [row0, row0+ROWS) -> shared memory; out-of-range rows / k zero-filled
template <class Cfg, int ROWS>
__device__ __forceinline__ void load_rows(double* dst, const double* __restrict__ src, long long ld, int row0,
                                          int nrows, int k0, int K) {
    constexpr int CPR = Cfg::BK / Cfg::VEC;                 // chunks per row
    constexpr int CHUNKS = ROWS * CPR;
    constexpr int ITERS = (CHUNKS + Cfg::THREADS - 1) / Cfg::THREADS;
#pragma unroll
    for (int i = 0; i < ITERS; ++i) {
        const int c = threadIdx.x + i * Cfg::THREADS;
        if (CHUNKS % Cfg::THREADS != 0 && c >= CHUNKS) break;
        const int r = c / CPR, kc = (c % CPR) * Cfg::VEC;
        const int gr = row0 + r, gk = k0 + kc;
        int bytes = (gr < nrows) ? (K - gk) * 8 : 0;
        bytes = bytes < 0 ? 0 : (bytes > Cfg::VEC * 8 ? Cfg::VEC * 8 : bytes);
        const double* g = bytes > 0 ? src + (long long)gr * ld + gk : src;
        cp_async_zfill<Cfg::VEC * 8>(dst + r * Cfg::LDS + kc, g, bytes);
    }
}

// acc += A[m0:m0+BM, :] . B[n0:n0+BN, :]^T   (all threads of the CTA participate; smem ring is reused)
template <class Cfg>
__device__ __forceinline__ void gemm_mainloop(const GemmOperands& g, const double* __restrict__ A,
                                              const double* __restrict__ B, int m0, int n0, double* smem,
                                              double (&acc)[Cfg::MI][Cfg::NI][2]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm0 = (warp / Cfg::WARPS_N) * Cfg::WM, wn0 = (warp % Cfg::WARPS_N) * Cfg::WN;
    const int gq = lane >> 2, t4 = lane & 3;
    const int KT = (g.K + Cfg::BK - 1) / Cfg::BK;

    auto load_stage = [&](int slot, int kt) {
        double* As = smem + slot * Cfg::STAGE_DOUBLES;
        double* Bs = As + Cfg::BM * Cfg::LDS;
        load_rows<Cfg, Cfg::BM>(As, A, g.lda, m0, g.M, kt * Cfg::BK, g.K);
        load_rows<Cfg, Cfg::BN>(Bs, B, g.ldb, n0, g.N, kt * Cfg::BK, g.K);
    };
#pragma unroll
    for (int s = 0; s < Cfg::STAGES - 1; ++s) {
        if (s < KT) load_stage(s, s);
        cp_async_commit();
    }
    for (int kt = 0; kt < KT; ++kt) {
        cp_async_wait<Cfg::STAGES - 2>();
        __syncthreads();
        const int nk = kt + Cfg::STAGES - 1;
        if (nk < KT) load_stage(nk % Cfg::STAGES, nk);
        cp_async_commit();
        const double* As = smem + (kt % Cfg::STAGES) * Cfg::STAGE_DOUBLES + (wm0 + gq) * Cfg::LDS + t4;
        const double* Bs = smem + (kt % Cfg::STAGES) * Cfg::STAGE_DOUBLES + (Cfg::BM + wn0 + gq) * Cfg::LDS + t4;
#pragma unroll
        for (int k4 = 0; k4 < Cfg::BK / 4; ++k4) {
            double a[Cfg::MI], b[Cfg::NI];
#pragma unroll
            for (int mi = 0; mi < Cfg::MI; ++mi) a[mi] = As[mi * 8 * Cfg::LDS + k4 * 4];
#pragma unroll
            for (int ni = 0; ni < Cfg::NI; ++ni) b[ni] = Bs[ni * 8 * Cfg::LDS + k4 * 4];
#pragma unroll
            for (int mi = 0; mi < Cfg::MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < Cfg::NI; ++ni) dmma884(acc[mi][ni], a[mi], b[ni]);
        }
    }
    cp_async_wait<0>();
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------------
// Kernel 1: C = alpha * A.B^T + beta * C   (optionally only the lower-triangular tiles: SYRK-style)
struct StoreEpilogue {
    double* C; long long ldc; long long strideC;
    double alpha, beta;
    int lower_only;      // 1: blockIdx.x enumerates tiles (ti >= tj) of a square tiling (BM == BN); 2: the same in the tile
                         //    configuration the full product would use (its lower tiles bit-identical to the full product's)
    int vec_ok;          // 1: C rows are 16-byte aligned at even columns (set by the launcher)
    int in_place;        // 1: C aliases A (row-panel update); launcher picks a tile with BN >= N == K
    long long strideC2 = 0;   // outer batch stride (GemmOperands::zinner)
};

template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, Cfg::MINB) gemm_nt_store_kernel(GemmOperands g, StoreEpilogue ep) {
    extern __shared__ __align__(16) double smem[];
#ifdef PPBO_PDL
    // Programmatic dependent launch (an experiment on the Cholesky critical path, tuning key 7; measured slower and compiled out):
    // let the next kernel of the stream become resident now and hold this one until its predecessor has completed and flushed.
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
    int tm, tn;
    if (ep.lower_only) {
        // tiles that touch the lower triangle, row-tile major: row tile ti owns column tiles 0 .. R (ti + 1) - 1, R = BM / BN
        constexpr int R = (Cfg::BM >= Cfg::BN) ? Cfg::BM / Cfg::BN : 1;     // launchers only use lower_only with BM >= BN
        const long long L = blockIdx.x;
        int ti = (int)((sqrt(1.0 + 8.0 * (double)L / R) - 1.0) * 0.5);
        while ((long long)R * (ti + 1) * (ti + 2) / 2 <= L) ++ti;
        while ((long long)R * ti * (ti + 1) / 2 > L) --ti;
        tm = ti;
        tn = (int)(L - (long long)R * ti * (ti + 1) / 2);
    } else {
        tm = blockIdx.x;
        tn = blockIdx.y;
    }
    const int m0 = tm * Cfg::BM, n0 = tn * Cfg::BN;
    const long long zo = g.zinner ? blockIdx.z / g.zinner : 0, zi = g.zinner ? blockIdx.z % g.zinner : blockIdx.z;
    const double* A = g.A + zi * g.strideA + zo * g.strideA2;
    const double* B = g.B + zi * g.strideB + zo * g.strideB2;
    double* C = ep.C + zi * ep.strideC + zo * ep.strideC2;

    double acc[Cfg::MI][Cfg::NI][2];
#pragma unroll
    for (int mi = 0; mi < Cfg::MI; ++mi)
#pragma unroll
        for (int ni = 0; ni < Cfg::NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
    gemm_mainloop<Cfg>(g, A, B, m0, n0, smem, acc);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm0 = (warp / Cfg::WARPS_N) * Cfg::WM, wn0 = (warp % Cfg::WARPS_N) * Cfg::WN;
    const int gq = lane >> 2, t4 = lane & 3;
#pragma unroll
    for (int mi = 0; mi < Cfg::MI; ++mi) {
        const int row = m0 + wm0 + mi * 8 + gq;
        if (row >= g.M) continue;
        double* crow = C + (long long)row * ep.ldc;
#pragma unroll
        for (int ni = 0; ni < Cfg::NI; ++ni) {
            const int col = n0 + wn0 + ni * 8 + 2 * t4;
            if (col >= g.N) continue;
            double v0 = ep.alpha * acc[mi][ni][0], v1 = ep.alpha * acc[mi][ni][1];
            if (col + 1 < g.N && ep.vec_ok) {
                double2* p = reinterpret_cast<double2*>(crow + col);
                if (ep.beta != 0.0) {
                    const double2 old = *p;
                    v0 += ep.beta * old.x;
                    v1 += ep.beta * old.y;
                }
                *p = make_double2(v0, v1);
            } else {
                if (ep.beta != 0.0) v0 += ep.beta * crow[col];
                crow[col] = v0;
                if (col + 1 < g.N) {
                    if (ep.beta != 0.0) v1 += ep.beta * crow[col + 1];
                    crow[col + 1] = v1;
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Kernel 2: per-row max / first arg-max of (A.B^T + bias[n]) over ALL n, never materialising the S x P product.
// One CTA owns BM rows and walks the N tiles; batch index = blockIdx.y (one query direction per batch entry).
struct RowMaxEpilogue {
    const double* bias; long long strideBias;   // [N] per batch, may be null
    double* out_max; int* out_arg;              // [batch][M]
    double* out_full; long long ld_full; long long strideFull;   // optional dense S x P output (tests), may be null
    int batch, group_m;     // launch shape: 1-D grid over (row-tile group, batch entry, row tile in group), see the kernel
};

template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, Cfg::MINB) gemm_nt_rowmax_kernel(GemmOperands g, RowMaxEpilogue ep) {
    extern __shared__ __align__(16) double smem[];
    // CTA order: row tiles are taken in groups of group_m; inside a group all batch entries (query directions) are visited
    // before moving on, so the group's A rows (group_m x BM x K doubles, sized to sit in L2) are reused `batch` times from L2
    // and the B operand of one batch entry is shared by the ~SM-count CTAs running at the same time.
    const int tiles_m = (g.M + Cfg::BM - 1) / Cfg::BM;
    const int per_group = ep.group_m * ep.batch;
    const int grp = blockIdx.x / per_group, rem = blockIdx.x % per_group;
    const int rows_here = min(ep.group_m, tiles_m - grp * ep.group_m);
    const int bz = rem / rows_here;
    const int m0 = (grp * ep.group_m + rem % rows_here) * Cfg::BM;
    if (bz >= ep.batch) return;                  // tail of the last (smaller) group
    const double* A = g.A + (long long)bz * g.strideA;
    const double* B = g.B + (long long)bz * g.strideB;
    const double* bias = ep.bias ? ep.bias + (long long)bz * ep.strideBias : nullptr;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wmi = warp / Cfg::WARPS_N, wni = warp % Cfg::WARPS_N;
    const int wm0 = wmi * Cfg::WM, wn0 = wni * Cfg::WN;
    const int gq = lane >> 2, t4 = lane & 3;

    double best[Cfg::MI];
    int besti[Cfg::MI];
#pragma unroll
    for (int mi = 0; mi < Cfg::MI; ++mi) { best[mi] = -INFINITY; besti[mi] = 0x7fffffff; }

    const int NT = (g.N + Cfg::BN - 1) / Cfg::BN;
    for (int nt = 0; nt < NT; ++nt) {
        const int n0 = nt * Cfg::BN;
        double acc[Cfg::MI][Cfg::NI][2];
#pragma unroll
        for (int mi = 0; mi < Cfg::MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < Cfg::NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
        gemm_mainloop<Cfg>(g, A, B, m0, n0, smem, acc);
#pragma unroll
        for (int ni = 0; ni < Cfg::NI; ++ni) {
            const int col = n0 + wn0 + ni * 8 + 2 * t4;
            double b0 = 0.0, b1 = 0.0;
            if (bias) {
                if (col < g.N) b0 = bias[col];
                if (col + 1 < g.N) b1 = bias[col + 1];
            }
#pragma unroll
            for (int mi = 0; mi < Cfg::MI; ++mi) {
                const double v0 = acc[mi][ni][0] + b0, v1 = acc[mi][ni][1] + b1;
                if (col < g.N && v0 > best[mi]) { best[mi] = v0; besti[mi] = col; }       // columns visited in
                if (col + 1 < g.N && v1 > best[mi]) { best[mi] = v1; besti[mi] = col + 1; }  // increasing order
                if (ep.out_full) {
                    const int row = m0 + wm0 + mi * 8 + gq;
                    double* o = ep.out_full + (long long)bz * ep.strideFull + (long long)row * ep.ld_full;
                    if (row < g.M && col < g.N) o[col] = v0;
                    if (row < g.M && col + 1 < g.N) o[col + 1] = v1;
                }
            }
        }
    }
    // combine the 4 lanes that share a row, then the WARPS_N warps that share it (smallest index wins ties)
    double* red_v = smem;                                   // [WARPS_N][BM]
    int* red_i = reinterpret_cast<int*>(smem + Cfg::WARPS_N * Cfg::BM);
#pragma unroll
    for (int mi = 0; mi < Cfg::MI; ++mi) {
        double v = best[mi];
        int ix = besti[mi];
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, ix, o);
            if (ov > v || (ov == v && oi < ix)) { v = ov; ix = oi; }
        }
        if (t4 == 0) {
            red_v[wni * Cfg::BM + wm0 + mi * 8 + gq] = v;
            red_i[wni * Cfg::BM + wm0 + mi * 8 + gq] = ix;
        }
    }
    __syncthreads();
    for (int r = threadIdx.x; r < Cfg::BM; r += Cfg::THREADS) {
        const int row = m0 + r;
        if (row >= g.M) continue;
        double v = red_v[r];
        int ix = red_i[r];
#pragma unroll
        for (int w = 1; w < Cfg::WARPS_N; ++w) {
            const double ov = red_v[w * Cfg::BM + r];
            const int oi = red_i[w * Cfg::BM + r];
            if (ov > v || (ov == v && oi < ix)) { v = ov; ix = oi; }
        }
        ep.out_max[(long long)bz * g.M + row] = v;
        if (ep.out_arg) ep.out_arg[(long long)bz * g.M + row] = ix;
    }
}

// host-side launchers (linalg.cu)
int launch_gemm_nt(const GemmOperands& g, const StoreEpilogue& ep, int batch, cudaStream_t st);
int launch_gemm_nt_rowmax(const GemmOperands& g, const RowMaxEpilogue& ep, int batch, cudaStream_t st);

}  // namespace ppbo
