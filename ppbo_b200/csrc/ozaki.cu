// ppbo_b200 -- K3 on the 5th-generation tensor cores: the RFF sampling contraction  Fs = Omega[S x F] . PhiT[P x F]^T
// (batched form of the objective of Hsampler.return_xstar, src/random_fourier_sampler.py:166,170) evaluated to FP64 accuracy
// with INT8 tcgen05.mma and INT32 accumulators in TMEM (error-free splitting, "Ozaki scheme"), fused with the per-sample
// max / first arg-max over the grid.
//
// tcgen05 has no f64 kind; the FP64 DMMA pipe of sm_100a peaks at 37 TFLOP/s, the INT8 tensor pipe at ~4.5 POP/s.  Every row
// of an operand is scaled by a power of two (|x| 2^-e < 1/4), rounded once to a fixed-point integer of 8 KS bits and cut into
// KS balanced base-256 digits d_0..d_{KS-1} in [-128, 127]:
//
//      x  ~=  2^e * sum_i d_i 256^-(i+1)                                   (exact when the row's dynamic range fits 8 KS - 2 bits)
//
// The digit planes are INT8 matrices; products of digit planes are exact in INT32 (|sum| <= KS * Kpad * 2^14 < 2^31), so
//
//      C[r][c] = 2^(ea_r + eb_c) * sum_{d < KS} 256^-(d+2) * acc_d[r][c],    acc_d = sum_{i+j=d} A_i . B_j^T     (exact integers)
//
// drops only the digit pairs with i + j >= KS (relative weight 256^-KS against |row|_max |col|_max).  KS (KS+1)/2 INT8 GEMMs
// replace one FP64 GEMM; the result is a deterministic function of the inputs (no dependence on tile shape, launch shape or
// rank), which the oracle reproduces bit for bit with integer arithmetic (oracle/ppbo_oracle.py ozaki_*).
//
// Kernel structure (one persistent CTA per SM, 320 threads):
//   warp 0      producer: one cp.async.bulk per operand and k-block (the digit planes are stored in HBM already in the
//               shared-memory image the tensor core reads, see slice layout below) -> 3-stage mbarrier ring
//   warp 1      one elected lane issues tcgen05.mma.kind::i8 (M=128, N=BN, K=32): KS accumulators of BN columns in TMEM
//   warps 2..9  epilogue: tcgen05.ld the KS INT32 accumulators, recombine in INT64 -> FP64, scale, running row max/arg-max.
//               Two warps per TMEM lane quarter, each takes one half of the tile's columns: the accumulators are single-buffered
//               (KS BN = 384 of 512 TMEM columns), so the epilogue is exposed and its length, not its throughput, is what counts
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <mutex>

#include "../../include/ppbo_b200.h"
#include "common.cuh"
#include "philox.cuh"

namespace ppbo {
extern int g_tuning[16];
namespace oz {

constexpr int BM = 128;                      // rows of the A tile = TMEM lanes
constexpr int KB = 64;                       // bytes of K per pipeline stage and digit plane
constexpr int UMMA_K = 32;                   // K of one tcgen05.mma.kind::i8
constexpr int LBO = 128;                     // byte distance of K-adjacent 8 x 16 B core matrices
constexpr int SBO = (KB / 16) * 128;         // byte distance of 8-row groups
constexpr int MAX_KS = 7;
constexpr int EPI_WARPS = 8;                 // two per TMEM lane quarter (warp w may only read lanes 32 (w & 3) ..)
constexpr int THREADS = 64 + 32 * EPI_WARPS; // producer warp + MMA warp + epilogue warps
constexpr int MERGE_BYTES = 2 * BM * 12;     // (max, arg) of the upper column half, double-buffered over work items

// Slice layout in HBM for an operand of `batch` matrices with rows padded to tiles of TR rows and K padded to KBLK blocks of
// KB bytes:  plane(b, rt, kb, s) is a contiguous TR x KB byte block at  ((((b NT + rt) KBLK + kb) KS + s) TR KB, stored in the
// canonical no-swizzle K-major core-matrix order of the UMMA shared-memory descriptor:
__host__ __device__ inline int tile_offset(int rr, int kk) { return (rr >> 3) * SBO + (kk >> 4) * LBO + (rr & 7) * 16 + (kk & 15); }

// ------------------------------------------------------------------------------------------------ slicing
// scale[b][r] = 2^(E+2) with max_k |x[r][k]| = m 2^E, m in [1/2, 1)   (1 for an all-zero or padding row; NaN if not finite)
__global__ void __launch_bounds__(256) ozaki_rowscale_kernel(const double* __restrict__ X, long long ldx, long long strideX,
                                                             int rows, int rows_pad, int K, double* __restrict__ scale) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + warp, b = blockIdx.y;
    if (r >= rows_pad) return;
    double amax = 0.0;
    if (r < rows) {
        const double* x = X + (long long)b * strideX + (long long)r * ldx;
        for (int k = lane; k < K; k += 32) {
            const double v = fabs(x[k]);
            amax = (v > amax || v != v) ? v : amax;                 // NaN sticks
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double w = __shfl_xor_sync(0xffffffffu, amax, o);
            amax = (w > amax || w != w) ? w : amax;
        }
    }
    if (lane == 0) {
        double s = 1.0;
        if (amax != amax || amax > 1.7e308) s = nan("");
        else if (amax > 0.0) {
            int e;
            frexp(amax, &e);
            s = ldexp(1.0, e + 2);
        }
        scale[(long long)b * rows_pad + r] = s;
    }
}

// One warp = 8 rows x 4 sixteen-byte chunks = one (row group, k-block): its KS stores are 512 contiguous bytes each.
template <int KS>
__global__ void __launch_bounds__(256) ozaki_slice_kernel(const double* __restrict__ X, long long ldx, long long strideX,
                                                          int rows, int rows_pad, int K, int KBLK, int TR,
                                                          const double* __restrict__ scale, int8_t* __restrict__ out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rg = blockIdx.x, b = blockIdx.y;               // row group of 8 rows
    const int rr8 = lane & 7, c = lane >> 3;
    const int r = rg * 8 + rr8;                              // row inside the batch entry (padded)
    const int rt = r / TR, rr = r % TR;
    const int NT = rows_pad / TR;
    const double sc = scale[(long long)b * rows_pad + r];
    const double mult = ldexp(1.0 / sc, 8 * KS);             // exact: power of two
    const double* x = X + (long long)b * strideX + (long long)r * ldx;
    for (int kb = blockIdx.z * 8 + warp; kb < KBLK; kb += gridDim.z * 8) {
        const int k0 = kb * KB + c * 16;
        uint32_t w[KS][4];
#pragma unroll
        for (int s = 0; s < KS; ++s)
#pragma unroll
            for (int q = 0; q < 4; ++q) w[s][q] = 0u;
        if (r < rows) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const int k = k0 + e;
                const double v = (k < K) ? x[k] : 0.0;
                long long Y = __double2ll_rn(v * mult);      // |Y| < 2^(8 KS - 2)
#pragma unroll
                for (int s = KS - 1; s >= 0; --s) {
                    const long long d = ((Y + 128) & 255) - 128;          // balanced digit in [-128, 127]
                    Y = (Y - d) >> 8;
                    w[s][e >> 2] |= (uint32_t)((uint8_t)(int8_t)d) << (8 * (e & 3));
                }
            }
        }
        int8_t* base = out + ((((long long)b * NT + rt) * KBLK + kb) * KS) * ((long long)TR * KB) + tile_offset(rr, c * 16);
#pragma unroll
        for (int s = 0; s < KS; ++s)
            *reinterpret_cast<uint4*>(base + (long long)s * TR * KB) = make_uint4(w[s][0], w[s][1], w[s][2], w[s][3]);
    }
}

// Posterior weight draws straight into digit planes: Omega[s][f] = omega_map[f] + z[s][f] / sqrt(-hess_diag[f]) (sample_omega_kernel,
// acq.cu; z = normal number (sample0 + s) F + f of the Philox stream) is generated into shared memory (one warp per row, 8 rows per
// CTA), its row scale is taken there, and the planes are cut from shared memory exactly as ozaki_slice_kernel does from HBM.  The
// S x F matrix of draws (262 MB at S = 32768, F = 1000) never exists: 8 B written + 16 B read per element become 0.
// Bit-identical to sample_omega_kernel -> ozaki_rowscale_kernel -> ozaki_slice_kernel (same expressions, same rounding).
// RAW: the planes of z itself (no omega_map / hess_diag applied): the draws of the full-covariance contraction, whose covariance
// sits in the grid operand instead (ppbo_ozaki_normal_slice); bit-identical to ppbo_normal_fill -> ppbo_ozaki_slice.
template <int KS, bool RAW = false>
__global__ void __launch_bounds__(256) ozaki_sample_slice_kernel(const double* __restrict__ omega_map, const double* __restrict__ hess_diag,
                                                                 unsigned long long seed, uint32_t stream_id, long long sample0, int S,
                                                                 int rows_pad, int F, int KBLK, double* __restrict__ scale,
                                                                 int8_t* __restrict__ out) {
    extern __shared__ double xs[];                           // [8][KBLK * KB] draws of this row group, zero-padded in K
    __shared__ double sc_s[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rg = blockIdx.x, Kp = KBLK * KB;
    {   // ---- phase 1: warp w draws row rg * 8 + w
        const int r = rg * 8 + warp;
        double* x = xs + warp * Kp;
        double amax = 0.0;
        for (int k = F + lane; k < Kp; k += 32) x[k] = 0.0;
        if (r < S) {
            for (int fp = lane; 2 * fp < F; fp += 32) {
                const int f0 = 2 * fp;
                double z0, z1 = 0.0;
                const long long e = (sample0 + r) * (long long)F + f0;   // global normal index of (r, f0)
                if ((e & 1) == 0) {
                    philox_normal2(seed, (unsigned long long)(e >> 1), stream_id, z0, z1);
                } else {                                                  // odd F: the pair straddles two counters
                    double a, b;
                    philox_normal2(seed, (unsigned long long)(e >> 1), stream_id, a, b);
                    z0 = b;
                    philox_normal2(seed, (unsigned long long)((e + 1) >> 1), stream_id, a, b);
                    z1 = a;
                }
                const double v0 = RAW ? z0 : omega_map[f0] + z0 * rsqrt(-hess_diag[f0]);
                x[f0] = v0;
                double v = fabs(v0);
                amax = (v > amax || v != v) ? v : amax;
                if (f0 + 1 < F) {
                    const double v1 = RAW ? z1 : omega_map[f0 + 1] + z1 * rsqrt(-hess_diag[f0 + 1]);
                    x[f0 + 1] = v1;
                    v = fabs(v1);
                    amax = (v > amax || v != v) ? v : amax;
                }
            }
        } else {
            for (int k = lane; k < F; k += 32) x[k] = 0.0;
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double w = __shfl_xor_sync(0xffffffffu, amax, o);
            amax = (w > amax || w != w) ? w : amax;
        }
        if (lane == 0) {
            double s = 1.0;
            if (amax != amax || amax > 1.7e308) s = nan("");
            else if (amax > 0.0) {
                int ex;
                frexp(amax, &ex);
                s = ldexp(1.0, ex + 2);
            }
            sc_s[warp] = s;
            scale[r] = s;
        }
    }
    __syncthreads();
    // ---- phase 2: one warp = 8 rows x 4 sixteen-byte chunks = one k-block (ozaki_slice_kernel)
    const int rr8 = lane & 7, c = lane >> 3;
    const int r = rg * 8 + rr8;
    const int rt = r / BM, rr = r % BM;
    const double mult = ldexp(1.0 / sc_s[rr8], 8 * KS);
    const double* x = xs + rr8 * Kp;
    for (int kb = warp; kb < KBLK; kb += 8) {
        const int k0 = kb * KB + c * 16;
        uint32_t w[KS][4];
#pragma unroll
        for (int s = 0; s < KS; ++s)
#pragma unroll
            for (int q = 0; q < 4; ++q) w[s][q] = 0u;
        if (r < S) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                long long Y = __double2ll_rn(x[k0 + e] * mult);
#pragma unroll
                for (int s = KS - 1; s >= 0; --s) {
                    const long long d = ((Y + 128) & 255) - 128;
                    Y = (Y - d) >> 8;
                    w[s][e >> 2] |= (uint32_t)((uint8_t)(int8_t)d) << (8 * (e & 3));
                }
            }
        }
        int8_t* base = out + (((long long)rt * KBLK + kb) * KS) * ((long long)BM * KB) + tile_offset(rr, c * 16);
#pragma unroll
        for (int s = 0; s < KS; ++s)
            *reinterpret_cast<uint4*>(base + (long long)s * BM * KB) = make_uint4(w[s][0], w[s][1], w[s][2], w[s][3]);
    }
}

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// A lost arrival must not hang the GPU box: after ~2 s of spinning the kernel records which wait starved and traps.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* err, int code) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            if (err) atomicExch(err, code);
            __threadfence_system();
            __trap();
        }
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, INT8 x INT8 -> INT32
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand from TMEM (lane = row, 32-bit column = 4 consecutive K bytes)
__device__ __forceinline__ void tc_mma_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// shared memory (128 rows x 32 B in core-matrix order) -> TMEM (128 lanes x 8 columns); ordered with tcgen05.mma in the pipe
__device__ __forceinline__ void tc_cp_128x256b(uint32_t taddr, uint64_t sdesc) {
    asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(taddr), "l"(sdesc) : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns: thread t of the warp receives columns [col, col+16) of TMEM lane (lane_base + t)
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major, no swizzle (PTX ISA "matrix descriptor"; CUTLASS cute/arch/mma_sm100_desc.hpp):
// [0,14) address >> 4, [16,30) leading byte offset >> 4, [32,46) stride byte offset >> 4, [46,48) version = 1, [61,64) layout 0
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(LBO >> 4) << 16) | ((uint64_t)(SBO >> 4) << 32) | (1ull << 46);
}
// The same descriptor `bytes` further into the buffer (bytes % 16 == 0): one 32-bit add on the low word, so the issuing thread
// does not re-derive the address field for every MMA (a dependent shift/mask/or chain per instruction otherwise).
__device__ __forceinline__ uint64_t umma_desc_advance(uint64_t desc, uint32_t bytes) {
    return (desc & 0xFFFFFFFF00000000ull) | (uint64_t)((uint32_t)desc + (bytes >> 4));
}

// Both operands are read from shared memory.  Copying the A digit planes of a stage into TMEM (tcgen05.cp) so that only the
// narrow B planes are re-read was measured slower (13.0 ms against 9.8): the copies serialise with the MMAs in the tensor pipe.
template <int KS, int BN>
struct Cfg {
    static constexpr int A_PLANE = BM * KB, B_PLANE = BN * KB;
    static constexpr int A_STAGE = KS * A_PLANE, B_STAGE = KS * B_PLANE;
    static constexpr int STAGE_BYTES = A_STAGE + B_STAGE;
    static constexpr int STAGES = (3 * STAGE_BYTES + 256 + MERGE_BYTES <= 232448) ? 3 : 2;
    static constexpr int TMEM_USED = KS * BN;
    static constexpr int TMEM_COLS = TMEM_USED <= 32 ? 32 : TMEM_USED <= 64 ? 64 : TMEM_USED <= 128 ? 128 : TMEM_USED <= 256 ? 256 : 512;
    static constexpr int SMEM = STAGES * STAGE_BYTES + 256 + MERGE_BYTES;
    static constexpr int G1 = KS < 3 ? KS : 3;               // accumulators recombined into the high INT64 word
    // instruction descriptor (cute::UMMA::InstrDescriptor): c_format S32 = 2 @4, a/b format INT8 = 1 @7/@10, K-major A and B,
    // N >> 3 @17, M >> 4 @24
    static constexpr uint32_t IDESC_BASE = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BM >> 4) << 24);
    static_assert(TMEM_USED <= 512, "accumulators exceed TMEM");
    static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "UMMA N");
    static_assert(SMEM <= 232448, "shared memory");
};

struct Params {
    const int8_t* A; const double* ascale; int S, MT;          // MT row tiles of BM samples
    const int8_t* B; const double* bscale; int P, NT, batch;   // NT column tiles of BN grid points per batch entry
    int KBLK;
    int NG, ntg;                                               // column tiles are taken in NG groups of ntg tiles: one work item each
    int GB;                                                    // grids are visited in blocks of GB (work order, see decode_item)
    double* fmax; int* arg;                                    // [batch][S] (NG == 1) or partial results [batch][NG][S]
    double* full; long long ld_full, stride_full;              // optional dense output (tests)
    int* err;
};
// The biased instantiations take the offsets in a derived parameter block: a field added to Params itself changes the code ptxas
// emits for the unbiased kernels (same arithmetic, other registers and layout).
// (bias at offset 128 rather than right behind Params at 120: there ptxas spills 12 bytes in the KS = 7 kernel)
struct BiasParams : Params {
    alignas(16) const double* bias;                            // [batch][P] column offsets
};
template <bool BIAS> struct ParamsOf { using T = Params; };
template <> struct ParamsOf<true> { using T = BiasParams; };
__device__ __forceinline__ const double* bias_row(const Params&, int, int) { return nullptr; }
__device__ __forceinline__ const double* bias_row(const BiasParams& p, int b, int P) { return p.bias + (long long)b * P; }

// Work order.  item -> (grid b, row tile mt, column-tile group ng):  grids in blocks of GB; inside a block the row tiles; inside a
// row tile the GB grids of the block; inside a grid the NG column groups (fastest).  The ~SM-count items in flight then cover
// SMs / (GB NG) row tiles (their A planes, KBLK x A_STAGE = 768 KB each at F = 1000, are read from DRAM once per grid BLOCK and from
// L2 by the GB NG items that share them) and the B planes of GB grids (GB x 6.3 MB, L2-resident for the whole block).  With the
// earlier order (grid outermost) every grid re-streamed all A planes from DRAM: 4.5 GB of DRAM reads per launch at B = 20 against
// 0.33 GB of planes (profiles/r01_ncu_ozaki_rowmax.txt).
__device__ __forceinline__ void decode_item(const Params& p, int item, int& b, int& mt, int& ng) {
    const int per_grid_row = p.NG, full = p.batch / p.GB, rem = p.batch - full * p.GB;
    const int block_items = p.GB * p.MT * per_grid_row, items_full = full * block_items;
    int gb, nb_, r;
    if (item < items_full) { gb = item / block_items; r = item - gb * block_items; nb_ = p.GB; }
    else { gb = full; r = item - items_full; nb_ = rem; }
    mt = r / (nb_ * per_grid_row);
    const int r2 = r - mt * nb_ * per_grid_row;
    const int bl = r2 / per_grid_row;
    ng = r2 - bl * per_grid_row;
    b = gb * p.GB + bl;
}

// 16 columns of one row: recombine the KS INT32 accumulators into two exact INT64 words (hi: diagonals < G1, lo: the rest),
// convert, add with ONE rounding, scale by the column's power of two and update the running max / first arg-max.
// v = (hi + lo 2^-8(KS-G1)) * bs;  the common factor 2^-8(G1+1) and the row scale are applied once per row by the caller.
// For KS <= 6 both words stay below 2^44 and are converted by adding them to the bit pattern of 2^52 + 2^51 (exact; the
// INT64 -> FP64 convert instruction is a quarter-rate op and was a third of the epilogue's issue slots).
// BIAS: every element gets its column's offset, e = fma(v, as2, brow[col]) (one rounding: v as2 is exact, a power-of-two scale), so
// the row scale is applied per element and the max runs over e; without it the scale is applied once per row after the max.
template <int KS, int G1, bool CHECKED, int NC, bool BIAS = false>
__device__ __forceinline__ void epi_columns(const uint32_t (&acc)[KS][NC], const double* __restrict__ bs, int col0, int P,
                                            double* __restrict__ full_row, double as2, double& best, int& best_arg,
                                            const double* __restrict__ brow = nullptr) {
    constexpr long long MAGIC = 0x4338000000000000LL;             // bits of 2^52 + 2^51
    const double magic_d = 6755399441055744.0, lo_w = 1.0 / (double)(1ull << (8 * (KS - G1)));
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        long long hi = (KS <= 6) ? MAGIC : 0, lo = hi;
#pragma unroll
        for (int d = 0; d < G1; ++d) hi += (long long)(int)acc[d][c] << (8 * (G1 - 1 - d));
#pragma unroll
        for (int d = G1; d < KS; ++d) lo += (long long)(int)acc[d][c] << (8 * (KS - 1 - d));
        double hd, ld;
        if (KS <= 6) {
            hd = __longlong_as_double(hi) - magic_d;
            ld = __longlong_as_double(lo) - magic_d;
        } else {
            hd = (double)hi;
            ld = (double)lo;
        }
        const double v = fma(ld, lo_w, hd) * __ldg(bs + c);
        const int col = col0 + c;
        if (CHECKED) {
            if (col < P) {
                const double e = BIAS ? fma(v, as2, __ldg(brow + col)) : v;
                if (full_row) full_row[col] = BIAS ? e : v * as2;
                if (e > best) { best = e; best_arg = col; }
            }
        } else {
            const double e = BIAS ? fma(v, as2, __ldg(brow + col)) : v;
            if (e > best) {
                best = e;
                best_arg = col;
            }
        }
    }
}

template <int KS, int BN, bool BIAS = false>
__global__ void __launch_bounds__(THREADS, 1) ozaki_rowmax_kernel(const typename ParamsOf<BIAS>::T p) {
    using C = Cfg<KS, BN>;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + C::STAGES;
    uint64_t* tfull_bar = bars + 2 * C::STAGES;
    uint64_t* tempty_bar = tfull_bar + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 1);
    double* merge_best = reinterpret_cast<double*>(smem + C::STAGES * C::STAGE_BYTES + 256);       // [2][BM]
    int* merge_arg = reinterpret_cast<int*>(merge_best + 2 * BM);                                   // [2][BM]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < C::STAGES; ++s) {
            mbar_init(full_bar + s, 1);
            mbar_init(empty_bar + s, 1);
        }
        mbar_init(tfull_bar, 1);
        mbar_init(tempty_bar, EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)C::TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Work item = (grid b, row tile mt, column-tile group ng), ng fastest: the ~SM-count items in flight cover only
    // SMs / NG row tiles, so their A planes (KBLK x A_STAGE = 768 KB per row tile at F = 1000) stay L2-resident while the NG
    // CTAs of a row tile and the ntg column tiles of each CTA re-read them.  With NG = 1 every CTA streams its own row tile 16
    // times: 113 MB of live A planes thrash the L2 (ncu: 62 GB of DRAM reads per launch, 12 % L2 hit rate).
    const int items = p.MT * p.batch * p.NG;

    if (warp == 0) {
        // ------------------------------------------------------------------------------------- producer
        uint32_t stage = 0, phase = 0;
        for (int item = blockIdx.x; item < items; item += gridDim.x) {
            int ng, mt, b;
            decode_item(p, item, b, mt, ng);
            const int nt0 = ng * p.ntg, nt1 = min(p.NT, nt0 + p.ntg);
            const int8_t* Ab = p.A + (long long)mt * p.KBLK * C::A_STAGE;
            for (int nt = nt0; nt < nt1; ++nt) {
                const int8_t* Bb = p.B + ((long long)b * p.NT + nt) * p.KBLK * C::B_STAGE;
                for (int kb = 0; kb < p.KBLK; ++kb) {
                    mbar_wait(empty_bar + stage, phase ^ 1, p.err, 1);
                    if (lane == 0) {
                        const uint32_t dst = smem_u32(smem + stage * C::STAGE_BYTES);
                        mbar_expect_tx(full_bar + stage, C::STAGE_BYTES);
                        bulk_g2s(dst, Ab + (long long)kb * C::A_STAGE, C::A_STAGE, full_bar + stage);
                        bulk_g2s(dst + C::A_STAGE, Bb + (long long)kb * C::B_STAGE, C::B_STAGE, full_bar + stage);
                    }
                    __syncwarp();
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------------------------- MMA issuer
        uint32_t stage = 0, phase = 0, tile = 0;
        for (int item = blockIdx.x; item < items; item += gridDim.x) {
            int ng, mt, b;
            decode_item(p, item, b, mt, ng);
            const int nt0 = ng * p.ntg, nt1 = min(p.NT, nt0 + p.ntg);
            for (int nt = nt0; nt < nt1; ++nt, ++tile) {
                mbar_wait(tempty_bar, (tile & 1) ^ 1, p.err, 2);         // epilogue has drained the accumulators
                tc_fence_after();
                for (int kb = 0; kb < p.KBLK; ++kb) {
                    mbar_wait(full_bar + stage, phase, p.err, 3);
                    tc_fence_after();
                    if (lane == 0) {
                        const uint64_t a_desc0 = umma_desc(smem_u32(smem + stage * C::STAGE_BYTES));
                        const uint64_t b_desc0 = umma_desc_advance(a_desc0, C::A_STAGE);
                        // Digit plane A_i meets B_0 .. B_{KS-1-i}; those B planes are consecutive 8-row groups of one tall
                        // K-major matrix in shared memory and their accumulators d = i .. KS-1 are consecutive TMEM columns, so
                        // the KS - i products are ONE MMA of N = (KS - i) BN columns (cut into <= 256-column pieces).  A single
                        // thread cannot issue N = 64 MMAs fast enough to fill the pipe (measured ~57 clk per instruction
                        // against a 32 clk execution slot); wide instructions also read A once per (KS - i) BN columns.
#pragma unroll
                        for (int kk = 0; kk < KB / UMMA_K; ++kk) {
#pragma unroll
                            for (int i = 0; i < KS; ++i) {
                                const uint64_t adesc = umma_desc_advance(a_desc0, i * C::A_PLANE + kk * (UMMA_K / 16) * LBO);
                                const int ncols = (KS - i) * BN;
                                const int pieces = (ncols + 255) / 256;
                                const int width = ((ncols + pieces - 1) / pieces + 15) / 16 * 16;
#pragma unroll
                                for (int c0 = 0; c0 < ncols; c0 += width) {
                                    const int n = (ncols - c0 < width) ? ncols - c0 : width;
                                    const uint64_t bdesc = umma_desc_advance(b_desc0, c0 * KB + kk * (UMMA_K / 16) * LBO);
                                    const uint32_t d_tmem = tmem_base + (uint32_t)(i * BN + c0);
                                    const uint32_t accum = (uint32_t)((kb | kk | i) != 0);
                                    const uint32_t idesc = C::IDESC_BASE | ((uint32_t)(n >> 3) << 17);
                                    tc_mma_i8(d_tmem, adesc, bdesc, idesc, accum);
                                }
                            }
                        }
                        tc_commit(empty_bar + stage);                    // frees the stage when these MMAs have read it
                        if (kb == p.KBLK - 1) tc_commit(tfull_bar);      // accumulators complete
                    }
                    __syncwarp();
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else {
        // ------------------------------------------------------------------------------------- epilogue
        const int q = warp & 3;                                          // TMEM lane quarter this warp may read
        const int half = (warp - 2) >> 2;                                // which half of the tile's columns (warps 2..5: 0, 6..9: 1)
        constexpr int HC = BN / 2;                                       // columns per epilogue warp and tile
        const int cbase = half * HC;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        const double c_hi = ldexp(1.0, -8 * (C::G1 + 1));
        uint32_t tile = 0, nitem = 0;
        for (int item = blockIdx.x; item < items; item += gridDim.x, ++nitem) {
            int ng, mt, b;
            decode_item(p, item, b, mt, ng);
            const int nt0 = ng * p.ntg, nt1 = min(p.NT, nt0 + p.ntg);
            const int row = mt * BM + q * 32 + lane;
            const double as2 = ((row < p.S) ? p.ascale[row] : 1.0) * c_hi;     // row scale and the weight of the high word
            const double* brow = bias_row(p, b, p.P);
            double best = -INFINITY;
            int best_arg = 0;
            for (int nt = nt0; nt < nt1; ++nt, ++tile) {
                const double* bs = p.bscale + ((long long)b * p.NT + nt) * BN + cbase;
                mbar_wait(tfull_bar, tile & 1, p.err, 4);
                tc_fence_after();
                const bool checked = p.full != nullptr || (nt + 1) * BN > p.P;     // partial tile or dense output wanted
                double* full_row = (p.full && row < p.S) ? p.full + (long long)b * p.stride_full + (long long)row * p.ld_full : nullptr;
                // 8-column chunks, double-buffered in registers: the TMEM loads of chunk k+1 are in flight while chunk k is
                // recombined (tcgen05.wait::ld waits for every outstanding load, so the wait sits right before the next issue)
                uint32_t acc[2][KS][8];
#pragma unroll
                for (int d = 0; d < KS; ++d) tc_ld8(lane_addr + (uint32_t)(d * BN + cbase), acc[0][d]);
#pragma unroll
                for (int k = 0; k < HC / 8; ++k) {
                    tc_ld_wait();
                    if (k + 1 < HC / 8) {
#pragma unroll
                        for (int d = 0; d < KS; ++d) tc_ld8(lane_addr + (uint32_t)(d * BN + cbase + (k + 1) * 8), acc[(k + 1) & 1][d]);
                    }
                    const int col0 = nt * BN + cbase + k * 8;
                    if (checked) epi_columns<KS, C::G1, true, 8, BIAS>(acc[k & 1], bs + k * 8, col0, p.P, full_row, as2, best, best_arg, brow);
                    else epi_columns<KS, C::G1, false, 8, BIAS>(acc[k & 1], bs + k * 8, col0, p.P, nullptr, as2, best, best_arg, brow);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar);
            }
            // the two column halves of a row meet in shared memory (slot alternates with the work item: the next write to a slot
            // is two items later, behind the next item's barrier); equal maxima keep the lower column = first arg-max
            double* mb = merge_best + (nitem & 1) * BM;
            int* ma = merge_arg + (nitem & 1) * BM;
            if (half == 1) {
                mb[q * 32 + lane] = best;
                ma[q * 32 + lane] = best_arg;
            }
            asm volatile("bar.sync 1, %0;" ::"r"(32 * EPI_WARPS) : "memory");
            if (half == 0) {
                const double v1 = mb[q * 32 + lane];
                const int a1 = ma[q * 32 + lane];
                if (v1 > best || (v1 == best && a1 < best_arg)) { best = v1; best_arg = a1; }
                if (row < p.S) {
                    p.fmax[((long long)b * p.NG + ng) * p.S + row] = BIAS ? best : best * as2;
                    p.arg[((long long)b * p.NG + ng) * p.S + row] = best_arg;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS) : "memory");
    }
}

// per-sample max over the NG column-tile groups, lowest column index on ties (groups ascend in column index)
__global__ void __launch_bounds__(256) ozaki_merge_kernel(const double* __restrict__ pmax, const int* __restrict__ parg, int NG,
                                                          int S, double* __restrict__ fmax, int* __restrict__ arg) {
    const int s = blockIdx.x * 256 + threadIdx.x, b = blockIdx.y;
    if (s >= S) return;
    double best = -INFINITY;
    int ba = 0;
    for (int g = 0; g < NG; ++g) {
        const double v = pmax[((long long)b * NG + g) * S + s];
        if (v > best) { best = v; ba = parg[((long long)b * NG + g) * S + s]; }
    }
    fmax[(long long)b * S + s] = best;
    arg[(long long)b * S + s] = ba;
}

// ------------------------------------------------------------------------------------------------ host side
constexpr int BN_DEFAULT = 64;
// Number of column-tile groups: the fewest for which the A planes of the row tiles in flight (SMs / NG of them, KBLK x KS x 8 KB
// each) fit in about half of the 126 MB L2 (measured at F = 1000, 6 planes: NG = 1 12.1 ms, 2 9.2 ms, 4 9.8 ms, 8 10.3 ms).
static int column_groups(int NT, int KBLK, int KS) {
    int want = g_tuning[4];                                   // tuning key 4 overrides
    if (want <= 0) {
        const long long tile_bytes = (long long)KBLK * KS * BM * KB;
        want = (int)ceil_div_ll((long long)PPBO_SM_COUNT * tile_bytes, 64LL << 20);
    }
    want = want < 1 ? 1 : (want > NT ? NT : want);
    const int ntg = ceil_div(NT, want);
    return ceil_div(NT, ntg);
}

struct Shape {
    int rows_pad, KBLK;
    long long plane_bytes, scale_doubles;
};
static Shape shape_of(int rows, int K, int TR, int batch, int KS) {
    Shape s;
    s.rows_pad = ceil_div(rows, TR) * TR;
    s.KBLK = ceil_div(K, KB);
    s.plane_bytes = (long long)batch * s.rows_pad * s.KBLK * KB * KS;
    s.scale_doubles = (long long)batch * s.rows_pad;
    return s;
}

template <int KS>
static int slice_launch(const double* X, long long ldx, long long strideX, int rows, int K, int TR, int batch, double* scale,
                        int8_t* planes, cudaStream_t st) {
    const Shape s = shape_of(rows, K, TR, batch, KS);
    dim3 g1(s.rows_pad / 8, batch);
    PPBO_CL ozaki_rowscale_kernel<<<g1, 256, 0, st>>>(X, ldx, strideX, rows, s.rows_pad, K, scale);
    dim3 g2(s.rows_pad / 8, batch, min(8, ceil_div(s.KBLK, 8)));
    PPBO_CL ozaki_slice_kernel<KS><<<g2, 256, 0, st>>>(X, ldx, strideX, rows, s.rows_pad, K, s.KBLK, TR, scale, planes);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

template <int KS, int BN, bool BIAS = false>
static int rowmax_launch(const typename ParamsOf<BIAS>::T& p, cudaStream_t st) {
    using C = Cfg<KS, BN>;
    static std::once_flag once;
    static cudaError_t err = cudaSuccess;
    std::call_once(once, [] {
        err = cudaFuncSetAttribute(ozaki_rowmax_kernel<KS, BN, BIAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM);
    });
    PPBO_CUDA_CHECK(err);
    int dev = 0, sms = PPBO_SM_COUNT;
    PPBO_CUDA_CHECK(cudaGetDevice(&dev));
    PPBO_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int items = p.MT * p.batch * p.NG;
    if (items <= 0) return PPBO_OK;
    // tuning key 14 = R > 0: leave R SMs free (persistent grid of SMs - R CTAs; a CTA fills its SM: 224 KB of shared memory and
    // 53k registers).  A launch that shares the GPU with the latency-bound GP fit (run_iteration on one GPU: the contraction needs
    // the weight-space fit only) keeps the tensor pipes of its SMs busy while the fit's kernels find the reserved SMs free at
    // once.  Measured alternative, one CTA per work item on all SMs (key 14 = -1): the fit's wide bandwidth-bound kernels then
    // collect their SMs one by one as ~120 us work items end and the GP fit stretches from 10.6 to 15.3 ms.
    const int reserve = g_tuning[14];
    const int grid = reserve < 0 ? items : min(items, max(sms - reserve, 1));
    PPBO_CL ozaki_rowmax_kernel<KS, BN, BIAS><<<grid, THREADS, C::SMEM, st>>>(p);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}


// ------------------------------------------------------------------------------------------------ issue-rate probe
// Diagnostic (scripts/ozaki_probe.py --ubench): `iters` back-to-back tcgen05.mma.kind::i8 of shape 128 x N x 32 on resident
// shared-memory operands, one issuing thread per SM; reports SM clocks per MMA.  mode 0: A and B from shared memory, 1: A from
// TMEM, 2: as 0 but the same B plane re-used by consecutive MMAs (A alternates).
template <int N>
__global__ void __launch_bounds__(128, 1) ozaki_mma_rate_kernel(int mode, int nacc, int iters, long long* out) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (BM + N) * KB * 2 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0x01010101u;
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    if (warp == 0) {
        long long t0 = 0, t1 = 0;
        const uint32_t a_base = smem_u32(smem), b_base = a_base + 2 * BM * KB;
        if (lane == 0) {
            tc_cp_128x256b(tmem_base + 448, umma_desc(a_base));
            tc_cp_128x256b(tmem_base + 456, umma_desc(a_base + BM * KB));
            tc_commit(&bar);
        }
        __syncwarp();
        mbar_wait(&bar, 0, nullptr, 0);
        tc_fence_after();
        if (lane == 0) {
            const uint64_t ad0 = umma_desc(a_base), bd0 = umma_desc(b_base);
            t0 = clock64();
            int acc = 0;
            for (int it = 0; it < iters; it += 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t d = tmem_base + (uint32_t)(acc * N);
                    acc = (acc + 1 == nacc) ? 0 : acc + 1;
                    const uint64_t ad = umma_desc_advance(ad0, (u & 1) * BM * KB + (u >> 1) * 2 * LBO);
                    const uint64_t bd = umma_desc_advance(bd0, (mode == 2 ? 0 : (u & 1)) * N * KB + (u >> 1) * 2 * LBO);
                    if (mode == 1) tc_mma_i8_ts(d, tmem_base + 448 + (u & 1) * 8, bd, IDESC, 1u);
                    else tc_mma_i8(d, ad, bd, IDESC, 1u);
                }
            }
            tc_commit(&bar);
        }
        __syncwarp();
        mbar_wait(&bar, 1, nullptr, 0);
        if (lane == 0) {
            t1 = clock64();
            out[blockIdx.x] = t1 - t0;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

template <int N>
static int mma_rate_launch(int mode, int nacc, int iters, int blocks, long long* out, cudaStream_t st) {
    const int smem = (BM + N) * KB * 2;
    PPBO_CUDA_CHECK(cudaFuncSetAttribute(ozaki_mma_rate_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PPBO_CL ozaki_mma_rate_kernel<N><<<blocks, 128, smem, st>>>(mode, nacc, iters, out);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}

}  // namespace oz
}  // namespace ppbo

using namespace ppbo;

extern "C" int ppbo_ozaki_mma_rate(int N, int mode, int nacc, int iters, int blocks, long long* clocks_out, void* stream) {
    PPBO_REQUIRE(iters >= 4 && iters % 4 == 0 && blocks >= 1 && mode >= 0 && mode <= 2, "arguments");
    PPBO_REQUIRE(nacc >= 1 && nacc * N <= 448, "accumulators must fit 448 TMEM columns");
    cudaStream_t st = (cudaStream_t)stream;
    switch (N) {
        case 32: return oz::mma_rate_launch<32>(mode, nacc, iters, blocks, clocks_out, st);
        case 64: return oz::mma_rate_launch<64>(mode, nacc, iters, blocks, clocks_out, st);
        case 128: return oz::mma_rate_launch<128>(mode, nacc, iters, blocks, clocks_out, st);
        case 256: return oz::mma_rate_launch<256>(mode, nacc, iters, blocks, clocks_out, st);
        default: PPBO_REQUIRE(false, "N in {32, 64, 128, 256}");
    }
}

extern "C" int ppbo_ozaki_tile_rows(int operand) { return operand == 0 ? oz::BM : oz::BN_DEFAULT; }

extern "C" long long ppbo_ozaki_plane_bytes(int rows, int K, int tile_rows, int batch, int slices) {
    if (rows < 0 || K < 1 || tile_rows < 8 || batch < 1 || slices < 1) return -1;
    return oz::shape_of(rows, K, tile_rows, batch, slices).plane_bytes;
}
extern "C" long long ppbo_ozaki_scale_doubles(int rows, int tile_rows, int batch) {
    if (rows < 0 || tile_rows < 8 || batch < 1) return -1;
    return (long long)batch * ceil_div(rows, tile_rows) * tile_rows;
}

extern "C" int ppbo_ozaki_slice(const double* X, long long ldx, long long strideX, int rows, int K, int tile_rows, int batch,
                                int slices, double* scale, signed char* planes, void* stream) {
    PPBO_REQUIRE(rows >= 0 && K >= 1 && batch >= 1, "shape");
    PPBO_REQUIRE(tile_rows >= 8 && tile_rows % 8 == 0, "tile_rows must be a multiple of 8");
    PPBO_REQUIRE(slices >= 2 && slices <= oz::MAX_KS, "slices in [2, 7]");
    PPBO_REQUIRE((reinterpret_cast<uintptr_t>(planes) & 15) == 0, "planes must be 16-byte aligned");
    if (rows == 0) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int8_t* pl = reinterpret_cast<int8_t*>(planes);
    switch (slices) {
        case 2: return oz::slice_launch<2>(X, ldx, strideX, rows, K, tile_rows, batch, scale, pl, st);
        case 3: return oz::slice_launch<3>(X, ldx, strideX, rows, K, tile_rows, batch, scale, pl, st);
        case 4: return oz::slice_launch<4>(X, ldx, strideX, rows, K, tile_rows, batch, scale, pl, st);
        case 5: return oz::slice_launch<5>(X, ldx, strideX, rows, K, tile_rows, batch, scale, pl, st);
        case 6: return oz::slice_launch<6>(X, ldx, strideX, rows, K, tile_rows, batch, scale, pl, st);
        default: return oz::slice_launch<7>(X, ldx, strideX, rows, K, tile_rows, batch, scale, pl, st);
    }
}

namespace ppbo { namespace oz {
template <int KS, bool RAW = false>
static int sample_slice_launch(const double* omega_map, const double* hess_diag, unsigned long long seed, unsigned int stream_id,
                               long long sample0, int S, int F, double* scale, int8_t* planes, cudaStream_t st) {
    const Shape s = shape_of(S, F, BM, 1, KS);
    const int smem = 8 * s.KBLK * KB * (int)sizeof(double);
    static std::once_flag once;
    static cudaError_t err = cudaSuccess;
    std::call_once(once, [] { err = cudaFuncSetAttribute(ozaki_sample_slice_kernel<KS, RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
    PPBO_CUDA_CHECK(err);
    PPBO_REQUIRE(smem <= 200 * 1024, "F too large for the fused draw (8 rows of F doubles must fit shared memory)");
    PPBO_CL ozaki_sample_slice_kernel<KS, RAW><<<s.rows_pad / 8, 256, smem, st>>>(omega_map, hess_diag, seed, stream_id, sample0, S,
                                                                                   s.rows_pad, F, s.KBLK, scale, planes);
    PPBO_LAUNCH_CHECK();
    return PPBO_OK;
}
}}

extern "C" int ppbo_ozaki_sample_slice(const double* omega_map, const double* hess_diag, unsigned long long seed, unsigned int stream_id,
                                       long long sample0, int S, int F, int slices, double* scale, signed char* planes, void* stream) {
    PPBO_REQUIRE(S >= 0 && F >= 1, "shape");
    PPBO_REQUIRE(slices >= 5 && slices <= oz::MAX_KS, "slices in [5, 7]");
    PPBO_REQUIRE((reinterpret_cast<uintptr_t>(planes) & 15) == 0, "planes must be 16-byte aligned");
    if (S == 0) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int8_t* pl = reinterpret_cast<int8_t*>(planes);
    switch (slices) {
        case 5: return oz::sample_slice_launch<5>(omega_map, hess_diag, seed, stream_id, sample0, S, F, scale, pl, st);
        case 6: return oz::sample_slice_launch<6>(omega_map, hess_diag, seed, stream_id, sample0, S, F, scale, pl, st);
        default: return oz::sample_slice_launch<7>(omega_map, hess_diag, seed, stream_id, sample0, S, F, scale, pl, st);
    }
}

extern "C" int ppbo_ozaki_normal_slice(unsigned long long seed, unsigned int stream_id, long long sample0, int S, int F, int slices,
                                       double* scale, signed char* planes, void* stream) {
    PPBO_REQUIRE(S >= 0 && F >= 1, "shape");
    PPBO_REQUIRE(slices >= 5 && slices <= oz::MAX_KS, "slices in [5, 7]");
    PPBO_REQUIRE((reinterpret_cast<uintptr_t>(planes) & 15) == 0, "planes must be 16-byte aligned");
    if (S == 0) return PPBO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int8_t* pl = reinterpret_cast<int8_t*>(planes);
    switch (slices) {
        case 5: return oz::sample_slice_launch<5, true>(nullptr, nullptr, seed, stream_id, sample0, S, F, scale, pl, st);
        case 6: return oz::sample_slice_launch<6, true>(nullptr, nullptr, seed, stream_id, sample0, S, F, scale, pl, st);
        default: return oz::sample_slice_launch<7, true>(nullptr, nullptr, seed, stream_id, sample0, S, F, scale, pl, st);
    }
}

extern "C" long long ppbo_ozaki_rowmax_workspace_bytes(int S, int P, int batch) {
    if (S < 0 || P < 1 || batch < 1) return -1;
    const int NT = ceil_div(P, oz::BN_DEFAULT);               // room for any grouping
    return NT > 1 ? (long long)batch * NT * S * 12 + 16 : 0;
}

static int ozaki_rowmax_impl(const signed char* Aplanes, const double* ascale, int S, const signed char* Bplanes,
                             const double* bscale, const double* bias, int P, int batch, int K, int slices, double* fmax, int* arg,
                             double* Fs_full, void* workspace, long long workspace_bytes, int* err_flag, void* stream) {
    PPBO_REQUIRE(S >= 0 && P >= 1 && batch >= 1 && K >= 1, "shape");
    PPBO_REQUIRE(slices >= 5 && slices <= oz::MAX_KS, "slices in [5, 7]");
    PPBO_REQUIRE(ceil_div(K, oz::KB) * oz::KB <= 16384, "K <= 16384 (INT32 accumulator range)");
    PPBO_REQUIRE((reinterpret_cast<uintptr_t>(Aplanes) & 15) == 0 && (reinterpret_cast<uintptr_t>(Bplanes) & 15) == 0,
                 "digit planes must be 16-byte aligned");
    if (S == 0) return PPBO_OK;
    oz::BiasParams p;
    p.A = reinterpret_cast<const int8_t*>(Aplanes); p.ascale = ascale; p.S = S; p.MT = ceil_div(S, oz::BM);
    p.B = reinterpret_cast<const int8_t*>(Bplanes); p.bscale = bscale; p.P = P; p.NT = ceil_div(P, oz::BN_DEFAULT); p.batch = batch;
    p.KBLK = ceil_div(K, oz::KB);
    p.NG = oz::column_groups(p.NT, p.KBLK, slices);
    p.ntg = ceil_div(p.NT, p.NG);
    // grids per block: as many as keep the block's B planes within ~48 MB of L2 (1 = the earlier order, grid outermost).
    // Measured on the bench shape under sustained load (round-robin): 1 -> 9.79 ms, 2 -> 9.77, 4 -> 9.68, 7 -> 9.83,
    // 20 -> 10.28: the kernel is bound by the tensor pipe under the power cap, the order only moves DRAM traffic.
    {
        const long long grid_bytes = (long long)p.NT * p.KBLK * slices * oz::BN_DEFAULT * oz::KB;
        const int gbk = (int)std::max<long long>(1, (48LL << 20) / std::max<long long>(grid_bytes, 1));
        p.GB = std::min(gbk, batch);
    }
    PPBO_REQUIRE(workspace_bytes >= ppbo_ozaki_rowmax_workspace_bytes(S, P, batch), "workspace too small");
    PPBO_REQUIRE(p.NG == 1 || workspace != nullptr, "workspace missing");
    double* pmax = reinterpret_cast<double*>(workspace);
    int* parg = reinterpret_cast<int*>(pmax + (long long)batch * p.NG * S);
    p.fmax = p.NG > 1 ? pmax : fmax; p.arg = p.NG > 1 ? parg : arg; p.full = Fs_full; p.ld_full = P; p.stride_full = (long long)S * P; p.err = err_flag;
    p.bias = bias;
    const oz::Params& p0 = p;                  // the unbiased kernels take the base block
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (bias) {
        switch (slices) {
            case 5: rc = oz::rowmax_launch<5, oz::BN_DEFAULT, true>(p, st); break;
            case 6: rc = oz::rowmax_launch<6, oz::BN_DEFAULT, true>(p, st); break;
            default: rc = oz::rowmax_launch<7, oz::BN_DEFAULT, true>(p, st); break;
        }
    } else switch (slices) {
        case 5: rc = oz::rowmax_launch<5, oz::BN_DEFAULT>(p0, st); break;
        case 6: rc = oz::rowmax_launch<6, oz::BN_DEFAULT>(p0, st); break;
        default: rc = oz::rowmax_launch<7, oz::BN_DEFAULT>(p0, st); break;
    }
    if (rc) return rc;
    if (p.NG > 1) {
        PPBO_CL oz::ozaki_merge_kernel<<<dim3(ceil_div(S, 256), batch), 256, 0, st>>>(pmax, parg, p.NG, S, fmax, arg);
        PPBO_LAUNCH_CHECK();
    }
    return PPBO_OK;
}

extern "C" int ppbo_ozaki_rowmax(const signed char* Aplanes, const double* ascale, int S, const signed char* Bplanes,
                                 const double* bscale, int P, int batch, int K, int slices, double* fmax, int* arg,
                                 double* Fs_full, void* workspace, long long workspace_bytes, int* err_flag, void* stream) {
    return ozaki_rowmax_impl(Aplanes, ascale, S, Bplanes, bscale, nullptr, P, batch, K, slices, fmax, arg, Fs_full, workspace,
                             workspace_bytes, err_flag, stream);
}

extern "C" int ppbo_ozaki_rowmax_bias(const signed char* Aplanes, const double* ascale, int S, const signed char* Bplanes,
                                      const double* bscale, const double* bias, int P, int batch, int K, int slices, double* fmax,
                                      int* arg, double* Fs_full, void* workspace, long long workspace_bytes, int* err_flag,
                                      void* stream) {
    PPBO_REQUIRE(bias != nullptr, "bias missing");
    return ozaki_rowmax_impl(Aplanes, ascale, S, Bplanes, bscale, bias, P, batch, K, slices, fmax, arg, Fs_full, workspace,
                             workspace_bytes, err_flag, stream);
}
