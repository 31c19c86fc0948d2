// ppbo_b200 -- internal declarations of the dense linear-algebra layer (linalg.cu)
#pragma once
#include "common.cuh"

namespace ppbo {

constexpr int CHOL_NB = 128;   // Cholesky block size: K of the trailing DMMA updates

long long potrf_dinv_doubles(int n);
// in-place blocked lower Cholesky; dinv receives the inverted diagonal blocks; *info_d (device) = 0 or first bad pivot (1-based)
int potrf_lower(double* A, long long lda, int n, double* dinv, int* info_d, cudaStream_t st);
// (L L^T) x = t in place; t must hold n + CHOL_NB doubles
int potrs_vec(const double* L, long long ldl, int n, const double* dinv, double* t, cudaStream_t st);
// X[nrhs x n] <- X . L^-T
int trsm_right_lower_t(const double* L, long long ldl, int n, const double* dinv, double* X, long long ldx, int nrhs,
                       cudaStream_t st);
// block-inverse solves for factors that serve many right-hand sides (see linalg.cu)
long long blockinv_doubles(int n);
int blockinv_build(const double* L, long long ldl, int n, const double* dinv, double* W, cudaStream_t st, int first_block = 0);
int potrs_vec_blockinv(const double* L, long long ldl, int n, double* W, double* t, cudaStream_t st, const double* skip = nullptr);
// the two halves of potrs_vec_blockinv (y = L^-1 t lands in blockinv_y(W, n); t = L^-T y) and the few-row right solve
double* blockinv_y(double* W, int n);
int potrs_fwd_blockinv(const double* L, long long ldl, int n, double* W, double* t, cudaStream_t st, const double* skip = nullptr);
int potrs_bwd_blockinv(const double* L, long long ldl, int n, double* W, double* t, cudaStream_t st, const double* skip = nullptr);
int trsm_right_blockinv(const double* L, long long ldl, int n, const double* W, double* T, long long ldt, double* R, long long ldr,
                        int nrhs, cudaStream_t st);
int gemv(const double* A, long long lda, int M, int N, const double* x, double* y, cudaStream_t st, const double* skip = nullptr);
// y = A x for a symmetric n x n A of which only the lower triangle is read; part: symv_scratch_doubles(n) doubles.  The result
// does not depend on the launch grid.
long long symv_scratch_doubles(int n);
int symv_lower(const double* A, long long lda, int n, const double* x, double* y, double* part, cudaStream_t st,
               const double* skip = nullptr);

}  // namespace ppbo
