// Full-precision fallback of the mixed-precision solve, LAPACK dsgesv style (dsgesv.f: "if the iterative refinement
// fails ... the routine falls back to a double precision factorization and solve"; ITER < 0 tells why).
// When the low-precision factorization cannot be used (16-bit overflow in fp16 AND bf16, an exact zero pivot without
// pivoting) or refinement does not reach the tolerance in max_iters, opts.fp64_fallback = 1 redoes the solve with an fp64
// LU WITH row pivoting: the reference's own algorithm -- fp16 pivot discovery + fp64 elimination, MPF.cu:100-241, on the
// device-resident copy (csrc/mpf_compat.cu: mpf_device) -- followed by fp64 triangular solves and fp64 refinement with
// those factors.  mplu_stats::fp64_fallback = 1 and mplu_stats::dsgesv_iter < 0 report it (-2 overflow, -3 zero pivot /
// unusable low-precision factors, -(max_iters + 1) refinement stalled: dsgesv's ITER convention).
// A rare path: written for clarity, not speed (one launch per 128-block of each triangular sweep).
#include "lu_internal.h"

#include <algorithm>

namespace mplu_detail {

cudaError_t mpf_device(double* d_A, int N, int r, int* d_ipiv);  // mpf_compat.cu

namespace {

constexpr int FB = 128;

// x <- P x for the sequential row interchanges ipiv (1-based, dlaswp order): the interchanges are applied to an index
// vector in shared memory by one thread, then all threads gather
__global__ void permute_kernel(const double* __restrict__ x, double* __restrict__ out, const int* __restrict__ ipiv, int n) {
    extern __shared__ int perm[];
    for (int i = threadIdx.x; i < n; i += blockDim.x) perm[i] = i;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int j = 0; j < n; ++j) {
            const int p = ipiv[j] - 1;
            if (p != j && p >= 0 && p < n) { const int t = perm[j]; perm[j] = perm[p]; perm[p] = t; }
        }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = x[perm[i]];
}

// the FB x FB diagonal block at k0: unit-lower forward substitution (lower = 1) or upper backward substitution
__global__ void tri_block_kernel(const double* __restrict__ LU, long long lda, int k0, int nb, double* x, int lower) {
    __shared__ double xs[FB];
    const int t = threadIdx.x;
    if (t < nb) xs[t] = x[k0 + t];
    __syncthreads();
    for (int s = 0; s < nb; ++s) {
        const int j = lower ? s : nb - 1 - s;
        if (!lower) {
            if (t == j) xs[j] = xs[j] / LU[(k0 + j) + (long long)(k0 + j) * lda];
            __syncthreads();
        }
        const double xj = xs[j];
        if (t < nb && (lower ? t > j : t < j)) xs[t] -= LU[(k0 + t) + (long long)(k0 + j) * lda] * xj;
        __syncthreads();
    }
    if (t < nb) x[k0 + t] = xs[t];
}

// x[r0 .. r0+nrows) -= LU[r0.., c0 .. c0+nb) * x[c0 .. c0+nb)
__global__ void gemv_sub_kernel(const double* __restrict__ LU, long long lda, int r0, int nrows, int c0, int nb, double* x) {
    __shared__ double xs[FB];
    if (threadIdx.x < nb) xs[threadIdx.x] = x[c0 + threadIdx.x];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows) return;
    const double* a = LU + (r0 + i) + (long long)c0 * lda;
    double acc0 = 0.0, acc1 = 0.0;
    int c = 0;
    for (; c + 1 < nb; c += 2) {
        acc0 = fma(a[(long long)c * lda], xs[c], acc0);
        acc1 = fma(a[(long long)(c + 1) * lda], xs[c + 1], acc1);
    }
    if (c < nb) acc0 = fma(a[(long long)c * lda], xs[c], acc0);
    x[r0 + i] -= acc0 + acc1;
}

__global__ void axpy_kernel(double* x, const double* d, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] += d[i];
}

// x <- U^-1 L^-1 P x with the fp64 factors
int lu_solve_fp64(const double* LU, int n, const int* ipiv, const double* rhs, double* x, double* tmp, cudaStream_t st) {
    if ((size_t)n * sizeof(int) > 200 * 1024) return MPLU_E_ARG;  // the index vector must fit shared memory (n <= 51200)
    CK(cudaFuncSetAttribute(permute_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));  // per device: not cached
    permute_kernel<<<1, 1024, (size_t)n * sizeof(int), st>>>(rhs, tmp, ipiv, n);
    CK(cudaMemcpyAsync(x, tmp, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
    for (int k0 = 0; k0 < n; k0 += FB) {
        const int nb = n - k0 < FB ? n - k0 : FB, below = n - k0 - nb;
        tri_block_kernel<<<1, FB, 0, st>>>(LU, n, k0, nb, x, 1);
        if (below > 0) gemv_sub_kernel<<<(below + 127) / 128, 128, 0, st>>>(LU, n, k0 + nb, below, k0, nb, x);
    }
    for (int k0 = ((n - 1) / FB) * FB; k0 >= 0; k0 -= FB) {
        const int nb = n - k0 < FB ? n - k0 : FB;
        tri_block_kernel<<<1, FB, 0, st>>>(LU, n, k0, nb, x, 0);
        if (k0 > 0) gemv_sub_kernel<<<(k0 + 127) / 128, 128, 0, st>>>(LU, n, 0, k0, k0, nb, x);
    }
    return (int)cudaGetLastError();
}

}  // namespace

// why: the MPLU_E_* code the low-precision path ended with.  Returns 0 when the fp64 solve met the stopping rule.
int fp64_fallback_solve(mplu_context* c, int n, const double* dA, long long lda, int nrhs, const double* dB, long long ldb,
                        double* dX, long long ldx, int why, double* berr, mplu_stats* stats) {
    CK(cudaStreamSynchronize(c->stream));
    cudaStream_t st = 0;  // mpf_device runs on the legacy default stream
    double* LU = nullptr;
    double* tmp = nullptr;
    double* d = nullptr;
    int* ipiv = nullptr;
    int rc = 0;
    auto body = [&]() -> int {
        CK(cudaMalloc(&LU, (size_t)n * n * sizeof(double)));
        CK(cudaMalloc(&tmp, (size_t)n * sizeof(double)));
        CK(cudaMalloc(&d, (size_t)n * sizeof(double)));
        CK(cudaMalloc(&ipiv, (size_t)n * sizeof(int)));
        CK(cudaMemcpy2DAsync(LU, (size_t)n * sizeof(double), dA, (size_t)lda * sizeof(double), (size_t)n * sizeof(double), n,
                             cudaMemcpyDeviceToDevice, st));
        {   // identity pivots for the entry a trailing 1 x 1 panel never writes (MPF.cu:104)
            std::vector<int> id(n);
            for (int i = 0; i < n; ++i) id[i] = i + 1;
            CK(cudaMemcpyAsync(ipiv, id.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));
        }
        CK(mpf_device(LU, n, 32, ipiv));
        // every column is solved and refined on its own, at most 5 corrections each; stats report the worst column
        const double* db = nullptr;
        double* dx = nullptr;
        bool first = true;
        RefineOps ops;
        ops.norms = c->norms;
        ops.anorm = c->anorm;
        ops.st = st;
        ops.first_solve = [&]() -> int {
            CKI(mplu::launch_column_absmax(db, n, n, 1, c->norms + 2, st));
            return lu_solve_fp64(LU, n, ipiv, db, dx, tmp, st);
        };
        ops.residual = [&](bool* formed_anorm) -> int {
            // the row sums of |A| ride along in the first pass (the low-precision path may not have got that far)
            *formed_anorm = first;
            first = false;
            return mplu::launch_residual(dA, lda, n, dx, db, c->r, c->partial, c->nchunk, c->norms, st,
                                         *formed_anorm ? c->rowsum_part : nullptr, *formed_anorm ? c->anorm : nullptr);
        };
        ops.correct = [&](int*) -> int {
            CKI(lu_solve_fp64(LU, n, ipiv, c->r, d, tmp, st));
            axpy_kernel<<<(n + 255) / 256, 256, 0, st>>>(dx, d, n);
            return 0;
        };
        ops.wait = [&]() -> int { return (int)cudaStreamSynchronize(st); };
        RefineResult all;
        all.converged = 1;
        for (int col = 0; col < nrhs; ++col) {
            db = dB + (long long)col * ldb;
            dx = dX + (long long)col * ldx;
            first = true;
            RefineResult one;
            CKI(refine(ops, n, 1, 5, c->opts.tol, &one));
            all.col.push_back(one.col[0]);
            all.anorm = one.anorm;
            all.iters = std::max(all.iters, one.iters);
            all.converged &= one.converged;
        }
        refine_stats(all, n, berr, stats);
        if (stats) {
            stats->fp64_fallback = 1;
            stats->dsgesv_iter = dsgesv_iter(why, c->opts.max_iters > 0 ? c->opts.max_iters : 30);
        }
        return refine_rc(all.converged, 0);
    };
    rc = body();
    cudaStreamSynchronize(st);
    cudaFree(LU); cudaFree(tmp); cudaFree(d); cudaFree(ipiv);
    return rc;
}

}  // namespace mplu_detail
