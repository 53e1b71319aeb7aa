// Equilibration of badly scaled matrices before the 16-bit factorization (mplu_options::equilibrate): LAPACK dgeequb's
// power-of-two row and column scales, computed on the device, and dlaqge's decision which of them to apply (EQUED).
// Scaling by powers of two is exact, and a no-pivot LU of diag(r) A diag(c) is the same factorization up to those
// scales, but it keeps row and column spreads of the input out of the fp16 range (Higham, Pranesh & Zounon, "Squeezing
// a matrix into half precision", SISC 2019).  All passes stream A once from HBM:
//   row pass      max_j |a_ij|           thread per row over a column chunk (like first_touch_kernel), one slot per chunk
//   row scales    r_i, ROWCND, AMAX      thread per row over the chunk slots
//   column pass   max_i r_i |a_ij| -> c_j, COLCND     block per column, 16-byte loads down the column
//   decision      EQUED, r / c = 1 on the side that is not applied
// The scaled first touch (W = fp32(r_i a_ij c_j)) is first_touch_kernel<true> in panel.cu.
#include "kernels.h"

#include <cfloat>
#include <cstdint>

namespace mplu {

namespace {

constexpr double kSmlnum = DBL_MIN;                    // dlamch('S') = 2^-1022
constexpr double kBignum = 1.0 / DBL_MIN;              // 2^1022
constexpr double kSmall = DBL_MIN / DBL_EPSILON;       // dlaqge: dlamch('S') / dlamch('P') = 2^-970
constexpr double kLarge = 1.0 / kSmall;
constexpr double kThresh = 0.1;                        // dlaqge THRESH

// max that keeps a NaN once it has met one (fmax would drop it)
__device__ __forceinline__ double max_nan(double m, double v) { return (v > m || v != v) ? v : m; }

// 2^int(log2 m) for a finite m > 0 with int() truncating toward zero -- dgeequb's RADIX**INT(LOG(m)/LOG(RADIX)) --
// computed exactly: m = f 2^k, f in [0.5, 1)
__device__ __forceinline__ double pow2_trunc_log2(double m) {
    int k;
    const double f = frexp(m, &k);
    return ldexp(1.0, m >= 1.0 ? k - 1 : (f > 0.5 ? k : k - 1));
}

// non-negative doubles order like their bit patterns
__device__ __forceinline__ unsigned long long bits(double v) { return (unsigned long long)__double_as_longlong(v); }
__device__ __forceinline__ double from_bits(unsigned long long b) { return __longlong_as_double((long long)b); }

// per-warp min / max of the power-of-two maxima and "a bad row or column was seen", one atomic each per warp
__device__ __forceinline__ void reduce_to(unsigned long long* eq, int slot_min, int slot_max, double pmin, double pmax,
                                          bool bad) {
    for (int o = 16; o > 0; o >>= 1) {
        pmin = fmin(pmin, __shfl_xor_sync(0xffffffffu, pmin, o));
        pmax = fmax(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
    }
    bad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0) {
        atomicMin(eq + slot_min, bits(pmin));
        atomicMax(eq + slot_max, bits(pmax));
        if (bad) atomicOr(eq + EQ_BAD, 1ull);
    }
}

// part[y * n + i] = max |a_ij| over the columns of chunk y (grid (ceil(n/256), nchunk))
__global__ void equil_row_max_kernel(const double* __restrict__ A, long long lda, int n, double* __restrict__ part) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    const int per = (n + gridDim.y - 1) / gridDim.y;
    const int c0 = blockIdx.y * per, c1 = min(n, c0 + per);
    double m = 0.0;
#pragma unroll 4
    for (int c = c0; c < c1; ++c) m = max_nan(m, fabs(__ldg(A + row + (long long)c * lda)));
    part[(long long)blockIdx.y * n + row] = m;
}

// r_i = 1 / 2^int(log2 max_j |a_ij|) (clamped like dgeequb); a zero row or a non-finite maximum marks the matrix bad
__global__ void equil_row_scale_kernel(const double* __restrict__ part, int nchunk, int n, double* __restrict__ r,
                                       unsigned long long* eq) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    double pmin = INFINITY, pmax = 0.0;
    bool bad = false;
    if (row < n) {
        double m = 0.0;
        for (int y = 0; y < nchunk; ++y) m = max_nan(m, part[(long long)y * n + row]);
        if (m > 0.0 && m <= DBL_MAX) {
            const double p = pow2_trunc_log2(m);
            r[row] = 1.0 / fmin(fmax(p, kSmlnum), kBignum);
            pmin = pmax = p;
        } else {
            bad = true;
            r[row] = 1.0;
        }
    }
    reduce_to(eq, EQ_RMIN, EQ_RMAX, pmin, pmax, bad);
}

// c_j = 1 / 2^int(log2 max_i r_i |a_ij|): one block per column, 16-byte loads down the column
__global__ void __launch_bounds__(256) equil_col_kernel(const double* __restrict__ A, long long lda, int n,
                                                        const double* __restrict__ r, double* __restrict__ cs,
                                                        unsigned long long* eq) {
    const int j = blockIdx.x;
    const double* col = A + (long long)j * lda;
    const int head = (reinterpret_cast<uintptr_t>(col) & 15) ? 1 : 0;  // odd lda: every other column starts mid-pair
    const int pairs = (n - head) / 2;
    const double2* col2 = reinterpret_cast<const double2*>(col + head);
    double m = 0.0;
#pragma unroll 4
    for (int i = threadIdx.x; i < pairs; i += blockDim.x) {
        const double2 v = __ldg(col2 + i);
        const int k = head + 2 * i;
        m = max_nan(m, fabs(v.x) * __ldg(r + k));
        m = max_nan(m, fabs(v.y) * __ldg(r + k + 1));
    }
    if (threadIdx.x == 0) {
        if (head) m = max_nan(m, fabs(col[0]) * r[0]);
        if (head + 2 * pairs < n) m = max_nan(m, fabs(col[n - 1]) * r[n - 1]);
    }
    for (int o = 16; o > 0; o >>= 1) m = max_nan(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ double sm[8];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x >= 32) return;
    m = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.0;
    for (int o = 16; o > 0; o >>= 1) m = max_nan(m, __shfl_xor_sync(0xffffffffu, m, o));
    double pmin = INFINITY, pmax = 0.0;
    bool bad = false;
    if (threadIdx.x == 0) {
        if (m > 0.0 && m <= DBL_MAX) {
            const double p = pow2_trunc_log2(m);
            cs[j] = 1.0 / fmin(fmax(p, kSmlnum), kBignum);
            pmin = pmax = p;
        } else {
            bad = true;
            cs[j] = 1.0;
        }
    }
    reduce_to(eq, EQ_CMIN, EQ_CMAX, pmin, pmax, bad);
}

// dlaqge: scale the rows if ROWCND < 0.1 or AMAX outside [SMALL, LARGE], the columns if COLCND < 0.1; nothing after a
// zero row / column or a non-finite entry.  Every thread takes the (same) decision and resets its r_i / c_i to 1 on a
// side that is not applied; thread 0 publishes EQUED (bit 0 rows, bit 1 columns).
__global__ void equil_decide_kernel(unsigned long long* eq, double* __restrict__ r, double* __restrict__ cs, int n) {
    int equed = 0;
    if (eq[EQ_BAD] == 0) {
        const double rmin = from_bits(eq[EQ_RMIN]), rmax = from_bits(eq[EQ_RMAX]);
        const double cmin = from_bits(eq[EQ_CMIN]), cmax = from_bits(eq[EQ_CMAX]);
        const double rowcnd = fmax(rmin, kSmlnum) / fmin(rmax, kBignum);
        const double colcnd = fmax(cmin, kSmlnum) / fmin(cmax, kBignum);
        const double amax = rmax;
        if (!(rowcnd >= kThresh && amax >= kSmall && amax <= kLarge)) equed |= 1;
        if (!(colcnd >= kThresh)) equed |= 2;
    }
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        if (!(equed & 1)) r[i] = 1.0;
        if (!(equed & 2)) cs[i] = 1.0;
    }
    if (i == 0) eq[EQ_EQUED] = (unsigned long long)equed;
}

// out(:, j) = s o in(:, j), or out(:, j) += s o in(:, j), for j < k (in may be out)
__global__ void diag_scale_kernel(const double* __restrict__ s, int n, const double* in, long long ldi, double* out,
                                  long long ldo, int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long j = blockIdx.y;
    const double v = s[i] * in[i + j * ldi];
    out[i + j * ldo] = accumulate ? out[i + j * ldo] + v : v;
}

}  // namespace

int launch_equilibrate(const double* A, long long lda, int n, double* part, int nchunk, double* r, double* c,
                       unsigned long long* eq, cudaStream_t st) {
    // minima start at +inf's bit pattern and above (0xFF..), maxima, the bad flag and EQUED at 0
    if (cudaMemsetAsync(eq, 0xFF, 2 * sizeof(unsigned long long), st) != cudaSuccess) return (int)cudaGetLastError();
    if (cudaMemsetAsync(eq + 2, 0, (EQ_WORDS - 2) * sizeof(unsigned long long), st) != cudaSuccess)
        return (int)cudaGetLastError();
    const int rb = (n + 255) / 256;
    equil_row_max_kernel<<<dim3(rb, nchunk), 256, 0, st>>>(A, lda, n, part);
    equil_row_scale_kernel<<<rb, 256, 0, st>>>(part, nchunk, n, r, eq);
    equil_col_kernel<<<n, 256, 0, st>>>(A, lda, n, r, c, eq);
    equil_decide_kernel<<<rb, 256, 0, st>>>(eq, r, c, n);
    return (int)cudaGetLastError();
}

int launch_diag_scale(const double* s, int n, int k, const double* in, long long ldi, double* out, long long ldo,
                      int accumulate, cudaStream_t st) {
    if (n <= 0 || k <= 0) return 0;
    diag_scale_kernel<<<dim3((n + 255) / 256, k), 256, 0, st>>>(s, n, in, ldi, out, ldo, accumulate);
    return (int)cudaGetLastError();
}

}  // namespace mplu
