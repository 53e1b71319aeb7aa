// Panel-side kernels of the no-pivot mixed-precision LU:
//   * first touch: fp64 A -> fp32 working matrix W (zero/identity padded), |A| max and row sums (for ||A||_inf)
//   * power-of-two scale selection for the 16-bit shadows (fp16 range: SURVEY.md section 7 hard part 3)
//   * fp32 -> 16-bit shadow casts
//   * diag_lu: no-pivot LU of one 128x128 diagonal block held on chip, together with inv(L11) and inv(U11), so
//     the panel solves L21 = A21*inv(U11), U12 = inv(L11)*A12 become tensor-core GEMMs.
// The diagonal-block LU is the no-pivot column elimination of /root/reference/dgetf2_native_npv.cu:18-35 (multiplier
// = a[r,j]/a[j,j], rank-1 update of the columns to the right), restated for one CTA with the block in registers
// and one __syncthreads() per column instead of one grid.sync() per column straight from global memory.
#include "kernels.h"
#include "leaf.cuh"
#include "ptx.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace mplu {

namespace {

using namespace leaf;

__device__ __forceinline__ void atomic_max_float_nonneg(float* addr, float v) {
    // valid for non-negative floats: integer order == float order
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
}

// ---------------------------------------------------------------------------------------------------------------
// first touch: W = fp32(A) on [0,n)^2, identity on the padding diagonal, zero elsewhere in the padding.
// grid: (ceil(npad/256), NCHUNK); block 256 threads; thread = one row, loops over its column chunk of [cb, ce).
// Row sums of chunk y go to slot slot0 + y of rowsum_part (the streamed host path touches one block column at a time).
// kScaled (equilibration, csrc/equil.cu): W = fp32(rscale_i a_ij cscale_j) and amax over those scaled values; the row sums stay
// those of the unscaled |a_ij| (||A||_inf of the caller's matrix).  The scales are powers of two, so the product is exact.
template <bool kScaled>
__global__ void first_touch_kernel(const double* __restrict__ A, long long lda, int n, float* __restrict__ W,
                                   long long ldw, int npad, int cb, int ce, int slot0, float* amax,
                                   double* rowsum_part, int rend, const double* __restrict__ rscale = nullptr,
                                   const double* __restrict__ cscale = nullptr) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rend) npad = 0;  // rows beyond rend are not touched (block-row variant); the block still reduces amax
    const int nchunk = gridDim.y;
    const int cols_per = (ce - cb + nchunk - 1) / nchunk;
    const int c0 = cb + blockIdx.y * cols_per;
    const int c1 = min(ce, c0 + cols_per);
    float lmax = 0.f;
    double rs = 0.0;
    if (row < npad) {
        double ri = 1.0;
        if constexpr (kScaled) ri = row < n ? __ldg(rscale + row) : 1.0;
#pragma unroll 4
        for (int c = c0; c < c1; ++c) {
            float w;
            if (row < n && c < n) {
                const double a = __ldg(A + row + (long long)c * lda);
                if constexpr (kScaled)
                    w = static_cast<float>(ri * a * __ldg(cscale + c));
                else
                    w = static_cast<float>(a);
                rs += fabs(a);
                lmax = fmaxf(lmax, fabsf(w));
            } else {
                w = (row == c) ? 1.f : 0.f;
            }
            W[row + (long long)c * ldw] = w;
        }
        if (row < n && rowsum_part) rowsum_part[(long long)(slot0 + blockIdx.y) * n + row] = rs;
    }
    // block max -> one atomic
    __shared__ float smax[8];
    for (int o = 16; o > 0; o >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = lmax;
    __syncthreads();
    if (threadIdx.x == 0) {
        float m = 0.f;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) m = fmaxf(m, smax[i]);
        atomic_max_float_nonneg(amax, m);
    }
}

// ||A||_inf = max_i sum_chunks rowsum_part[chunk][i]; grid-stride over rows, one atomicMax per warp (anorm zeroed by
// the launcher; non-negative doubles order like their bit patterns)
__global__ void anorm_kernel(const double* __restrict__ rowsum_part, int n, int nchunk, double* anorm) {
    double m = 0.0;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int c = 0; c < nchunk; ++c) s += rowsum_part[(long long)c * n + r];
        m = fmax(m, s);
    }
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0)
        atomicMax(reinterpret_cast<unsigned long long*>(anorm), (unsigned long long)__double_as_longlong(m));
}

// scales[SC_A] = 2^e with amax*2^e in (2^(target-1), 2^target]; scales[SC_L] fixed; plus reciprocals.
__global__ void scales_kernel(const float* amax, float* scales, int target_exp_a, int exp_l, int bf16) {
    float a = *amax;
    float sA = 1.f, sL = 1.f;
    if (!bf16) {
        if (a > 0.f && isfinite(a)) {
            int e;
            frexpf(a, &e);  // a = f * 2^e, f in [0.5,1)  ->  a <= 2^e
            sA = ldexpf(1.f, target_exp_a - e);
        }
        sL = ldexpf(1.f, exp_l);
    }
    scales[SC_A] = sA;
    scales[SC_A_INV] = 1.f / sA;
    scales[SC_L] = sL;
    scales[SC_L_INV] = 1.f / sL;
    scales[SC_NEG_LA_INV] = -1.f / (sL * sA);
    scales[SC_ONE] = 1.f;
}

// H(r,c) = cvt16(W(r,c) * *scale) on a rows x cols block; thread handles 4 consecutive rows
__global__ void shadow_cast_kernel(const float* __restrict__ W, long long ldw, void* __restrict__ H, long long ldh,
                                   int rows, int cols, const float* scale, int bf16, int* status) {
    const float s = scale ? __ldg(scale) : 1.f;
    const float hmax = bf16 ? 3.0e38f : 65504.f;
    const int r4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    bool ovf = false;
    if (r4 < rows) {
        for (int c = blockIdx.y; c < cols; c += gridDim.y) {
            const float* src = W + r4 + (long long)c * ldw;
            if (r4 + 3 < rows && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((ldh & 3) == 0)) {
                const float4 v = *reinterpret_cast<const float4*>(src);
                const float a = v.x * s, b = v.y * s, cc = v.z * s, d = v.w * s;
                ovf |= !(fabsf(a) <= hmax) | !(fabsf(b) <= hmax) | !(fabsf(cc) <= hmax) | !(fabsf(d) <= hmax);
                uint2 pk;
                if (bf16) {
                    __nv_bfloat162 p0 = __floats2bfloat162_rn(a, b), p1 = __floats2bfloat162_rn(cc, d);
                    pk.x = *reinterpret_cast<uint32_t*>(&p0);
                    pk.y = *reinterpret_cast<uint32_t*>(&p1);
                } else {
                    __half2 p0 = __floats2half2_rn(a, b), p1 = __floats2half2_rn(cc, d);
                    pk.x = *reinterpret_cast<uint32_t*>(&p0);
                    pk.y = *reinterpret_cast<uint32_t*>(&p1);
                }
                *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(H) + r4 + (long long)c * ldh) = pk;
            } else {
                for (int i = 0; i < 4 && r4 + i < rows; ++i) {
                    const float a = src[i] * s;
                    ovf |= !(fabsf(a) <= hmax);
                    store16(H, r4 + i + (long long)c * ldh, a, bf16);
                }
            }
        }
    }
    if (status && ovf) atomicOr(status, 1);
}

// ---------------------------------------------------------------------------------------------------------------
// diag_lu: the 128x128 leaf (leaf.cuh) as a stand-alone cluster-of-2 kernel; the fused GETRF kernel (getrf_fused.cu)
// runs the same body inside its persistent grid.
__global__ void __launch_bounds__(DL_THREADS, 1)
diag_lu_kernel(float* __restrict__ W, long long ldw, int k0, void* __restrict__ Linv16, void* __restrict__ Uinv16,
               long long ld16, float* __restrict__ Linv32, float* __restrict__ Uinv32, float* tile_scales,
               int first_in_tile, int blk, int bf16, int* status, long long* dbg_clk, int valid) {
    extern __shared__ float dl_smem[];
    ptx::griddep_launch();
    ptx::griddep_wait();  // programmatic launch: the predecessor's writes to W are visible from here on
    diag_lu_body(dl_smem, (int)blockIdx.x, W, ldw, k0, Linv16, Uinv16, ld16, Linv32, Uinv32, tile_scales, first_in_tile, blk,
                 bf16, status, dbg_clk, valid);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
int launch_first_touch(const double* A, long long lda, int n, float* W, long long ldw, int npad, float* amax,
                       double* rowsum_part, int nchunk, double* anorm, cudaStream_t st, const double* rscale,
                       const double* cscale) {
    cudaMemsetAsync(amax, 0, sizeof(float), st);
    dim3 grid((npad + 255) / 256, nchunk);
    if (rscale)
        first_touch_kernel<true><<<grid, 256, 0, st>>>(A, lda, n, W, ldw, npad, 0, npad, 0, amax, rowsum_part, npad, rscale,
                                                       cscale);
    else
        first_touch_kernel<false><<<grid, 256, 0, st>>>(A, lda, n, W, ldw, npad, 0, npad, 0, amax, rowsum_part, npad);
    cudaMemsetAsync(anorm, 0, sizeof(double), st);
    anorm_kernel<<<(n + 255) / 256, 256, 0, st>>>(rowsum_part, n, nchunk, anorm);
    return (int)cudaGetLastError();
}

int launch_first_touch_cols(const double* A, long long lda, int n, float* W, long long ldw, int npad, int cb, int ce,
                            float* amax, double* rowsum_part, int slot0, int nslots, cudaStream_t st) {
    if (ce <= cb || nslots <= 0) return 0;
    dim3 grid((npad + 255) / 256, nslots);
    first_touch_kernel<false><<<grid, 256, 0, st>>>(A, lda, n, W, ldw, npad, cb, ce, slot0, amax, rowsum_part, npad);
    return (int)cudaGetLastError();
}

int launch_first_touch_block(const double* A, long long lda, int n, float* W, long long ldw, int npad, int rows, int cb, int ce,
                             float* amax, cudaStream_t st) {
    if (ce <= cb || rows <= 0) return 0;
    dim3 grid((rows + 255) / 256, 64);
    first_touch_kernel<false><<<grid, 256, 0, st>>>(A, lda, n, W, ldw, npad, cb, ce, 0, amax, nullptr, rows);
    return (int)cudaGetLastError();
}

int launch_anorm(const double* rowsum_part, int n, int nslots, double* anorm, cudaStream_t st) {
    cudaMemsetAsync(anorm, 0, sizeof(double), st);
    anorm_kernel<<<(n + 255) / 256, 256, 0, st>>>(rowsum_part, n, nslots, anorm);
    return (int)cudaGetLastError();
}

int launch_scales(const float* amax, float* scales, int target_exp_a, int exp_l, int bf16, cudaStream_t st) {
    scales_kernel<<<1, 1, 0, st>>>(amax, scales, target_exp_a, exp_l, bf16);
    return (int)cudaGetLastError();
}

int launch_shadow_cast(const float* W, long long ldw, void* H, long long ldh, int rows, int cols, const float* scale,
                       int bf16, int* status, cudaStream_t st) {
    if (rows <= 0 || cols <= 0) return 0;
    dim3 grid((rows + 1023) / 1024, cols < 2048 ? cols : 2048);
    shadow_cast_kernel<<<grid, 256, 0, st>>>(W, ldw, H, ldh, rows, cols, scale, bf16, status);
    return (int)cudaGetLastError();
}

int panel_init() {
    return (int)cudaFuncSetAttribute(diag_lu_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DL_SMEM_BYTES);
}

int launch_diag_lu(float* W, long long ldw, int k0, void* Linv16, void* Uinv16, long long ld16, float* Linv32,
                   float* Uinv32, float* tile_scales, int first_in_tile, int blk, int bf16, int* status, cudaStream_t st,
                   long long* dbg_clk, int pdl, int valid) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2);  // CTA 0: L\U + inv(L11), CTA 1: inv(U11)
    cfg.blockDim = dim3(DL_THREADS);
    cfg.dynamicSmemBytes = DL_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 2 : 1;
    return (int)cudaLaunchKernelEx(&cfg, diag_lu_kernel, W, ldw, k0, Linv16, Uinv16, ld16, Linv32, Uinv32, tile_scales,
                                   first_in_tile, blk, bf16, status, dbg_clk, valid);
}

}  // namespace mplu
