// 2D block-cyclic mixed-precision LU + fp64 iterative refinement across the GPUs of one box (SURVEY.md section 8e).
// The reference is single-GPU (cudaSetDevice(0), /root/reference/MPF.cu:77); this is the multi-GPU form of the same
// hot path: tile (I,J) of the nb-tiled matrix lives on process (I mod P, J mod Q) in ScaLAPACK local order.
//
// Per step k (diagonal tile owner (k mod P, k mod Q)):
//   chain lane  owner: GETRF of the nb x nb tile with merged inverses (lu.cu: getrf_resident_tile)
//               broadcast inv(U11) down the owner's process column and inv(L11) along its process row; the factored
//               tile and its fp32 block inverses go to every rank (they are replicated for the triangular solves)
//               process column: L panel = A21 inv(U11) (one tcgen05 GEMM);  process row: U panel = inv(L11) A12
//               broadcast the 16-bit L panel along process rows and the U panel along process columns (NCCL, NVLink)
//   bulk lane   trailing update  A22 -= Lpanel * Upanel  on every rank; the next tile column / tile row first, so
//               that step k+1's chain work overlaps the rest of update k (depth-1 look-ahead)
// Refinement: every rank keeps full-length x, b, r; r = b - A x is a local fp64 GEMV + one all-reduce; the triangular
// solves walk the tile rows (local fp32 GEMV + one nb-float all-reduce + the replicated diagonal tile's solve).
//
// One process hosts either ONE rank of an NCCL communicator (production: one process per GPU) or ALL P*Q logical
// ranks on one device without NCCL ("local" mode: collectives become device copies) -- the same schedule code runs
// in both, which is how the block-cyclic logic is tested on a single GPU.
#include "lu_internal.h"

#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>
#include <new>

using namespace mplu;
using namespace mplu_detail;

// ------------------------------------------------------------------------------------------------ NCCL (dlopen)
namespace {

typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { ncclSuccess = 0 };
enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2, ncclFloat32 = 7, ncclFloat64 = 8 };
enum { ncclSum = 0, ncclMax = 2 };

struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(ncclUniqueId*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    int (*CommSplit)(ncclComm_t, int, int, ncclComm_t*, void*) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};

NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.handle ? &api : nullptr;
    tried = true;
    const char* names[] = {getenv("MPLU_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        if (!nm || !*nm) continue;
        api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.handle) break;
    }
    if (!api.handle) return nullptr;
#define LOADSYM(field, sym)                                            \
    *(void**)(&api.field) = dlsym(api.handle, sym);                    \
    if (!api.field) { api.handle = nullptr; return nullptr; }
    LOADSYM(GetUniqueId, "ncclGetUniqueId")
    LOADSYM(CommInitRank, "ncclCommInitRank")
    LOADSYM(CommSplit, "ncclCommSplit")
    LOADSYM(CommDestroy, "ncclCommDestroy")
    LOADSYM(Broadcast, "ncclBroadcast")
    LOADSYM(AllReduce, "ncclAllReduce")
    LOADSYM(GroupStart, "ncclGroupStart")
    LOADSYM(GroupEnd, "ncclGroupEnd")
    LOADSYM(GetErrorString, "ncclGetErrorString")
#undef LOADSYM
    return &api;
}


#define NK(expr)                                   \
    do {                                           \
        int _e = (expr);                           \
        if (_e != ncclSuccess) return MPLU_E_NCCL; \
    } while (0)

// ------------------------------------------------------------------------------------------------ layout helpers
// local tiles of a dimension with T tiles dealt round-robin to P processes
inline int tiles_local(int T, int P, int p) { return p < T ? (T - p + P - 1) / P : 0; }
// number of local tiles (of process p) whose global index is <= k / < k
inline int cnt_le(int k, int P, int p) { return k >= p ? (k - p) / P + 1 : 0; }
inline int cnt_lt(int k, int P, int p) { return k > p ? (k - 1 - p) / P + 1 : 0; }

// ------------------------------------------------------------------------------------------------ kernels
// W = fp32(A_loc) on the local mloc x nloc block, |A| max, partial row sums scattered to GLOBAL row positions.
// grid (ceil(mloc/256), chunks); thread = one local row, loops over its chunk of local columns.
__global__ void local_first_touch_kernel(const double* __restrict__ A, long long lda, int mloc, int nloc,
                                         float* __restrict__ W, long long ldw, float* amax, double* rowsum_full,
                                         int nb, int P, int p) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    const int per = (nloc + gridDim.y - 1) / gridDim.y;
    const int c0 = blockIdx.y * per, c1 = min(nloc, c0 + per);
    float lmax = 0.f;
    if (row < mloc) {
        double rs = 0.0;
#pragma unroll 4
        for (int c = c0; c < c1; ++c) {
            const double a = __ldg(A + row + (long long)c * lda);
            const float w = static_cast<float>(a);
            rs += fabs(a);
            lmax = fmaxf(lmax, fabsf(w));
            W[row + (long long)c * ldw] = w;
        }
        const long long grow = ((long long)(row / nb) * P + p) * nb + row % nb;
        atomicAdd(rowsum_full + grow, rs);
    }
    for (int o = 16; o > 0; o >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(amax), __float_as_int(lmax));
}

// y_full[global row] += sum_{local cols in chunk} A_loc(row, c) * x[global col(c)]   (fp64, HBM-bound: 8 B / element)
// grid (ceil(mloc/256), chunks); thread = 2 consecutive local rows (mloc, nb even).
__global__ void __launch_bounds__(128)
local_gemv_f64_kernel(const double* __restrict__ A, long long lda, int mloc, int nloc, const double* __restrict__ x,
                      double* y_full, int nb, int P, int p, int Q, int q) {
    extern __shared__ double xs[];
    const int per = (nloc + gridDim.y - 1) / gridDim.y;
    const int c0 = blockIdx.y * per, c1 = min(nloc, c0 + per);
    for (int c = c0 + threadIdx.x; c < c1; c += blockDim.x)
        xs[c - c0] = x[((long long)(c / nb) * Q + q) * nb + c % nb];
    __syncthreads();
    const int r0 = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (r0 >= mloc) return;
    const double* Ap = A + r0 + (long long)c0 * lda;
    double a0 = 0.0, a1 = 0.0;
    const int nc = c1 - c0;
    const bool vec = ((lda & 1) == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
    int c = 0;
    if (vec) {
        for (; c + 8 <= nc; c += 8) {
            double2 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = __ldg(reinterpret_cast<const double2*>(Ap + (long long)(c + u) * lda));
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                a0 = fma(v[u].x, xs[c + u], a0);
                a1 = fma(v[u].y, xs[c + u], a1);
            }
        }
    }
    for (; c < nc; ++c) {
        a0 = fma(__ldg(Ap + (long long)c * lda), xs[c], a0);
        a1 = fma(__ldg(Ap + 1 + (long long)c * lda), xs[c], a1);
    }
    const long long grow = ((long long)(r0 / nb) * P + p) * nb + r0 % nb;
    atomicAdd(y_full + grow, a0);
    atomicAdd(y_full + grow + 1, a1);
}

// r = b - ax; norms[0] = max|r|, norms[1] = max|x|
__global__ void residual_full_kernel(const double* __restrict__ b, const double* __restrict__ ax,
                                     const double* __restrict__ x, double* __restrict__ r, int n, double* norms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double rv = 0.0, xv = 0.0;
    if (i < n) {
        rv = b[i] - ax[i];
        r[i] = rv;
        rv = fabs(rv);
        xv = fabs(x[i]);
    }
    for (int o = 16; o > 0; o >>= 1) {
        rv = fmax(rv, __shfl_xor_sync(0xffffffffu, rv, o));
        xv = fmax(xv, __shfl_xor_sync(0xffffffffu, xv, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(reinterpret_cast<unsigned long long*>(&norms[0]), (unsigned long long)__double_as_longlong(rv));
        atomicMax(reinterpret_cast<unsigned long long*>(&norms[1]), (unsigned long long)__double_as_longlong(xv));
    }
}

// part[global row of r] += sum_{c < nb} W_loc(r, c0 + c) * v[c]   for the local rows r in [r0, r1)   (fp32 factors, fp32 vector)
// One tile column of the local factors against the solution block that column multiplies: the right-looking half of the
// block-cyclic triangular solves.  HBM-bound (4 bytes per element).  grid (ceil((r1-r0)/128), nb/128), 256 threads: a block
// owns 128 rows x 128 columns, warp w the columns 16 w .. 16 w + 15, a lane 4 consecutive rows (128-bit loads, all 16 in
// flight: a single tile -- the latency-critical call -- is then two memory round trips, not sixteen); the eight warps'
// partial sums meet in shared memory and one warp adds them to `part` atomically (several columns' kernels may be adding to
// the same rows from two streams).
__global__ void __launch_bounds__(256)
tile_col_gemv_kernel(const float* __restrict__ W, long long ldw, int r0, int r1, int c0, const float* v,
                     float* part, int nb, int P, int p, const unsigned* wait_flag, unsigned wait_val, unsigned* dbg) {
    __shared__ float4 red[8][32];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wait_flag) {  // launched ahead of its operand (tile chain): the solution block is complete when the tile sweep's step
        if (threadIdx.x == 0) {  // counter has reached its final value
            unsigned f;
            const long long t0 = clock64();  // (never hang the GPU: give up after ~2 s, the solve then fails to converge)
            do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(f) : "l"(wait_flag) : "memory"); }
            while (f != wait_val && clock64() - t0 < 4000000000LL);
            if (f != wait_val && dbg) atomicOr(dbg, 2u);
        }
        __syncthreads();
    }
    const int cb = blockIdx.y * 128 + 16 * w;
    const int r = r0 + 128 * blockIdx.x + 4 * lane;  // r0, r1 are multiples of nb (a multiple of 128): no ragged block
    const float4* wp = reinterpret_cast<const float4*>(W + r + (long long)(c0 + cb) * ldw);
    const long long ld4 = ldw / 4;
    float4 t[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) t[u] = __ldcs(wp + u * ld4);
    float x[16];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float4 xv = __ldcg(reinterpret_cast<const float4*>(v + cb) + u);
        x[4 * u] = xv.x; x[4 * u + 1] = xv.y; x[4 * u + 2] = xv.z; x[4 * u + 3] = xv.w;
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < 16; ++u) {
        acc.x = fmaf(t[u].x, x[u], acc.x); acc.y = fmaf(t[u].y, x[u], acc.y);
        acc.z = fmaf(t[u].z, x[u], acc.z); acc.w = fmaf(t[u].w, x[u], acc.w);
    }
    red[w][lane] = acc;
    __syncthreads();
    if (w == 0) {
#pragma unroll
        for (int g = 1; g < 8; ++g) {
            const float4 o = red[g][lane];
            acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
        }
        float* out = part + ((long long)(r / nb) * P + p) * nb + r % nb;
        atomicAdd(out, acc.x); atomicAdd(out + 1, acc.y); atomicAdd(out + 2, acc.z); atomicAdd(out + 3, acc.w);
    }
}

// step counters of the tile sweeps: T forward sweeps start at step 0, T backward sweeps at step nblk
__global__ void fill_ready_kernel(unsigned* ready, int T, unsigned nblk) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * T) ready[i] = i < T ? 0u : nblk;
}
// ---- peer exchange of the triangular solves' partial sums (NCCL mode; replaces one ncclAllReduce of nb floats per tile step)
// Every rank owns one exchange buffer mapped into all its peers (CUDA IPC over NVLink): kPxFlagWords flag words, then slots
// of nb floats.  Slot / flag index of (sweep, tile row k, process column q) = (sweep T + k) Q + q.  A rank of the tile
// row's process row stores its nb partial sums into that slot of EVERY rank and then raises the slot's flag to the solve's
// epoch; every rank's tile sweep (lu_solve_kernel, csrc/ir.cu: SweepPx) waits for the Q flags of the step and adds the Q slots
// up itself.  One NVLink store + one flag per hop instead of a collective launch: the ranks' only per-step synchronisation.
constexpr size_t kPxDataFloats = (size_t)16 << 20;

__global__ void __launch_bounds__(256)
px_send_kernel(const float* __restrict__ src, float* const* __restrict__ peers, size_t slot, int nb, unsigned epoch) {
    float* base = peers[blockIdx.x];  // one block per destination rank
    float4* dst = reinterpret_cast<float4*>(base + kPxFlagWords + slot * nb);
    const float4* s4 = reinterpret_cast<const float4*>(src);
    for (int i = threadIdx.x; i < nb / 4; i += blockDim.x) dst[i] = s4[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0)
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(reinterpret_cast<unsigned*>(base) + slot), "r"(epoch) : "memory");
}

// x (+)= d
__global__ void apply_correction_kernel(const float* __restrict__ d, double* x, int n, int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = accumulate ? x[i] + (double)d[i] : (double)d[i];
}
// local-mode collectives
__global__ void sum_into_f32_kernel(float* dst, const float* src, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}
__global__ void sum_into_f64_kernel(double* dst, const double* src, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}
__global__ void max_into_f32_kernel(float* dst, const float* src, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = fmaxf(dst[i], src[i]);
}

// ------------------------------------------------------------------------------------------------ rank state
struct DRank {
    int p = 0, q = 0;
    mplu_context* ctx = nullptr;   // options / status / small device words for the GEMM launches of this rank
    mplu_context* dctx = nullptr;  // nb x nb context that factors diagonal tiles
    cudaStream_t chain = nullptr, bulk = nullptr;
    cudaStream_t hi = nullptr, hi2 = nullptr;  // greatest priority: the triangular solves' tile sweeps / their near GEMVs and sends (owned by this struct)
    cudaEvent_t ev_tmp = nullptr, ev_chain = nullptr, ev_bulk = nullptr, ev_e1 = nullptr, ev_d = nullptr, ev_panel[2] = {nullptr, nullptr};
    cudaEvent_t ev_t[4] = {nullptr, nullptr, nullptr, nullptr};
    static constexpr int kSolveRing = 8;
    cudaEvent_t ev_sol[kSolveRing] = {}, ev_far[kSolveRing] = {}, ev_swp[kSolveRing] = {};  // triangular solves: chain -> bulk (block solved), bulk -> chain
    int mt = 0, nt = 0;
    long long mloc = 0, nloc = 0;
    const double* A = nullptr;
    long long lda = 0;
    float* W = nullptr;
    uint16_t* Wh = nullptr;
    uint16_t* Lp[2] = {nullptr, nullptr};
    uint16_t* Up[2] = {nullptr, nullptr};
    uint16_t* InvL[2] = {nullptr, nullptr};
    uint16_t* InvU[2] = {nullptr, nullptr};
    float* tsc[2] = {nullptr, nullptr};  // {s_Linv, 1/s_Linv, s_Uinv, 1/s_Uinv} of the step's tile
    float* Dw = nullptr;    // T x (nb x nb) replicated factored diagonal tiles
    float* Dl32 = nullptr;  // T x nb/128 x (128 x 128) replicated fp32 inverses of their diagonal blocks
    float* Du32 = nullptr;
    Operand16 opWh, opLp[2], opUp[2], opInvL[2], opInvU[2];
    // refinement vectors (full length, replicated)
    double *r = nullptr, *ax = nullptr, *rowsum = nullptr, *norms = nullptr, *anorm = nullptr, *rhsbuf = nullptr;
    float *yv = nullptr, *xv = nullptr, *part = nullptr;  // part: 2 x n partial sums of the two sweeps (global row order)
    unsigned* ready = nullptr;
};

}  // namespace

struct mplu_dist {
    int device = 0;
    int P = 1, Q = 1;
    bool local_mode = true;
    int rank = 0, nranks = 1;
    ncclComm_t world = nullptr, rowc = nullptr, colc = nullptr;
    NcclApi* nccl = nullptr;
    std::vector<DRank> ranks;  // logical ranks hosted by this process (1 with NCCL, P*Q in local mode)
    int n = 0, nb = 0, T = 0;
    mplu_options opts{};
    int num_sms = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    int gemm_launches = 0, kernel_launches = 0;
    // device timing of the first hosted rank's trailing updates (the dominant kernel), like mplu_context::trail_ev
    std::vector<cudaEvent_t> trail_ev;
    int trail_count = 0;
    double trail_flops = 0, trail_bytes = 0;
    // staging of the host-buffer variant (one entry per logical rank)
    std::vector<double*> stA, stb, stx;
    std::vector<size_t> stA_cap;
    int st_n = 0;
    // the triangular solve of a single-rank process as a CUDA graph (captured on its second use for the current buffers)
    cudaGraphExec_t solve_exec = nullptr;
    int solve_uses = 0, solve_launches = 0;
    // peer exchange of the solves' partial sums (NCCL mode): own buffer, the peers' mappings, device table of all of them
    bool px_on = false;
    float* px_mine = nullptr;
    std::vector<void*> px_opened;
    float** px_peers = nullptr;
    unsigned px_epoch = 0;
    unsigned* px_dbg = nullptr;  // device word: bit 0 / 1 = a tile-chain / GEMV wait timed out (development)
    unsigned* px_started_h = nullptr;  // pinned, mapped: CTAs of the tile chain that are resident
    unsigned* px_started_d = nullptr;
};

namespace {

void free_rank_work(DRank& r) {
    cudaFree(r.W); cudaFree(r.Wh);
    for (int i = 0; i < 2; ++i) { cudaFree(r.Lp[i]); cudaFree(r.Up[i]); cudaFree(r.InvL[i]); cudaFree(r.InvU[i]); cudaFree(r.tsc[i]); }
    cudaFree(r.Dw); cudaFree(r.Dl32); cudaFree(r.Du32);
    cudaFree(r.r); cudaFree(r.ax); cudaFree(r.rowsum); cudaFree(r.norms); cudaFree(r.anorm); cudaFree(r.rhsbuf);
    cudaFree(r.yv); cudaFree(r.xv); cudaFree(r.part); cudaFree(r.ready);
    r.W = nullptr; r.Wh = nullptr;
    for (int i = 0; i < 2; ++i) { r.Lp[i] = r.Up[i] = r.InvL[i] = r.InvU[i] = nullptr; r.tsc[i] = nullptr; }
    r.Dw = r.Dl32 = r.Du32 = nullptr;
    r.r = r.ax = r.rowsum = r.norms = r.anorm = r.rhsbuf = nullptr;
    r.yv = r.xv = r.part = nullptr;
    r.ready = nullptr;
}

int alloc_rank_work(mplu_dist* d, DRank& r) {
    const int n = d->n, nb = d->nb, T = d->T;
    if (d->solve_exec) { cudaGraphExecDestroy(d->solve_exec); d->solve_exec = nullptr; }
    d->solve_uses = 0;
    free_rank_work(r);
    r.mt = tiles_local(T, d->P, r.p);
    r.nt = tiles_local(T, d->Q, r.q);
    r.mloc = (long long)r.mt * nb;
    r.nloc = (long long)r.nt * nb;
    const size_t ml = (size_t)(r.mloc > 0 ? r.mloc : nb), nl = (size_t)(r.nloc > 0 ? r.nloc : nb);
    CK(cudaMalloc(&r.W, ml * nl * sizeof(float)));
    CK(cudaMalloc(&r.Wh, ml * nl * sizeof(uint16_t)));
    for (int i = 0; i < 2; ++i) {
        CK(cudaMalloc(&r.Lp[i], ml * nb * sizeof(uint16_t)));
        CK(cudaMalloc(&r.Up[i], nl * nb * sizeof(uint16_t)));
        CK(cudaMalloc(&r.InvL[i], (size_t)nb * nb * sizeof(uint16_t)));
        CK(cudaMalloc(&r.InvU[i], (size_t)nb * nb * sizeof(uint16_t)));
        CK(cudaMalloc(&r.tsc[i], 4 * sizeof(float)));
    }
    CK(cudaMalloc(&r.Dw, (size_t)T * nb * nb * sizeof(float)));
    CK(cudaMalloc(&r.Dl32, (size_t)n * kDiagBlock * sizeof(float)));
    CK(cudaMalloc(&r.Du32, (size_t)n * kDiagBlock * sizeof(float)));
    CK(cudaMalloc(&r.r, n * sizeof(double)));
    CK(cudaMalloc(&r.ax, n * sizeof(double)));
    CK(cudaMalloc(&r.rowsum, n * sizeof(double)));
    CK(cudaMalloc(&r.norms, 3 * sizeof(double)));  // ||r||, ||x||, ||b||: RefineOps::norms for one column
    CK(cudaMalloc(&r.anorm, sizeof(double)));
    CK(cudaMalloc(&r.yv, n * sizeof(float)));
    CK(cudaMalloc(&r.xv, n * sizeof(float)));
    CK(cudaMalloc(&r.part, 2 * (size_t)n * sizeof(float)));
    CK(cudaMalloc(&r.rhsbuf, n * sizeof(double)));
    CK(cudaMalloc(&r.ready, (2 * (size_t)T + 1) * sizeof(unsigned)));  // one step counter per tile sweep
    CKI(make_operand(&r.opWh, r.Wh, ml, nl, ml));
    for (int i = 0; i < 2; ++i) {
        CKI(make_operand(&r.opInvL[i], r.InvL[i], nb, nb, nb));
        CKI(make_operand(&r.opInvU[i], r.InvU[i], nb, nb, nb));
        CKI(make_operand(&r.opUp[i], r.Up[i], nb, nl, nb));
    }
    // the nb x nb factorization context
    r.dctx->opts = d->opts;
    r.dctx->opts.nb = nb;
    r.dctx->opts.lookahead = 0;
    r.dctx->opts.use_graph = 0;
    CKI(ensure_work(r.dctx, nb));
    r.ctx->opts = d->opts;
    return 0;
}

DRank* find_rank(mplu_dist* d, int p, int q) {
    for (auto& r : d->ranks)
        if (r.p == p && r.q == q) return &r;
    return nullptr;
}

// ---- collectives.  scope: 0 = world, 1 = process row `line` (ranks (line, *)), 2 = process column `line`.
// `root` = the q (row scope) / p (column scope) / world rank p*Q+q of the sender.  get(rank) returns the rank's buffer;
// stream_of(rank) the stream the operation is ordered on.
template <class GetBuf, class GetStream>
int bcast(mplu_dist* d, int scope, int line, int root, size_t bytes, GetBuf get, GetStream stream_of) {
    if (bytes == 0) return 0;
    if (!d->local_mode) {
        DRank& r = d->ranks[0];
        if ((scope == 1 && r.p != line) || (scope == 2 && r.q != line)) return 0;
        ncclComm_t comm = scope == 0 ? d->world : (scope == 1 ? d->rowc : d->colc);
        void* buf = get(r);
        NK(d->nccl->Broadcast(buf, buf, bytes, ncclUint8, root, comm, stream_of(r)));
        return 0;
    }
    DRank* src = nullptr;
    for (auto& r : d->ranks) {
        const bool in = scope == 0 || (scope == 1 && r.p == line) || (scope == 2 && r.q == line);
        if (!in) continue;
        const int id = scope == 0 ? r.p * d->Q + r.q : (scope == 1 ? r.q : r.p);
        if (id == root) src = &r;
    }
    if (!src) return MPLU_E_ARG;
    CK(cudaEventRecord(src->ev_tmp, stream_of(*src)));
    for (auto& r : d->ranks) {
        const bool in = scope == 0 || (scope == 1 && r.p == line) || (scope == 2 && r.q == line);
        if (!in || &r == src) continue;
        CK(cudaStreamWaitEvent(stream_of(r), src->ev_tmp, 0));
        CK(cudaMemcpyAsync(get(r), get(*src), bytes, cudaMemcpyDeviceToDevice, stream_of(r)));
        // the sender must not overwrite its buffer before the copy ran
        CK(cudaEventRecord(r.ev_tmp, stream_of(r)));
        CK(cudaStreamWaitEvent(stream_of(*src), r.ev_tmp, 0));
    }
    return 0;
}

// in-place all-reduce over the world; dtype: 0 f32 sum, 1 f64 sum, 2 f32 max
template <class GetBuf, class GetStream>
int allreduce(mplu_dist* d, int dtype, size_t count, GetBuf get, GetStream stream_of) {
    if (count == 0) return 0;
    if (!d->local_mode) {
        DRank& r = d->ranks[0];
        void* buf = get(r);
        NK(d->nccl->AllReduce(buf, buf, count, dtype == 1 ? ncclFloat64 : ncclFloat32, dtype == 2 ? ncclMax : ncclSum,
                              d->world, stream_of(r)));
        return 0;
    }
    if (d->ranks.size() == 1) return 0;
    DRank& r0 = d->ranks[0];
    cudaStream_t s0 = stream_of(r0);
    const int blocks = (int)((count + 255) / 256);
    for (size_t i = 1; i < d->ranks.size(); ++i) {
        DRank& r = d->ranks[i];
        CK(cudaEventRecord(r.ev_tmp, stream_of(r)));
        CK(cudaStreamWaitEvent(s0, r.ev_tmp, 0));
        if (dtype == 0) sum_into_f32_kernel<<<blocks, 256, 0, s0>>>((float*)get(r0), (const float*)get(r), count);
        else if (dtype == 1) sum_into_f64_kernel<<<blocks, 256, 0, s0>>>((double*)get(r0), (const double*)get(r), count);
        else max_into_f32_kernel<<<blocks, 256, 0, s0>>>((float*)get(r0), (const float*)get(r), count);
    }
    CK(cudaEventRecord(r0.ev_tmp, s0));
    const size_t bytes = count * (dtype == 1 ? 8 : 4);
    for (size_t i = 1; i < d->ranks.size(); ++i) {
        DRank& r = d->ranks[i];
        CK(cudaStreamWaitEvent(stream_of(r), r0.ev_tmp, 0));
        CK(cudaMemcpyAsync(get(r), get(r0), bytes, cudaMemcpyDeviceToDevice, stream_of(r)));
        CK(cudaEventRecord(r.ev_tmp, stream_of(r)));
        CK(cudaStreamWaitEvent(s0, r.ev_tmp, 0));
    }
    return 0;
}

// SMs for the chain lane at a step whose local trailing block is rows x cols: the smallest budget whose estimated chain
// time (diagonal-tile GETRF: latency part + work part, the two panel GEMMs, the panel broadcasts) stays under 3/4 of the
// estimated trailing-update time on the remaining SMs -- early steps of large matrices give almost the whole GPU to
// the update, late steps fall back to the configured maximum.  Rates: measured on B200 (DESIGN.md section 3).
int pick_side_sms(const mplu_dist* d, long long rows, long long cols, int max_side) {
    const double nb = d->nb, sms = d->num_sms;
    const double upd_ms = 2.0 * rows * cols * nb / 1.15e15 * 1e3;
    const double f = nb / 2048.0;
    const double bcast_ms = (rows + cols) * nb * 2.0 / 3.0e11 * 1e3;
    for (int s = 8; s < max_side; s += 8) {
        const double getrf_ms = 1.0 * f + 0.3 * f * f * f * 32.0 / s;
        const double panel_ms = 2.0 * nb * nb * (rows + cols) / (s * 9.4e12 * 0.6) * 1e3;
        if (getrf_ms + panel_ms + bcast_ms <= 0.75 * upd_ms * sms / (sms - s)) return s;
    }
    return max_side;
}

// ---- factorization schedule ------------------------------------------------------------------------------------
int enqueue_dist_factorization(mplu_dist* d) {
    const int nb = d->nb, T = d->T, P = d->P, Q = d->Q;
    const int bf16 = d->opts.precision == MPLU_BF16;
    // side_sms > 0: fixed chain-lane budget (default 32); side_sms < 0: adaptive per step up to |side_sms| (measured
    // slower on power-capped boxes, where the trailing GEMM does not speed up with more SMs: 900 vs 874 ms at n=131072, N=2)
    const bool adaptive = d->opts.side_sms < 0;
    int side_sms = d->opts.side_sms > 0 ? d->opts.side_sms : (adaptive ? -d->opts.side_sms : 32);
    side_sms -= side_sms % 2;
    const bool two = d->opts.lookahead != 0 && side_sms >= 2 && side_sms <= d->num_sms - 16;
    auto chain_of = [](DRank& r) { return r.chain; };

    // first touch: fp32 working copy, global |A| max, global row sums -> ||A||_inf; scales; full 16-bit shadow
    for (auto& r : d->ranks) {
        CK(cudaMemsetAsync(r.ctx->status, 0, sizeof(int), r.chain));
        CK(cudaMemsetAsync(r.dctx->status, 0, sizeof(int), r.chain));
        CK(cudaMemsetAsync(r.ctx->amax, 0, sizeof(float), r.chain));
        CK(cudaMemsetAsync(r.rowsum, 0, d->n * sizeof(double), r.chain));
        if (r.mloc > 0 && r.nloc > 0) {
            dim3 grid((unsigned)((r.mloc + 255) / 256), 32);
            local_first_touch_kernel<<<grid, 256, 0, r.chain>>>(r.A, r.lda, (int)r.mloc, (int)r.nloc, r.W, r.mloc,
                                                                 r.ctx->amax, r.rowsum, nb, P, r.p);
        }
    }
    CKI(allreduce(d, 2, 1, [](DRank& r) { return (void*)r.ctx->amax; }, chain_of));
    CKI(allreduce(d, 1, (size_t)d->n, [](DRank& r) { return (void*)r.rowsum; }, chain_of));
    for (auto& r : d->ranks) {
        CKI(launch_column_absmax(r.rowsum, d->n, d->n, 1, r.anorm, r.chain));
        CKI(launch_scales(r.ctx->amax, r.ctx->scales, d->opts.a_exp, d->opts.l_exp, bf16, r.chain));
        CK(cudaMemcpyAsync(r.dctx->scales, r.ctx->scales, SC_COUNT * sizeof(float), cudaMemcpyDeviceToDevice, r.chain));
        if (r.mloc > 0 && r.nloc > 0)
            CKI(launch_shadow_cast(r.W, r.mloc, r.Wh, r.mloc, (int)r.mloc, (int)r.nloc, r.ctx->scales + SC_A, bf16,
                                   r.ctx->status, r.chain));
        CK(cudaEventRecord(r.ev_chain, r.chain));
        CK(cudaStreamWaitEvent(r.bulk, r.ev_chain, 0));
        d->kernel_launches += 4;
    }

    std::vector<int> side(d->ranks.size(), side_sms);
    for (int k = 0; k < T; ++k) {
        const int pk = k % P, qk = k % Q, b = k & 1;
        for (size_t i = 0; i < d->ranks.size(); ++i) {
            DRank& r = d->ranks[i];
            const long long rows = r.mloc - (long long)cnt_le(k, P, r.p) * nb, cols = r.nloc - (long long)cnt_le(k, Q, r.q) * nb;
            side[i] = (two && adaptive) ? pick_side_sms(d, rows > 0 ? rows : 0, cols > 0 ? cols : 0, side_sms) : side_sms;
        }
        // ---- chain lane: GETRF on the owner
        for (auto& r : d->ranks) {
            if (r.p != pk || r.q != qk) continue;
            if (k > 0) CK(cudaStreamWaitEvent(r.chain, r.ev_d, 0));  // the diagonal tile carries update k-1
            const long long ik = k / P, jk = k / Q;
            mplu_context* dc = r.dctx;
            float* tile = r.W + ik * nb + jk * nb * r.mloc;
            CK(cudaMemcpy2DAsync(dc->W, (size_t)nb * sizeof(float), tile, (size_t)r.mloc * sizeof(float),
                                 (size_t)nb * sizeof(float), nb, cudaMemcpyDeviceToDevice, r.chain));
            dc->gemm_launches = dc->kernel_launches = 0;
            dc->opts.max_sms = two ? side[&r - &d->ranks[0]] : 0;
            CKI(getrf_resident_tile(dc, r.chain, nb));
            d->gemm_launches += dc->gemm_launches;
            d->kernel_launches += dc->kernel_launches + 1;
            CK(cudaMemcpy2DAsync(tile, (size_t)r.mloc * sizeof(float), dc->W, (size_t)nb * sizeof(float),
                                 (size_t)nb * sizeof(float), nb, cudaMemcpyDeviceToDevice, r.chain));
            // publish into this rank's slots of the replicated stores and the step's inverse buffers
            CK(cudaMemcpyAsync(r.Dw + (size_t)k * nb * nb, dc->W, (size_t)nb * nb * sizeof(float), cudaMemcpyDeviceToDevice, r.chain));
            CK(cudaMemcpyAsync(r.Dl32 + (size_t)k * nb * kDiagBlock, dc->Linv32, (size_t)nb * kDiagBlock * sizeof(float), cudaMemcpyDeviceToDevice, r.chain));
            CK(cudaMemcpyAsync(r.Du32 + (size_t)k * nb * kDiagBlock, dc->Uinv32, (size_t)nb * kDiagBlock * sizeof(float), cudaMemcpyDeviceToDevice, r.chain));
            CK(cudaMemcpy2DAsync(r.InvL[b], (size_t)nb * 2, dc->Linv16, (size_t)dc->cap_nb * 2, (size_t)nb * 2, nb, cudaMemcpyDeviceToDevice, r.chain));
            CK(cudaMemcpy2DAsync(r.InvU[b], (size_t)nb * 2, dc->Uinv16, (size_t)dc->cap_nb * 2, (size_t)nb * 2, nb, cudaMemcpyDeviceToDevice, r.chain));
            CK(cudaMemcpyAsync(r.tsc[b], dc->inv_scales, 4 * sizeof(float), cudaMemcpyDeviceToDevice, r.chain));
        }
        // ---- broadcasts of the tile's results
        const int owner = pk * Q + qk;
        if (!d->local_mode) NK(d->nccl->GroupStart());
        CKI(bcast(d, 0, 0, owner, (size_t)nb * nb * sizeof(float), [&](DRank& r) { return (void*)(r.Dw + (size_t)k * nb * nb); }, chain_of));
        CKI(bcast(d, 0, 0, owner, (size_t)nb * kDiagBlock * sizeof(float), [&](DRank& r) { return (void*)(r.Dl32 + (size_t)k * nb * kDiagBlock); }, chain_of));
        CKI(bcast(d, 0, 0, owner, (size_t)nb * kDiagBlock * sizeof(float), [&](DRank& r) { return (void*)(r.Du32 + (size_t)k * nb * kDiagBlock); }, chain_of));
        CKI(bcast(d, 0, 0, owner, 4 * sizeof(float), [&](DRank& r) { return (void*)r.tsc[b]; }, chain_of));
        CKI(bcast(d, 1, pk, qk, (size_t)nb * nb * 2, [&](DRank& r) { return (void*)r.InvL[b]; }, chain_of));
        CKI(bcast(d, 2, qk, pk, (size_t)nb * nb * 2, [&](DRank& r) { return (void*)r.InvU[b]; }, chain_of));
        if (!d->local_mode) NK(d->nccl->GroupEnd());
        if (k == T - 1) break;

        // ---- panel solves on the owner's process column / row, into compact panel buffers
        for (auto& r : d->ranks) {
            const int ilo = cnt_le(k, P, r.p), jlo = cnt_le(k, Q, r.q);
            const long long rows = r.mloc - (long long)ilo * nb, cols = r.nloc - (long long)jlo * nb;
            if (k > 0) CK(cudaStreamWaitEvent(r.chain, r.ev_e1, 0));  // tile column / row k carry update k-1
            // SM budget of the panel GEMMs: the chain lane's share while the previous step's trailing update is the
            // longer job, (almost) the whole GPU once the schedule is chain-bound and the bulk lane would idle anyway
            int panel_sms = 0;
            if (two) {
                const int sd = side[&r - &d->ranks[0]];
                const double upd_ms = 2.0 * (double)(rows + nb) * (double)(cols + nb) * nb / 1.0e15 * 1e3;
                const double pan_ms = 2.0 * (double)nb * nb * ((r.q == qk ? rows : 0) + (r.p == pk ? cols : 0)) / (sd * 9.4e12 * 0.6) * 1e3;
                panel_sms = (pan_ms + 1.5 > upd_ms) ? d->num_sms - 8 : sd;
            }
            const Lane ln{r.chain, panel_sms};
            if (k >= 2) CK(cudaStreamWaitEvent(r.chain, r.ev_panel[b], 0));  // update k-2 has consumed buffers b
            if (rows > 0) CKI(make_operand(&r.opLp[b], r.Lp[b], (uint64_t)rows, (uint64_t)nb, (uint64_t)rows));
            if (r.q == qk && rows > 0) {
                const long long jk = k / Q;
                GemmCall g{&r.opWh, (int)(ilo * nb), (int)(jk * nb), &r.opInvU[b], 0, 0, (int)rows, nb, nb,
                           r.W + (long long)ilo * nb + jk * nb * r.mloc, r.mloc, false,
                           r.Lp[b], rows, (int)rows, nb, 1.f, r.ctx->scales + SC_A_INV, r.tsc[b] + 3, r.ctx->scales + SC_L,
                           TRI_B_UPPER};
                CKI(run_gemm(r.ctx, ln, g));
            }
            if (r.p == pk && cols > 0) {
                const long long ik = k / P;
                GemmCall g{&r.opInvL[b], 0, 0, &r.opWh, (int)(ik * nb), (int)(jlo * nb), nb, (int)cols, nb,
                           r.W + ik * nb + (long long)jlo * nb * r.mloc, r.mloc, false,
                           r.Up[b] + (long long)jlo * nb * nb, nb, nb, (int)cols, 1.f, r.tsc[b] + 1,
                           r.ctx->scales + SC_A_INV, r.ctx->scales + SC_A, TRI_A_LOWER};
                CKI(run_gemm(r.ctx, ln, g));
            }
        }
        // ---- panel broadcasts: L panel along each process row (root column qk), U panel along each process column
        if (!d->local_mode) NK(d->nccl->GroupStart());
        for (int p = 0; p < P; ++p) {
            const long long rows = (long long)(tiles_local(T, P, p) - cnt_le(k, P, p)) * nb;
            if (rows > 0)
                CKI(bcast(d, 1, p, qk, (size_t)rows * nb * 2, [&](DRank& r) { return (void*)r.Lp[b]; }, chain_of));
        }
        for (int q = 0; q < Q; ++q) {
            const int jlo = cnt_le(k, Q, q);
            const long long cols = (long long)(tiles_local(T, Q, q) - jlo) * nb;
            if (cols > 0)
                CKI(bcast(d, 2, q, pk, (size_t)cols * nb * 2,
                          [&](DRank& r) { return (void*)(r.Up[b] + (long long)jlo * nb * nb); }, chain_of));
        }
        if (!d->local_mode) NK(d->nccl->GroupEnd());

        // ---- trailing update: next tile column and tile row first (16-bit shadows for step k+1), then the rest
        const int pn = (k + 1) % P, qn = (k + 1) % Q;
        for (auto& r : d->ranks) {
            const int ilo = cnt_le(k, P, r.p), jlo = cnt_le(k, Q, r.q);
            const long long rows = r.mloc - (long long)ilo * nb, cols = r.nloc - (long long)jlo * nb;
            CK(cudaEventRecord(r.ev_chain, r.chain));
            CK(cudaStreamWaitEvent(r.bulk, r.ev_chain, 0));
            if (rows <= 0 || cols <= 0) {
                CK(cudaEventRecord(r.ev_d, r.bulk));
                CK(cudaEventRecord(r.ev_e1, r.bulk));
                CK(cudaEventRecord(r.ev_panel[b], r.bulk));
                continue;
            }
            const Lane lb{r.bulk, two ? d->num_sms - side[&r - &d->ranks[0]] : 0};
            const float* alpha = r.ctx->scales + SC_NEG_LA_INV;
            const float* hs = r.ctx->scales + SC_A;
            auto update = [&](long long r0, long long r1, long long c0, long long c1, bool shadow) {
                // local rows [r0, r1), local columns [c0, c1)
                if (r1 <= r0 || c1 <= c0) return 0;
                GemmCall g{&r.opLp[b], (int)(r0 - (long long)ilo * nb), 0, &r.opUp[b], 0, (int)c0,
                           (int)(r1 - r0), (int)(c1 - c0), nb, r.W + r0 + c0 * r.mloc, r.mloc, true,
                           r.Wh + r0 + c0 * r.mloc, r.mloc, shadow ? (int)(r1 - r0) : 0, shadow ? (int)(c1 - c0) : 0,
                           1.f, alpha, nullptr, hs};
                return run_gemm(r.ctx, lb, g);
            };
            const long long R0 = (long long)ilo * nb, C0 = (long long)jlo * nb;
            long long c_rest = C0, r_rest = R0;
            if (r.q == qn && r.p == pn) {  // owns the next diagonal tile: update it first, its GETRF heads the next step
                CKI(update(R0, R0 + nb, C0, C0 + nb, true));
                CK(cudaEventRecord(r.ev_d, r.bulk));
                CKI(update(R0 + nb, r.mloc, C0, C0 + nb, true));
                c_rest = C0 + nb;
            } else if (r.q == qn) {  // owns tile column k+1: first local tile column of the region
                CKI(update(R0, r.mloc, C0, C0 + nb, true));
                c_rest = C0 + nb;
            }
            if (!(r.q == qn && r.p == pn)) CK(cudaEventRecord(r.ev_d, r.bulk));
            if (r.p == pn) {  // owns tile row k+1
                CKI(update(R0, R0 + nb, c_rest, r.nloc, true));
                r_rest = R0 + nb;
            }
            CK(cudaEventRecord(r.ev_e1, r.bulk));
            const bool timed = (&r == &d->ranks[0]) && r.mloc > r_rest && r.nloc > c_rest;
            if (timed) {
                if ((int)d->trail_ev.size() < 2 * (d->trail_count + 1)) {
                    cudaEvent_t a, bb;
                    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&bb));
                    d->trail_ev.push_back(a); d->trail_ev.push_back(bb);
                }
                CK(cudaEventRecord(d->trail_ev[2 * d->trail_count], r.bulk));
            }
            CKI(update(r_rest, r.mloc, c_rest, r.nloc, false));
            if (timed) {
                CK(cudaEventRecord(d->trail_ev[2 * d->trail_count + 1], r.bulk));
                d->trail_count++;
                d->trail_flops += 2.0 * (double)(r.mloc - r_rest) * (double)(r.nloc - c_rest) * nb;
                d->trail_bytes += 8.0 * (double)(r.mloc - r_rest) * (double)(r.nloc - c_rest);
            }
            CK(cudaEventRecord(r.ev_panel[b], r.bulk));
        }
    }
    for (auto& r : d->ranks) {
        CK(cudaEventRecord(r.ev_bulk, r.bulk));
        CK(cudaStreamWaitEvent(r.chain, r.ev_bulk, 0));
        d->gemm_launches += r.ctx->gemm_launches;
        d->kernel_launches += r.ctx->kernel_launches;
        r.ctx->gemm_launches = r.ctx->kernel_launches = 0;
    }
    return 0;
}

// ---- refinement ------------------------------------------------------------------------------------------------
// ax = A x over all ranks; r = b - ax; norms
int enqueue_residual(mplu_dist* d, const std::vector<const double*>& b, const std::vector<double*>& x) {
    auto chain_of = [](DRank& r) { return r.chain; };
    for (size_t i = 0; i < d->ranks.size(); ++i) {
        DRank& r = d->ranks[i];
        CK(cudaMemsetAsync(r.ax, 0, d->n * sizeof(double), r.chain));
        if (r.mloc > 0 && r.nloc > 0) {
            const int chunks = (int)std::max<long long>(16, (r.nloc + 4095) / 4096);
            const int per = (int)((r.nloc + chunks - 1) / chunks);
            dim3 grid((unsigned)((r.mloc / 2 + 127) / 128), chunks);
            local_gemv_f64_kernel<<<grid, 128, per * sizeof(double), r.chain>>>(r.A, r.lda, (int)r.mloc, (int)r.nloc, x[i],
                                                                                 r.ax, d->nb, d->P, r.p, d->Q, r.q);
        }
        d->kernel_launches += 2;
    }
    CKI(allreduce(d, 1, (size_t)d->n, [](DRank& r) { return (void*)r.ax; }, chain_of));
    for (size_t i = 0; i < d->ranks.size(); ++i) {
        DRank& r = d->ranks[i];
        CK(cudaMemsetAsync(r.norms, 0, 2 * sizeof(double), r.chain));
        residual_full_kernel<<<(d->n + 255) / 256, 256, 0, r.chain>>>(b[i], r.ax, x[i], r.r, d->n, r.norms);
    }
    return (int)cudaGetLastError();
}

// solve L U dvec = rhs with the distributed fp32 factors; result (float, full length) in r.xv of every rank.
// Right-looking with look-ahead: as soon as the solution block of tile column k is known, the ranks that own tile column k
// fold it into the partial sums `part` of the tile rows it multiplies -- the next D tile rows at once on the chain stream
// (they are needed within D steps), every tile row beyond on the bulk stream (one tall HBM-bound GEMV, off the critical path;
// the chain waits for it D + 1 steps later).  What is left on the dependency chain of a step is one all-reduce of nb
// floats (in place on the tile row's slice of `part`: the ranks outside its process row hold zeros there) and the replicated
// diagonal tile's sweep, which subtracts the reduced sums from its right-hand side itself.  (Round 1 formed each tile
// row's dot products inside the step: memset + tile-row GEMV + all-reduce + right-hand-side kernel + 3 launches of the sweep
// = 0.12 ms per tile step, 38 of the 52 ms the refinement took on 8 GPUs.)
int solve_body(mplu_dist* d, const std::vector<const double*>& rhs);

int enqueue_lu_solve(mplu_dist* d, const std::vector<const double*>& rhs) {
    static const int env_hi = [] { const char* e = getenv("MPLU_DIST_SOLVE_HI"); return e ? atoi(e) : 1; }();
    static const int env_graph = [] { const char* e = getenv("MPLU_DIST_SOLVE_GRAPH"); return e ? atoi(e) : 0; }();
    auto cs_of = [](DRank& r) { return env_hi ? r.hi : r.chain; };
    for (auto& r : d->ranks) {
        // earlier work of both streams (the previous solve's last GEMVs) is ordered before the accumulators are cleared
        CK(cudaEventRecord(r.ev_bulk, r.bulk));
        CK(cudaStreamWaitEvent(cs_of(r), r.ev_bulk, 0));
        if (cs_of(r) != r.chain) {
            CK(cudaEventRecord(r.ev_chain, r.chain));
            CK(cudaStreamWaitEvent(cs_of(r), r.ev_chain, 0));
        }
    }
    // One rank per process (the NCCL case): the ~1000 launches of a solve are the same every time -- replayed as a CUDA graph
    // (the host could not enqueue them as fast as the device runs them: 9 API calls per 50 us step).  The right-hand side goes
    // through a fixed buffer; the first solve on new buffers runs eagerly (NCCL sets its channels up outside a capture).
    const bool graphable = env_graph && !d->px_on && d->opts.use_graph && d->ranks.size() == 1 && cs_of(d->ranks[0]) != d->ranks[0].chain;  // (the exchange's epoch is a kernel argument)
    int rc = 0;
    if (!graphable) {
        rc = solve_body(d, rhs);
    } else {
        DRank& r = d->ranks[0];
        cudaStream_t cs = cs_of(r);
        CK(cudaMemcpyAsync(r.rhsbuf, rhs[0], (size_t)d->n * sizeof(double), cudaMemcpyDeviceToDevice, cs));
        const std::vector<const double*> fixed{r.rhsbuf};
        if (!d->solve_exec && d->solve_uses >= 1) {
            const int before = d->kernel_launches;
            cudaGraph_t graph = nullptr;
            CK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeRelaxed));
            rc = solve_body(d, fixed);
            cudaError_t e = cudaStreamEndCapture(cs, &graph);
            d->solve_launches = d->kernel_launches - before;
            d->kernel_launches = before;
            if (rc == 0 && e == cudaSuccess && graph) e = cudaGraphInstantiate(&d->solve_exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (rc != 0 || e != cudaSuccess) {  // not capturable here: launch by launch from now on
                cudaGetLastError();
                d->solve_exec = nullptr;
                d->solve_uses = -(1 << 30);
                rc = 0;
            }
        }
        d->solve_uses++;
        if (d->solve_exec) {
            CK(cudaGraphLaunch(d->solve_exec, cs));
            d->kernel_launches += d->solve_launches;
        } else {
            rc = solve_body(d, fixed);
        }
    }
    if (rc) return rc;
    for (auto& r : d->ranks) {  // the caller continues on the chain stream
        if (cs_of(r) == r.chain) continue;
        CK(cudaEventRecord(r.ev_chain, cs_of(r)));
        CK(cudaStreamWaitEvent(r.chain, r.ev_chain, 0));
    }
    return (int)cudaGetLastError();
}

int solve_body(mplu_dist* d, const std::vector<const double*>& rhs) {
    const int nb = d->nb, T = d->T, P = d->P, Q = d->Q, n = d->n;
    constexpr int RING = DRank::kSolveRing;
    static const int env_depth = [] { const char* e = getenv("MPLU_DIST_SOLVE_DEPTH"); return e ? atoi(e) : 2; }();
    const int D = env_depth < 1 ? 1 : (env_depth > RING - 2 ? RING - 2 : env_depth);
    // The steps' dependency chain runs on streams of the greatest priority: the sweep of a diagonal tile is a cluster launch
    // whose CTAs need most of an SM each, and behind the thousands of small blocks of a tall GEMV on a stream of equal priority
    // it would only start once that kernel drains.
    static const int env_hi = [] { const char* e = getenv("MPLU_DIST_SOLVE_HI"); return e ? atoi(e) : 1; }();
    static const int env_far = [] { const char* e = getenv("MPLU_DIST_SOLVE_FAR"); return e ? atoi(e) : 1; }();
    static const int env_plain = [] { const char* e = getenv("MPLU_DIST_SOLVE_PLAIN"); return e ? atoi(e) : 1; }();
    auto cs_of = [](DRank& r) { return env_hi ? r.hi : r.chain; };
    // Partial sums of a tile row reach every rank through ncclAllReduce (default) or, with MPLU_DIST_PEER_EXCHANGE=1, through
    // peer memory (px_send_kernel -> the sweep's own wait).  With the peer exchange the sweeps have the stream cs to
    // themselves: sweep k+1 is launched behind sweep k, is resident (tile loads under way) and polling its slots while the
    // GEMVs and sends of step k run on the stream gs.
    const bool px = d->px_on && d->ranks.size() == 1 && !d->solve_exec && env_hi && 2 * (size_t)T * Q <= kPxFlagWords &&
                    2 * (size_t)T * Q * nb <= kPxDataFloats;
    if (px) ++d->px_epoch;
    // MPLU_DIST_TILE_CHAIN=1 (with the peer exchange): ALL tile sweeps of the solve are one persistent launch on cs
    // (launch_tile_chain): nb/128 CTAs that stay resident, poll the exchange slots of the next tile row and count their steps
    // in r.ready; the GEMVs run on gs / bulk, launched ahead, and wait for those counters on the device.
    static const int env_chain = [] { const char* e = getenv("MPLU_DIST_TILE_CHAIN"); return e ? atoi(e) : 0; }();
    const bool chain = px && env_chain && nb / kDiagBlock <= 64;
    auto gs_of = [&](DRank& r) { return px ? r.hi2 : cs_of(r); };
    std::vector<char> far_on(d->ranks.size() * RING, 0), far_any(d->ranks.size(), 0);
    const int sweep_flags = SWEEP_PREPARED | (env_plain ? SWEEP_PLAIN_LAUNCH : 0);
    for (auto& r : d->ranks) {
        // once per solve instead of once per tile step: partial sums cleared, solution vectors NaN (the sweeps' consumers poll
        // the data), the tile sweeps' step counters at their first step (0 forward, nb/128 backward)
        CK(cudaMemsetAsync(r.part, 0, 2 * (size_t)n * sizeof(float), cs_of(r)));
        CK(cudaMemsetAsync(r.yv, 0xFF, (size_t)n * sizeof(float), cs_of(r)));
        CK(cudaMemsetAsync(r.xv, 0xFF, (size_t)n * sizeof(float), cs_of(r)));
        fill_ready_kernel<<<(2 * T + 255) / 256, 256, 0, cs_of(r)>>>(r.ready, T, (unsigned)(nb / kDiagBlock));
        if (gs_of(r) != cs_of(r)) {
            CK(cudaEventRecord(r.ev_swp[RING - 1], cs_of(r)));
            CK(cudaStreamWaitEvent(gs_of(r), r.ev_swp[RING - 1], 0));
            if (chain) CK(cudaStreamWaitEvent(r.bulk, r.ev_swp[RING - 1], 0));  // (its GEMVs wait on the device, not for events)
        }
    }
    // MPLU_DIST_SOLVE_TIMING=1 (development): the first hosted rank's average time per tile step of its first eager solves
    static const int env_timing = [] { const char* e = getenv("MPLU_DIST_SOLVE_TIMING"); return e ? atoi(e) : 0; }();
    static int timed_solves = 0;
    const bool timing = env_timing && timed_solves < 3;
    cudaEvent_t tev[2] = {nullptr, nullptr};
    if (timing) {
        CK(cudaEventCreate(&tev[0])); CK(cudaEventCreate(&tev[1]));
        CK(cudaEventRecord(tev[0], cs_of(d->ranks[0])));
    }
    if (chain) {  // every tile sweep of this solve: one persistent launch on cs
        DRank& r = d->ranks[0];
        if (!d->px_started_h && cudaHostAlloc(&d->px_started_h, sizeof(unsigned), cudaHostAllocMapped) == cudaSuccess)
            cudaHostGetDevicePointer(&d->px_started_d, d->px_started_h, 0);
        cudaGetLastError();
        const TileChain tc{2 * T, T, nb, r.Dw, r.Dl32, r.Du32, rhs[0], r.yv, r.xv, r.ready, d->px_mine, Q, d->px_epoch, d->px_dbg, d->px_started_d};
        if (d->px_started_h) *(volatile unsigned*)d->px_started_h = 0;
        CKI(launch_tile_chain(tc, cs_of(r)));
        d->kernel_launches++;
        // The GEMVs below wait for this launch ON THE DEVICE: were thousands of their blocks resident first, its CTAs (most of
        // an SM each) would find no room and everybody would wait.  Once per solve the host waits until all of them run.
        if (d->px_started_d) {
            const unsigned want = (unsigned)(nb / kDiagBlock);
            for (long long spin = 0; *(volatile unsigned*)d->px_started_h < want && spin < 2000000000LL; ++spin) {}
        }
    }
    for (int sweep = 0; sweep < 2; ++sweep) {
        for (int kk = 0; kk < T; ++kk) {
            const int k = sweep == 0 ? kk : T - 1 - kk;
            const size_t off = (size_t)sweep * n + (size_t)k * nb;
            // the tall GEMVs that touch tile row k: the newest one belongs to the step D + 1 back
            if (kk >= D + 1)
                for (size_t i = 0; i < d->ranks.size(); ++i)
                    if (far_on[i * RING + (kk - D - 1) % RING])
                        CK(cudaStreamWaitEvent(gs_of(d->ranks[i]), d->ranks[i].ev_far[(kk - D - 1) % RING], 0));
            if (kk > 0 && px) {
                DRank& r = d->ranks[0];
                if (r.p == k % P) {
                    px_send_kernel<<<d->nranks, 256, 0, gs_of(r)>>>(r.part + off, d->px_peers, ((size_t)sweep * T + k) * Q + r.q, nb, d->px_epoch);
                    d->kernel_launches++;
                }
            } else if (kk > 0) {
                CKI(allreduce(d, 0, (size_t)nb, [&](DRank& r) { return (void*)(r.part + off); }, cs_of));
            }
            for (size_t i = 0; i < d->ranks.size() && !chain; ++i) {
                DRank& r = d->ranks[i];
                const float* Dk = r.Dw + (size_t)k * nb * nb;
                const float* Li = r.Dl32 + (size_t)k * nb * kDiagBlock;
                const float* Ui = r.Du32 + (size_t)k * nb * kDiagBlock;
                const bool fused = px && kk > 0;  // the sweep itself waits for the peers' slots and adds them up
                const float* sub = (kk > 0 && !fused) ? r.part + off : nullptr;
                const SweepPx spx{d->px_mine, ((unsigned long long)sweep * T + k) * Q, Q, nb, d->px_epoch};
                const SweepPx* pxp = fused ? &spx : nullptr;
                if (sweep == 0)
                    CKI(launch_lu_sweep(Dk, nb, nb, nb, Li, Ui, rhs[i] + (size_t)k * nb, r.yv + (size_t)k * nb, nullptr, nullptr,
                                        nullptr, r.ready + k, 1, cs_of(r), sub, sweep_flags, pxp));
                else
                    CKI(launch_lu_sweep(Dk, nb, nb, nb, Li, Ui, nullptr, r.yv + (size_t)k * nb, r.xv + (size_t)k * nb, nullptr,
                                        nullptr, r.ready + T + k, 2, cs_of(r), sub, sweep_flags, pxp));
                d->kernel_launches += 1;
                if (gs_of(r) != cs_of(r) && kk < T - 1) {  // the GEMVs of this step read the block just solved
                    CK(cudaEventRecord(r.ev_swp[kk % (RING - 1)], cs_of(r)));
                    CK(cudaStreamWaitEvent(gs_of(r), r.ev_swp[kk % (RING - 1)], 0));
                }
            }
            if (kk == T - 1) break;
            // tile column k times its solution block, on the ranks of process column k mod Q
            for (size_t i = 0; i < d->ranks.size(); ++i) {
                DRank& r = d->ranks[i];
                far_on[i * RING + kk % RING] = 0;
                if (r.q != k % Q || r.mloc <= 0 || r.nloc <= 0) continue;
                int near0, near1, far0, far1;  // local tile rows
                if (sweep == 0) {  // global tile rows (k, k + D] and (k + D, T)
                    near0 = cnt_le(k, P, r.p); near1 = cnt_le(std::min(k + D, T - 1), P, r.p);
                    far0 = near1; far1 = r.mt;
                } else {           // global tile rows [k - D, k) and [0, k - D)
                    near0 = cnt_lt(std::max(k - D, 0), P, r.p); near1 = cnt_lt(k, P, r.p);
                    far0 = 0; far1 = near0;
                }
                const float* v = (sweep == 0 ? r.yv : r.xv) + (size_t)k * nb;
                float* part = r.part + (size_t)sweep * n;
                const int c0 = (k / Q) * nb;
                // with the tile chain the GEMVs are launched ahead and wait for tile sweep (sweep, k) on the device
                const unsigned* wf = chain ? r.ready + (size_t)sweep * T + k : nullptr;
                const unsigned wv = (unsigned)((sweep + 1) * (nb / kDiagBlock));
                auto gemv = [&](int t0, int t1, cudaStream_t st) {
                    const int r0 = t0 * nb, r1 = t1 * nb;
                    dim3 grid((unsigned)((r1 - r0) / 128), (unsigned)(nb / 128));
                    tile_col_gemv_kernel<<<grid, 256, 0, st>>>(r.W, r.mloc, r0, r1, c0, v, part, nb, P, r.p, wf, wv, d->px_dbg);
                    d->kernel_launches++;
                };
                if (near1 > near0) gemv(near0, near1, gs_of(r));
                if (far1 > far0 && !env_far) gemv(far0, far1, gs_of(r));  // experiment: everything in stream order
                else if (far1 > far0) {
                    if (!chain) {
                        CK(cudaEventRecord(r.ev_sol[kk % RING], gs_of(r)));
                        CK(cudaStreamWaitEvent(r.bulk, r.ev_sol[kk % RING], 0));
                    }
                    gemv(far0, far1, r.bulk);
                    CK(cudaEventRecord(r.ev_far[kk % RING], r.bulk));
                    far_on[i * RING + kk % RING] = 1;
                    far_any[i] = 1;
                }
            }
        }
    }
    if (timing) {
        ++timed_solves;
        CK(cudaEventRecord(tev[1], cs_of(d->ranks[0])));
        CK(cudaEventSynchronize(tev[1]));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, tev[0], tev[1]);
        unsigned dbg = 0;
        if (d->px_dbg) cudaMemcpy(&dbg, d->px_dbg, sizeof(dbg), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[mplu dist solve timing] rank %d: %d tile steps, %.1f us per step (%s%s), timed-out waits 0x%x\n", d->rank, 2 * T,
                1e3 * ms / (2 * T), px ? "peer exchange" : "ncclAllReduce / local copies", chain ? ", tile chain" : "", dbg);
        cudaEventDestroy(tev[0]); cudaEventDestroy(tev[1]);
    }
    for (size_t i = 0; i < d->ranks.size(); ++i) {  // the other streams' work belongs to this solve (and joins a capture)
        DRank& r = d->ranks[i];
        if (gs_of(r) != cs_of(r)) {
            CK(cudaEventRecord(r.ev_swp[RING - 1], gs_of(r)));
            CK(cudaStreamWaitEvent(cs_of(r), r.ev_swp[RING - 1], 0));
        }
        if (!far_any[i]) continue;
        CK(cudaEventRecord(r.ev_bulk, r.bulk));
        CK(cudaStreamWaitEvent(cs_of(r), r.ev_bulk, 0));
    }
    return (int)cudaGetLastError();
}

}  // namespace

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

int mplu_dist_unique_id(void* id128) {
    NcclApi* api = nccl_api();
    if (!api || !id128) return MPLU_E_NCCL;
    ncclUniqueId id;
    NK(api->GetUniqueId(&id));
    memcpy(id128, &id, sizeof(id));
    return 0;
}

void mplu_dist_destroy(mplu_dist* d);

static int dist_create_common(mplu_dist* d, int device, int P, int Q) {
    d->device = device;
    d->P = P;
    d->Q = Q;
    CK(cudaSetDevice(device));
    CK(cudaDeviceGetAttribute(&d->num_sms, cudaDevAttrMultiProcessorCount, device));
    mplu_default_options(&d->opts);
    CK(cudaEventCreate(&d->ev0)); CK(cudaEventCreate(&d->ev1)); CK(cudaEventCreate(&d->ev2));
    {   // The tile chain (MPLU_DIST_TILE_CHAIN) is a kernel that stays resident and WAITS for these two: with CUDA's lazy
        // module loading the first launch of a kernel may have to wait for running kernels to finish, i.e. for the chain's
        // time-outs (found the hard way: every wait of the first solve ran into its 2 s limit).  Load them now.
        cudaFuncAttributes fa;
        CK(cudaFuncGetAttributes(&fa, px_send_kernel));
        CK(cudaFuncGetAttributes(&fa, tile_col_gemv_kernel));
    }
    for (auto& r : d->ranks) {
        CKI(mplu_create(&r.ctx, device));
        CKI(mplu_create(&r.dctx, device));
        r.chain = r.ctx->stream;
        r.bulk = r.ctx->side;
        {
            int lo = 0, hi = 0;
            CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CK(cudaStreamCreateWithPriority(&r.hi, cudaStreamNonBlocking, hi));
            CK(cudaStreamCreateWithPriority(&r.hi2, cudaStreamNonBlocking, hi));
        }
        cudaEvent_t* evs[] = {&r.ev_tmp, &r.ev_chain, &r.ev_bulk, &r.ev_e1, &r.ev_d, &r.ev_panel[0], &r.ev_panel[1]};
        for (auto e : evs) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        for (int i = 0; i < DRank::kSolveRing; ++i) {
            CK(cudaEventCreateWithFlags(&r.ev_sol[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&r.ev_far[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&r.ev_swp[i], cudaEventDisableTiming));
        }
    }
    return 0;
}

// Peer exchange set-up (collective over the world communicator): every rank allocates its exchange buffer, the CUDA IPC handles
// travel through one byte-wise all-reduce, every rank maps every peer's buffer.  Any failure on any rank is agreed on with a
// second all-reduce and leaves all ranks on ncclAllReduce.  Opt-in (MPLU_DIST_PEER_EXCHANGE=1, the same on every rank).
static void px_teardown(mplu_dist* d) {
    for (void* p : d->px_opened) cudaIpcCloseMemHandle(p);
    d->px_opened.clear();
    cudaFree(d->px_peers); d->px_peers = nullptr;
    cudaFree(d->px_mine); d->px_mine = nullptr;
    cudaFree(d->px_dbg); d->px_dbg = nullptr;
    if (d->px_started_h) cudaFreeHost(d->px_started_h);
    d->px_started_h = d->px_started_d = nullptr;
    d->px_on = false;
}

static int px_setup(mplu_dist* d) {
    const char* env = getenv("MPLU_DIST_PEER_EXCHANGE");
    const int nr = d->nranks;
    cudaStream_t st = d->ranks[0].chain;
    int fail = (env && env[0] == '1') ? 0 : 1;  // opt-in: measured 69 us per tile step against 64 with ncclAllReduce (2 GPUs)
    const size_t bytes = (kPxFlagWords + kPxDataFloats) * sizeof(float);
    cudaIpcMemHandle_t h;
    memset(&h, 0, sizeof(h));
    if (!fail && cudaMalloc(&d->px_mine, bytes) != cudaSuccess) fail = 1;
    if (!fail && cudaMemset(d->px_mine, 0, kPxFlagWords * sizeof(unsigned)) != cudaSuccess) fail = 1;
    if (!fail && cudaIpcGetMemHandle(&h, d->px_mine) != cudaSuccess) fail = 1;
    if (!fail && (cudaMalloc(&d->px_dbg, sizeof(unsigned)) != cudaSuccess || cudaMemset(d->px_dbg, 0, sizeof(unsigned)) != cudaSuccess)) fail = 1;
    cudaGetLastError();
    // table: nr handles + one int of failure votes
    const size_t hb = sizeof(cudaIpcMemHandle_t);
    unsigned char* dtab = nullptr;
    CK(cudaMalloc(&dtab, nr * hb + 2 * sizeof(int)));
    CK(cudaMemsetAsync(dtab, 0, nr * hb + 2 * sizeof(int), st));
    int* dvote = reinterpret_cast<int*>(dtab + nr * hb);
    auto agree = [&](int mine, int slot, int* total) -> int {  // sum of the ranks' votes
        CK(cudaMemcpyAsync(dvote + slot, &mine, sizeof(int), cudaMemcpyHostToDevice, st));
        NK(d->nccl->AllReduce(dvote + slot, dvote + slot, 1, ncclInt32, ncclSum, d->world, st));
        CK(cudaMemcpyAsync(total, dvote + slot, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return 0;
    };
    if (!fail) CK(cudaMemcpyAsync(dtab + d->rank * hb, &h, hb, cudaMemcpyHostToDevice, st));
    NK(d->nccl->AllReduce(dtab, dtab, nr * hb, ncclUint8, ncclSum, d->world, st));
    int total = 0;
    int rc = agree(fail, 0, &total);
    if (rc) { cudaFree(dtab); px_teardown(d); return rc; }
    std::vector<float*> peers((size_t)nr, nullptr);
    if (total == 0) {
        std::vector<cudaIpcMemHandle_t> hs((size_t)nr);
        CK(cudaMemcpy(hs.data(), dtab, nr * hb, cudaMemcpyDeviceToHost));
        for (int i = 0; i < nr && !fail; ++i) {
            if (i == d->rank) { peers[i] = d->px_mine; continue; }
            void* ptr = nullptr;
            if (cudaIpcOpenMemHandle(&ptr, hs[i], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { fail = 1; cudaGetLastError(); break; }
            d->px_opened.push_back(ptr);
            peers[i] = static_cast<float*>(ptr);
        }
        if (!fail && cudaMalloc(&d->px_peers, nr * sizeof(float*)) != cudaSuccess) fail = 1;
        if (!fail && cudaMemcpy(d->px_peers, peers.data(), nr * sizeof(float*), cudaMemcpyHostToDevice) != cudaSuccess) fail = 1;
        rc = agree(fail, 1, &total);
        if (rc) { cudaFree(dtab); px_teardown(d); return rc; }
    }
    cudaFree(dtab);
    if (total == 0) d->px_on = true;
    else px_teardown(d);
    return 0;
}

int mplu_dist_create(mplu_dist** out, int device, int rank, int nranks, int P, int Q, const void* id128) {
    if (!out || P <= 0 || Q <= 0 || P * Q != nranks || rank < 0 || rank >= nranks || !id128) return MPLU_E_ARG;
    NcclApi* api = nccl_api();
    if (!api) return MPLU_E_NCCL;
    mplu_dist* d = new (std::nothrow) mplu_dist();
    if (!d) return MPLU_E_ARG;
    d->local_mode = false;
    d->nccl = api;
    d->rank = rank;
    d->nranks = nranks;
    d->ranks.resize(1);
    d->ranks[0].p = rank / Q;
    d->ranks[0].q = rank % Q;
    // Every rank joins the communicators even when its own device set-up failed (a rank that returned early would
    // leave its peers hung inside the collective ncclCommInitRank); the failure is reported after that.
    const int rc = dist_create_common(d, device, P, Q);
    auto comms = [&]() -> int {
        ncclUniqueId id;
        memcpy(&id, id128, sizeof(id));
        NK(api->CommInitRank(&d->world, nranks, id, rank));
        // process row p: ranks (p, *) ordered by q; process column q: ranks (*, q) ordered by p
        NK(api->CommSplit(d->world, d->ranks[0].p, d->ranks[0].q, &d->rowc, nullptr));
        NK(api->CommSplit(d->world, d->ranks[0].q, d->ranks[0].p, &d->colc, nullptr));
        return 0;
    };
    const int rc2 = comms();
    if (rc || rc2) { mplu_dist_destroy(d); return rc ? rc : rc2; }
    const int rc3 = px_setup(d);
    if (rc3) { mplu_dist_destroy(d); return rc3; }
    *out = d;
    return 0;
}

int mplu_dist_create_local(mplu_dist** out, int device, int P, int Q) {
    if (!out || P <= 0 || Q <= 0 || P * Q > 64) return MPLU_E_ARG;
    mplu_dist* d = new (std::nothrow) mplu_dist();
    if (!d) return MPLU_E_ARG;
    d->local_mode = true;
    d->nranks = P * Q;
    d->ranks.resize((size_t)P * Q);
    for (int p = 0; p < P; ++p)
        for (int q = 0; q < Q; ++q) {
            d->ranks[(size_t)p * Q + q].p = p;
            d->ranks[(size_t)p * Q + q].q = q;
        }
    const int rc = dist_create_common(d, device, P, Q);
    if (rc) { mplu_dist_destroy(d); return rc; }
    {   // a single hosted rank can run the peer-exchange code path against its own buffer (one-GPU testing of that path)
        const char* env = getenv("MPLU_DIST_PEER_EXCHANGE");
        if (env && env[0] == '1' && P * Q == 1) {
            const size_t bytes = (kPxFlagWords + kPxDataFloats) * sizeof(float);
            bool ok = cudaMalloc(&d->px_mine, bytes) == cudaSuccess && cudaMemset(d->px_mine, 0, kPxFlagWords * sizeof(unsigned)) == cudaSuccess &&
                      cudaMalloc(&d->px_peers, sizeof(float*)) == cudaSuccess &&
                      cudaMemcpy(d->px_peers, &d->px_mine, sizeof(float*), cudaMemcpyHostToDevice) == cudaSuccess &&
                      cudaMalloc(&d->px_dbg, sizeof(unsigned)) == cudaSuccess && cudaMemset(d->px_dbg, 0, sizeof(unsigned)) == cudaSuccess;
            if (ok) d->px_on = true;
            else px_teardown(d);
        }
    }
    *out = d;
    return 0;
}

void mplu_dist_release_staging(mplu_dist* d);

void mplu_dist_destroy(mplu_dist* d) {
    if (!d) return;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();
    if (d->solve_exec) { cudaGraphExecDestroy(d->solve_exec); d->solve_exec = nullptr; }
    px_teardown(d);
    for (auto& r : d->ranks) {
        free_rank_work(r);
        cudaEvent_t evs[] = {r.ev_tmp, r.ev_chain, r.ev_bulk, r.ev_e1, r.ev_d, r.ev_panel[0], r.ev_panel[1]};
        for (auto e : evs) if (e) cudaEventDestroy(e);
        for (int i = 0; i < DRank::kSolveRing; ++i) {
            if (r.ev_sol[i]) cudaEventDestroy(r.ev_sol[i]);
            if (r.ev_far[i]) cudaEventDestroy(r.ev_far[i]);
            if (r.ev_swp[i]) cudaEventDestroy(r.ev_swp[i]);
        }
        if (r.hi) cudaStreamDestroy(r.hi);
        if (r.hi2) cudaStreamDestroy(r.hi2);
        mplu_destroy(r.ctx);
        mplu_destroy(r.dctx);
    }
    if (d->nccl) {
        if (d->rowc) d->nccl->CommDestroy(d->rowc);
        if (d->colc) d->nccl->CommDestroy(d->colc);
        if (d->world) d->nccl->CommDestroy(d->world);
    }
    mplu_dist_release_staging(d);
    for (auto e : d->trail_ev) cudaEventDestroy(e);
    cudaEventDestroy(d->ev0); cudaEventDestroy(d->ev1); cudaEventDestroy(d->ev2);
    delete d;
}

int mplu_dist_num_local(const mplu_dist* d) { return d ? (int)d->ranks.size() : 0; }

// local tile-row / tile-column counts of logical rank i of this process for an n x n matrix tiled by nb
int mplu_dist_local_shape(const mplu_dist* d, int i, int n, int nb, int* p, int* q, long long* mloc, long long* nloc) {
    if (!d || i < 0 || i >= (int)d->ranks.size() || nb <= 0 || n % nb) return MPLU_E_ARG;
    const DRank& r = d->ranks[i];
    const int T = n / nb;
    if (p) *p = r.p;
    if (q) *q = r.q;
    if (mloc) *mloc = (long long)tiles_local(T, d->P, r.p) * nb;
    if (nloc) *nloc = (long long)tiles_local(T, d->Q, r.q) * nb;
    return 0;
}

// factor + solve.  dA[i] / lda[i]: local block-cyclic fp64 tiles of logical rank i (column-major, mloc x nloc);
// db[i], dx[i]: full-length (n) right-hand side and solution on every rank.  n % nb == 0, nb % 128 == 0.
int mplu_dist_gesv(mplu_dist* d, int n, int nb, const double* const* dA, const long long* lda,
                   const double* const* db, double* const* dx, const mplu_options* opts, mplu_stats* stats) {
    if (!d || n <= 0 || nb < kDiagBlock || nb % kDiagBlock || n % nb || !dA || !lda || !db || !dx) return MPLU_E_ARG;
    if (opts && opts->equilibrate != 0) return MPLU_E_ARG;  // no equilibration in the block-cyclic solver
    CK(cudaSetDevice(d->device));
    if (opts) d->opts = *opts;
    d->opts.nb = nb;
    const bool realloc = (n != d->n || nb != d->nb);
    d->n = n;
    d->nb = nb;
    d->T = n / nb;
    d->gemm_launches = d->kernel_launches = 0;
    d->trail_count = 0;
    d->trail_flops = d->trail_bytes = 0;
    std::vector<const double*> bv, rv;
    std::vector<double*> xv;
    for (size_t i = 0; i < d->ranks.size(); ++i) {
        DRank& r = d->ranks[i];
        if (realloc) CKI(alloc_rank_work(d, r));
        r.ctx->opts = d->opts;
        r.dctx->opts.precision = d->opts.precision;
        r.dctx->opts.gemm_variant = d->opts.gemm_variant;
        r.dctx->opts.group = d->opts.group;
        r.dctx->opts.pdl = d->opts.pdl;
        r.A = dA[i];
        r.lda = lda[i];
        if (r.mloc > 0 && lda[i] < r.mloc) return MPLU_E_ARG;
        bv.push_back(db[i]);
        xv.push_back(dx[i]);
        rv.push_back(r.r);
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    DRank& r0 = d->ranks[0];
    CK(cudaEventRecord(d->ev0, r0.chain));
    CKI(enqueue_dist_factorization(d));
    CK(cudaEventRecord(d->ev1, r0.chain));

    // ||b||_inf and the first solve x = (LU)^-1 b, then dsgesv's refinement.  Every process takes the decision from its
    // own (identical) copy of the norms.
    RefineOps ops;
    ops.norms = r0.norms;
    ops.anorm = r0.anorm;
    ops.st = r0.chain;
    ops.first_solve = [&]() -> int {
        for (size_t i = 0; i < d->ranks.size(); ++i)
            CKI(launch_column_absmax(bv[i], n, n, 1, d->ranks[i].norms + 2, d->ranks[i].chain));
        CKI(enqueue_lu_solve(d, bv));
        for (size_t i = 0; i < d->ranks.size(); ++i)
            apply_correction_kernel<<<(n + 255) / 256, 256, 0, d->ranks[i].chain>>>(d->ranks[i].xv, xv[i], n, 0);
        return 0;
    };
    ops.residual = [&](bool*) { return enqueue_residual(d, bv, xv); };
    ops.correct = [&](int*) -> int {
        CKI(enqueue_lu_solve(d, rv));
        for (size_t i = 0; i < d->ranks.size(); ++i)
            apply_correction_kernel<<<(n + 255) / 256, 256, 0, d->ranks[i].chain>>>(d->ranks[i].xv, xv[i], n, 1);
        return 0;
    };
    ops.wait = [&]() -> int {
        for (auto& r : d->ranks) CK(cudaStreamSynchronize(r.chain));
        return 0;
    };
    RefineResult res;
    CKI(refine(ops, n, 1, d->opts.max_iters, d->opts.tol, &res));
    CK(cudaEventRecord(d->ev2, r0.chain));
    CK(cudaEventSynchronize(d->ev2));
    int h_status = 0;
    for (auto& r : d->ranks) {
        int s1 = 0, s2 = 0;
        CK(cudaMemcpy(&s1, r.ctx->status, sizeof(int), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(&s2, r.dctx->status, sizeof(int), cudaMemcpyDeviceToHost));
        h_status |= s1 | s2;
    }
    refine_stats(res, n, nullptr, stats);
    if (stats) {
        stats->status_bits = h_status;
        stats->gemm_launches = d->gemm_launches;
        stats->kernel_launches = d->kernel_launches;
        stats->trailing_launches = d->trail_count;
        stats->trailing_flops = d->trail_flops;
        stats->trailing_bytes = d->trail_bytes;
        float tms = 0.f;
        for (int t = 0; t < d->trail_count; ++t) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, d->trail_ev[2 * t], d->trail_ev[2 * t + 1]) == cudaSuccess) tms += ms;
        }
        stats->trailing_ms = tms;
        cudaEventElapsedTime(&stats->factor_ms, d->ev0, d->ev1);
        cudaEventElapsedTime(&stats->solve_ms, d->ev1, d->ev2);
        cudaEventElapsedTime(&stats->total_ms, d->ev0, d->ev2);
    }
    return refine_rc(res.converged, h_status);
}

// Same solve from HOST buffers (pinned or pageable): hA[i] = local block-cyclic fp64 tiles of logical rank i (host,
// column-major, leading dimension lda[i]), hb[i] full right-hand side, hx[i] receives the full solution.  The H2D copies
// of the local tiles and the D2H copy of x are inside the call; stats->h2d_ms / d2h_ms report them.
int mplu_dist_gesv_host(mplu_dist* d, int n, int nb, const double* const* hA, const long long* lda,
                        const double* const* hb, double* const* hx, const mplu_options* opts, mplu_stats* stats) {
    if (!d || n <= 0 || nb < kDiagBlock || nb % kDiagBlock || n % nb || !hA || !lda || !hb || !hx) return MPLU_E_ARG;
    if (opts && opts->equilibrate != 0) return MPLU_E_ARG;
    CK(cudaSetDevice(d->device));
    const size_t L = d->ranks.size();
    if (d->stA.size() != L) { d->stA.assign(L, nullptr); d->stb.assign(L, nullptr); d->stx.assign(L, nullptr); d->stA_cap.assign(L, 0); d->st_n = 0; }
    const int T = n / nb;
    std::vector<long long> ld(L);
    std::vector<const double*> pa(L), pb(L);
    std::vector<double*> px(L);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0, d->ranks[0].chain));
    for (size_t i = 0; i < L; ++i) {
        DRank& r = d->ranks[i];
        const size_t ml = (size_t)tiles_local(T, d->P, r.p) * nb, nl = (size_t)tiles_local(T, d->Q, r.q) * nb;
        const size_t need = (ml ? ml : 1) * (nl ? nl : 1);
        if (need > d->stA_cap[i]) {
            cudaFree(d->stA[i]); d->stA[i] = nullptr; d->stA_cap[i] = 0;
            CK(cudaMalloc(&d->stA[i], need * sizeof(double)));
            d->stA_cap[i] = need;
        }
        if (n > d->st_n || !d->stb[i]) {
            cudaFree(d->stb[i]); cudaFree(d->stx[i]);
            CK(cudaMalloc(&d->stb[i], n * sizeof(double)));
            CK(cudaMalloc(&d->stx[i], n * sizeof(double)));
        }
        if (ml && nl) {
            if (lda[i] < (long long)ml) return MPLU_E_ARG;
            CK(cudaMemcpy2DAsync(d->stA[i], ml * sizeof(double), hA[i], (size_t)lda[i] * sizeof(double), ml * sizeof(double),
                                 nl, cudaMemcpyHostToDevice, r.chain));
        }
        CK(cudaMemcpyAsync(d->stb[i], hb[i], n * sizeof(double), cudaMemcpyHostToDevice, r.chain));
        ld[i] = (long long)(ml ? ml : 1);
        pa[i] = d->stA[i]; pb[i] = d->stb[i]; px[i] = d->stx[i];
    }
    d->st_n = n > d->st_n ? n : d->st_n;
    CK(cudaEventRecord(e1, d->ranks[0].chain));
    int rc = mplu_dist_gesv(d, n, nb, pa.data(), ld.data(), pb.data(), px.data(), opts, stats);
    if (rc != 0 && rc != MPLU_E_NOCONV) { cudaEventDestroy(e0); cudaEventDestroy(e1); return rc; }
    float h2d = 0.f, d2h = 0.f;
    cudaEventElapsedTime(&h2d, e0, e1);
    CK(cudaEventRecord(e0, d->ranks[0].chain));
    for (size_t i = 0; i < L; ++i)
        CK(cudaMemcpyAsync(hx[i], d->stx[i], n * sizeof(double), cudaMemcpyDeviceToHost, d->ranks[i].chain));
    CK(cudaEventRecord(e1, d->ranks[0].chain));
    for (size_t i = 0; i < L; ++i) CK(cudaStreamSynchronize(d->ranks[i].chain));
    cudaEventElapsedTime(&d2h, e0, e1);
    if (stats) { stats->h2d_ms = h2d; stats->d2h_ms = d2h; stats->total_ms += h2d + d2h; }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

// Release the device staging buffers of mplu_dist_gesv_host.
void mplu_dist_release_staging(mplu_dist* d) {
    if (!d) return;
    cudaSetDevice(d->device);
    for (auto& p : d->stA) { cudaFree(p); p = nullptr; }
    for (auto& p : d->stb) { cudaFree(p); p = nullptr; }
    for (auto& p : d->stx) { cudaFree(p); p = nullptr; }
    for (auto& c : d->stA_cap) c = 0;
    d->st_n = 0;
}

// Copy logical rank i's local fp32 factors (L\U in block-cyclic local order, mloc x nloc) widened to fp64.
int mplu_dist_get_local_factors(mplu_dist* d, int i, double* dLU, long long ld) {
    if (!d || i < 0 || i >= (int)d->ranks.size() || !dLU) return MPLU_E_ARG;
    DRank& r = d->ranks[i];
    if (ld < r.mloc) return MPLU_E_ARG;
    std::vector<float> h((size_t)r.mloc * r.nloc);
    CK(cudaMemcpy(h.data(), r.W, h.size() * sizeof(float), cudaMemcpyDeviceToHost));
    std::vector<double> hd(h.size());
    for (size_t e = 0; e < h.size(); ++e) hd[e] = h[e];
    CK(cudaMemcpy2D(dLU, (size_t)ld * sizeof(double), hd.data(), (size_t)r.mloc * sizeof(double),
                    (size_t)r.mloc * sizeof(double), (size_t)r.nloc, cudaMemcpyHostToDevice));
    return 0;
}

}  // extern "C"
