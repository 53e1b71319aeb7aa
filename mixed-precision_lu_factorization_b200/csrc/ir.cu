// Iterative-refinement kernels (fp64 residual, fp32 triangular solves with the stored factors).  The reference has
// no solve / refinement path (SURVEY.md section 0); these follow BASELINE.json's north_star and LAPACK dsgesv's
// structure: r = b - A*x in fp64, L U d = r in the factorization precision, x += d in fp64.
// All of them are HBM-bound: the residual streams 8*n^2 bytes, the solve pair 4*n^2 bytes.
#include "kernels.h"

#include <mutex>
#include "ptx.cuh"

#include <cstdlib>

namespace mplu {

namespace {

constexpr int RES_THREADS = 128;  // each thread owns 2 consecutive rows

// partial[chunk][row] = sum_{c in chunk} A(row,c) * x(c);  kAbs: also abs_partial[chunk][row] = sum |A(row,c)| -- the row
// sums behind ||A||_inf ride in the first residual, which streams all of A anyway, instead of a pass of their own
template <bool kAbs>
__global__ void __launch_bounds__(RES_THREADS)
residual_partial_kernel(const double* __restrict__ A, long long lda, int n, const double* __restrict__ x,
                        double* __restrict__ partial, int cols_per, double* __restrict__ abs_partial) {
    extern __shared__ double xs[];
    const int c0 = blockIdx.y * cols_per;
    const int c1 = min(n, c0 + cols_per);
    for (int c = c0 + threadIdx.x; c < c1; c += RES_THREADS) xs[c - c0] = x[c];
    __syncthreads();
    const int r0 = 2 * (blockIdx.x * RES_THREADS + threadIdx.x);
    if (r0 >= n) return;
    const int nc = c1 - c0;
    const double* Ap = A + r0 + (long long)c0 * lda;
    double a0 = 0.0, a1 = 0.0, s0 = 0.0, s1 = 0.0;
    const bool vec = (r0 + 1 < n) && ((lda & 1) == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
    if (vec) {
        int c = 0;
        for (; c + 8 <= nc; c += 8) {
            double2 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = __ldg(reinterpret_cast<const double2*>(Ap + (long long)(c + u) * lda));
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const double xv = xs[c + u];
                a0 = fma(v[u].x, xv, a0);
                a1 = fma(v[u].y, xv, a1);
                if (kAbs) { s0 += fabs(v[u].x); s1 += fabs(v[u].y); }
            }
        }
        for (; c < nc; ++c) {
            const double2 v = __ldg(reinterpret_cast<const double2*>(Ap + (long long)c * lda));
            a0 = fma(v.x, xs[c], a0);
            a1 = fma(v.y, xs[c], a1);
            if (kAbs) { s0 += fabs(v.x); s1 += fabs(v.y); }
        }
    } else {
        for (int c = 0; c < nc; ++c) {
            const double v0 = __ldg(Ap + (long long)c * lda);
            a0 = fma(v0, xs[c], a0);
            if (kAbs) s0 += fabs(v0);
            if (r0 + 1 < n) {
                const double v1 = __ldg(Ap + 1 + (long long)c * lda);
                a1 = fma(v1, xs[c], a1);
                if (kAbs) s1 += fabs(v1);
            }
        }
    }
    partial[(long long)blockIdx.y * n + r0] = a0;
    if (r0 + 1 < n) partial[(long long)blockIdx.y * n + r0 + 1] = a1;
    if (kAbs) {
        abs_partial[(long long)blockIdx.y * n + r0] = s0;
        if (r0 + 1 < n) abs_partial[(long long)blockIdx.y * n + r0 + 1] = s1;
    }
}

__device__ __forceinline__ void atomic_max_double_nonneg(double* addr, double v) {
    atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

// r = b - sum_chunks partial; norms[0] = max|r|, norms[1] = max|x|   (norms zeroed by the launcher)
__global__ void residual_finish_kernel(const double* __restrict__ partial, int n, int nchunk,
                                       const double* __restrict__ b, const double* __restrict__ x,
                                       double* __restrict__ r, double* norms, const double* __restrict__ abs_partial,
                                       double* anorm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double rv = 0.0, xv = 0.0, av = 0.0;
    if (i < n) {
        double s = 0.0;
        for (int c = 0; c < nchunk; ++c) s += partial[(long long)c * n + i];
        if (abs_partial)
            for (int c = 0; c < nchunk; ++c) av += abs_partial[(long long)c * n + i];
        rv = b[i] - s;
        r[i] = rv;
        rv = fabs(rv);
        xv = fabs(x[i]);
    }
    for (int o = 16; o > 0; o >>= 1) {
        rv = fmax(rv, __shfl_xor_sync(0xffffffffu, rv, o));
        xv = fmax(xv, __shfl_xor_sync(0xffffffffu, xv, o));
        av = fmax(av, __shfl_xor_sync(0xffffffffu, av, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomic_max_double_nonneg(&norms[0], rv);
        atomic_max_double_nonneg(&norms[1], xv);
        if (anorm) atomic_max_double_nonneg(anorm, av);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// lu_solve_kernel: both triangular solves of L U d = rhs in ONE cooperative launch (the previous version launched one
// kernel per 128-column block: 2*n/128 dependent launches per solve, 15 ms of the n = 16384 step).
//
// Work unit ("step") s = one 128-row block of one sweep: s < nblk forward (L y = rhs, block i = s), s >= nblk backward
// (U x = y, block i = 2*nblk-1-s).  A step is a left-looking dot-product form:
//     acc = rhs_i - sum_{j solved before i} W(i,j) * sol_j ;   sol_i = inv(D_i) * acc
// so a CTA streams the 128x128 fp32 tiles of its block row with 128-bit loads issued BEFORE it waits for sol_j, and
// only the last tile + the 64 KiB inverse sit on the dependency chain.  The inverse is simply the LAST ITEM of the tile
// stream: it arrives in the same double-buffered registers (4 rows x 16 columns per thread) and is applied the way a tile
// is, 64 FMAs per thread.  (Round 1 staged it in shared memory and every thread read a 64-entry row of it: 64 KiB through
// the 128 B/clk shared-memory port = 512+ cycles on every one of the 2*n/128 links of the chain.)
// Steps complete strictly in order; `ready` = number of completed steps is published with a release store and polled
// with acquire loads.  CTA c owns steps c, c+G, ... in ascending order and the launch is cooperative (all CTAs are
// co-resident), so every wait is on a step owned by a running CTA.  HBM-bound: 4*n^2 bytes per solve.
// Hand-off of a solved block: the solution vectors are pre-filled with NaN and consumers poll the DATA itself (the 16
// floats a thread needs) instead of the counter: one L2 round trip less on the 2*n/128-step dependency chain and no
// fence + flag store before the next step can start.  The counter is still published and is consulted every 64
// polls, so a genuine NaN in the solution (broken factorization) cannot hang the sweep.
// Step s -> step s+1 is the critical chain (2*n/128 links); consecutive steps belong to consecutive CTAs, which are
// launched as thread-block clusters of 8: the solver of step s also stores its block straight into mailboxes in the
// shared memory of the CTAs that own steps s+1 .. s+3 (DSMEM), which poll their own shared memory for their three
// newest operands instead of L2 (with only the newest one delivered, the second newest -- still in flight through L2
// when the newest arrives -- kept the chain at L2 latency).  Hand-offs across a cluster boundary and all older
// operands (which have slack) go through L2.
constexpr int TSV_THREADS = 256;
constexpr int DBS = kDiagBlock;
constexpr int TSV_SMEM_BYTES = 0;  // the inverse lives in registers
constexpr int TSV_MB = 3;  // mailbox depth: blocks of the TSV_MB preceding steps arrive through DSMEM

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(unsigned* p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float4 ld_relaxed_f4(const float4* p) {
    float4 v;
    asm volatile("ld.relaxed.gpu.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_relaxed_f1(const float* p) {
    float v;
    asm volatile("ld.relaxed.gpu.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_f1(float* p, float v) {
    asm volatile("st.relaxed.gpu.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

__global__ void __launch_bounds__(TSV_THREADS)
lu_solve_kernel(const float* __restrict__ W_, long long ldw, int n, int nblk, const float* __restrict__ Linv_,
                const float* __restrict__ Uinv_, const double* __restrict__ rhs_, float* ysol_, float* xsol_,
                double* __restrict__ d_out, double* __restrict__ x_accum, unsigned* ready_, int s_begin_, int s_end_,
                int use_mbox, const float* __restrict__ sub, const SweepPx px_, const TileChain tc) {
    __shared__ __align__(16) float s_part[8][DBS];
    __shared__ __align__(16) float s_acc[DBS];
    __shared__ __align__(16) float mbox[2][TSV_MB][DBS];  // [owned-step parity][distance-1]: blocks of steps s-1 .. s-TSV_MB
    const int tid = threadIdx.x;
    const int rg = tid & 31, cg = tid >> 5;  // rows 4rg.., columns 16cg.. of a tile
    unsigned seen = 0;
    unsigned crank = 0, csize = 1;
    if (use_mbox) {
        asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
        asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(csize));
        for (int e = tid; e < 2 * TSV_MB * DBS; e += TSV_THREADS) (&mbox[0][0][0])[e] = __int_as_float(0x7fffffff);
        ptx::cluster_sync_all();  // nobody stores into a mailbox that is not initialised yet
    }
    if (tc.count > 0 && tc.started && tid == 0) atomicAdd_system(tc.started, 1u);
    int kown = 0;
    // tc.count > 0: a chain of one-sweep problems (the diagonal tiles of a block-cyclic solve) in this one launch
    const int nprob = tc.count > 0 ? tc.count : 1;
    for (int ts = 0; ts < nprob; ++ts) {
    const float* W = W_; const float* Linv = Linv_; const float* Uinv = Uinv_; const double* rhs = rhs_;
    float* ysol = ysol_; float* xsol = xsol_; unsigned* ready = ready_;
    int s_begin = s_begin_, s_end = s_end_;
    SweepPx px = px_;
    if (tc.count > 0) {
        const int swp = ts / tc.T, kk = ts - swp * tc.T, k = swp == 0 ? kk : tc.T - 1 - kk;
        W = tc.Dw + (size_t)k * tc.nb * tc.nb;
        Linv = tc.Dl32 + (size_t)k * tc.nb * DBS;
        Uinv = tc.Du32 + (size_t)k * tc.nb * DBS;
        rhs = tc.rhs + (size_t)k * tc.nb;
        ysol = tc.yv + (size_t)k * tc.nb;
        xsol = tc.xv + (size_t)k * tc.nb;
        ready = tc.ready + (size_t)swp * tc.T + k;
        s_begin = swp == 0 ? 0 : nblk;
        s_end = swp == 0 ? nblk : 2 * nblk;
        px.base = kk > 0 ? tc.px_base : nullptr;
        px.slot0 = ((unsigned long long)swp * tc.T + k) * tc.Q;
        px.Q = tc.Q; px.nb = tc.nb; px.epoch = tc.epoch;
        seen = 0;
    }
    // steps [s_begin, s_end): [0, 2*nblk) = both sweeps; [0, nblk) forward only; [nblk, 2*nblk) backward only (its
    // right-hand side is then read from ysol and *ready must start at nblk)
    for (int s = s_begin + blockIdx.x; s < s_end; s += gridDim.x, ++kown) {
        const bool back = s >= nblk;
        // step s-d (d <= TSV_MB) was solved by CTA crank-d of this cluster: its block arrives in mbox[kown & 1][d-1]
        auto delivered = [&](int d) { return use_mbox && (int)crank >= d && s - d >= s_begin; };
        volatile float (*mb)[DBS] = mbox[kown & 1];
        const int t = back ? s - nblk : s;         // tiles in this block row
        const int i = back ? nblk - 1 - t : t;     // block row
        const float* solv = back ? xsol : ysol;
        const float* inv = (back ? Uinv : Linv) + (long long)i * DBS * DBS;  // 128 x 128, column-major
        // this row block's right-hand side: fetched NOW, long before the step's turn (loading it after the last operand
        // arrived put one L2/HBM latency on every link of the dependency chain)
        float a_pre = __int_as_float(0x7fffffff), sub_pre = 0.f;
        if (tid < DBS) {
            const int row = i * DBS + tid;
            if (sub) sub_pre = sub[row];  // one-sweep modes: what other block rows already contributed to this right-hand side
            if (back) a_pre = ld_relaxed_f1(ysol + row);  // may still be NaN = not solved yet: polled again below
            else a_pre = (row < n) ? static_cast<float>(rhs[row]) : 0.f;
        }
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        const float* wrow = W + (long long)i * DBS + 4 * rg;
        // 128-bit loads of this thread's 4 rows x 16 columns of tile tt
        // (item t of the stream is the inverse of the diagonal block, same thread layout)
        auto load_tile = [&](float4 (&v)[16], int tt) {
            if (tt < t) {
                const int j = back ? nblk - 1 - tt : tt;
                const float* wp = wrow + ((long long)j * DBS + 16 * cg) * ldw;
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = __ldcs(reinterpret_cast<const float4*>(wp + (long long)q * ldw));
            } else {
                const float* ip = inv + 4 * rg + 16 * cg * DBS;
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = __ldcs(reinterpret_cast<const float4*>(ip + q * DBS));
            }
        };
        // wait for the solution block tile tt multiplies (mailbox for the newest ones, else L2), then accumulate
        auto consume = [&](const float4 (&v)[16], int tt) {
            const int j = back ? nblk - 1 - tt : tt;
            const unsigned need = (back ? nblk : 0) + tt + 1;
            const float4* sp = reinterpret_cast<const float4*>(solv + j * DBS + 16 * cg);
            float sv[16];
            bool got = false;
            if (t - tt <= TSV_MB && delivered(t - tt)) {  // one of the newest operands: poll the local mailbox
                volatile float* m = mb[t - tt - 1];
                for (int spin = 0; spin < (1 << 20) && !got; ++spin) {
                    got = true;
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        sv[q] = m[16 * cg + q];
                        got &= (sv[q] == sv[q]);
                    }
                }
            }
            for (int spin = 0; !got; ++spin) {
                bool pending = false;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 x4 = ld_relaxed_f4(sp + q);
                    sv[4 * q] = x4.x; sv[4 * q + 1] = x4.y; sv[4 * q + 2] = x4.z; sv[4 * q + 3] = x4.w;
                    pending |= (x4.x != x4.x) | (x4.y != x4.y) | (x4.z != x4.z) | (x4.w != x4.w);
                }
                if (!pending || seen >= need) break;
                if ((spin & 63) == 63) seen = ld_acquire_u32(ready);  // a NaN that is data, not "not yet written"
            }
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                acc.x = fmaf(v[q].x, sv[q], acc.x);
                acc.y = fmaf(v[q].y, sv[q], acc.y);
                acc.z = fmaf(v[q].z, sv[q], acc.z);
                acc.w = fmaf(v[q].w, sv[q], acc.w);
            }
        };
        // Everything after the last operand arrived is the dependency chain's link: cross-warp reduction of the tile
        // products, the inverse (already in registers) applied to the 128 sums, cross-warp reduction, hand-off.
        auto finish = [&](const float4 (&vi)[16]) {
            *reinterpret_cast<float4*>(&s_part[cg][4 * rg]) = acc;
            __syncthreads();
            if (tid < DBS) {
                const int row = i * DBS + tid;
                float a = a_pre;
                if (back && a != a) {  // y of this block row must be final (written by the forward sweep of this launch, or given)
                    // y of block row i was solved at forward step i = s - (2t+1): near the turn it sits in a mailbox
                    if (2 * t + 1 <= TSV_MB && delivered(2 * t + 1))
                        for (int spin = 0; spin < (1 << 20) && a != a; ++spin) a = mb[2 * t][tid];
                    for (int spin = 0; a != a; ++spin) {
                        a = ld_relaxed_f1(ysol + row);
                        if (a == a || seen >= (unsigned)nblk) break;
                        if ((spin & 63) == 63) seen = ld_acquire_u32(ready);
                    }
                }
                if (px.base) {  // ... or what the peers' tile columns contributed: wait for their Q slots, add them up
                    const unsigned* f = reinterpret_cast<const unsigned*>(px.base) + px.slot0;
                    const long long t0 = clock64();  // a peer that never arrives must not hang the GPU (the solve then fails to converge)
                    for (int q = 0; q < px.Q; ++q) {
                        unsigned v;
                        do { asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f + q) : "memory"); }
                        while (v != px.epoch && clock64() - t0 < 4000000000LL);
                    }
                    if (tc.dbg && clock64() - t0 >= 4000000000LL) atomicOr(tc.dbg, 1u);
                    for (int q = 0; q < px.Q; ++q) sub_pre += __ldcv(px.base + kPxFlagWords + (px.slot0 + q) * px.nb + row);
                }
                a -= sub_pre;
#pragma unroll
                for (int g = 0; g < 8; ++g) a -= s_part[g][tid];
                s_acc[tid] = a;
            }
            __syncthreads();
            {   // sol_i = inv * acc: this thread's 4 rows x 16 columns of the inverse against s_acc[16 cg ..]
                float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {
                    const float4 sa = *reinterpret_cast<const float4*>(&s_acc[16 * cg + 4 * q4]);
                    const float sq[4] = {sa.x, sa.y, sa.z, sa.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float4 w = vi[4 * q4 + u];
                        o.x = fmaf(w.x, sq[u], o.x);
                        o.y = fmaf(w.y, sq[u], o.y);
                        o.z = fmaf(w.z, sq[u], o.z);
                        o.w = fmaf(w.w, sq[u], o.w);
                    }
                }
                *reinterpret_cast<float4*>(&s_part[cg][4 * rg]) = o;
            }
            __syncthreads();
            if (tid < DBS) {
                float v = 0.f;
#pragma unroll
                for (int g = 0; g < 8; ++g) v += s_part[g][tid];
                const int row = i * DBS + tid;
                if (use_mbox) {  // first of all: hand the block to the owners of the next steps through their shared memory
#pragma unroll
                    for (int d = 1; d <= TSV_MB; ++d)
                        if (crank + d < csize && s + d < s_end) {
                            unsigned remote;
                            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(ptx::smem_u32(&mbox[kown & 1][d - 1][tid])), "r"(crank + d));
                            asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(v) : "memory");
                        }
                }
                if (back) {
                    st_relaxed_f1(xsol + row, v);
                    if (row < n) {
                        if (d_out) d_out[row] = static_cast<double>(v);
                        if (x_accum) x_accum[row] += static_cast<double>(v);
                    }
                } else {
                    st_relaxed_f1(ysol + row, v);
                }
                // off the chain: every delivery is awaited (it may be one this step had no use for) and its slot re-armed
                // (the next delivery into this parity's slots is for this CTA's step after next)
#pragma unroll
                for (int d = 1; d <= TSV_MB; ++d)
                    if (delivered(d)) {
                        float w = mb[d - 1][tid];
                        for (int spin = 0; spin < (1 << 20) && w != w; ++spin) w = mb[d - 1][tid];
                        mb[d - 1][tid] = __int_as_float(0x7fffffff);
                    }
            }
        };
        // Two register buffers: the loads of item tt+1 are in flight while the thread waits for the operand of tile tt.
        // (With a single buffer a CTA that had caught up with the sweep's frontier paid one HBM latency per tile on
        // top of the operand latency and set the pace of the whole dependency chain: 2.4 us per step.)
        {
            float4 va[16], vb[16];
            load_tile(va, 0);
            for (int tt = 0; tt < t; tt += 2) {
                load_tile(vb, tt + 1);  // tt + 1 <= t: a tile, or the inverse
                consume(va, tt);
                if (tt + 1 < t) {
                    load_tile(va, tt + 2);
                    consume(vb, tt + 1);
                }
            }
            if (t & 1) finish(vb); else finish(va);
        }
        __syncthreads();
        if (tid == 0) {
            __threadfence();
            st_release_u32(ready, (unsigned)(s + 1));
        }
    }
    }  // ts
    if (use_mbox) ptx::cluster_sync_all();  // no CTA leaves while a neighbour may still store into its mailbox
}

// ---------------------------------------------------------------------------------------------------------------
// Several right-hand sides.  The single-vector kernels above read all of A (residual) or all of the factors (solve)
// for ONE column; these read them once for a block of columns.  A column's arithmetic is the same whatever its
// position in the block, the block's width or the other columns: the same products summed in the same order.

constexpr int RB_THREADS = 128;  // each thread owns 2 consecutive rows, as in residual_partial_kernel
constexpr int RB_TILE = 128;     // columns of A whose X entries are staged in shared memory at a time

__device__ __forceinline__ double nan_max(double a, double b) { return (a > b || a != a) ? a : b; }

// partial[(chunk * kstride + j) * n + row] = sum_{c in chunk} A(row,c) * X(c,j) for the kc <= K columns of this block:
// every entry of A is loaded once for all of them.  kAbs: abs_partial[chunk * n + row] = sum |A(row,c)| as well.
template <bool kAbs, int K>
__global__ void __launch_bounds__(RB_THREADS)
residual_block_partial_kernel(const double* __restrict__ A, long long lda, int n, const double* __restrict__ X,
                              long long ldx, int kc, double* __restrict__ partial, int kstride, int cols_per,
                              double* __restrict__ abs_partial) {
    __shared__ __align__(16) double xs[RB_TILE][K];
    const int c0 = blockIdx.y * cols_per;
    const int c1 = min(n, c0 + cols_per);
    const int r0 = 2 * (blockIdx.x * RB_THREADS + threadIdx.x);
    const bool vec = (r0 + 1 < n) && ((lda & 1) == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
    double a0[K], a1[K];
#pragma unroll
    for (int j = 0; j < K; ++j) a0[j] = a1[j] = 0.0;
    double s0 = 0.0, s1 = 0.0;
    for (int cb = c0; cb < c1; cb += RB_TILE) {
        const int nc = min(RB_TILE, c1 - cb);
        __syncthreads();  // the previous tile's X entries are consumed
        for (int e = threadIdx.x; e < RB_TILE * K; e += RB_THREADS) {
            const int c = e % RB_TILE, j = e / RB_TILE;
            xs[c][j] = (c < nc && j < kc) ? X[cb + c + (long long)j * ldx] : 0.0;
        }
        __syncthreads();
        if (r0 >= n) continue;
        const double* Ap = A + r0 + (long long)cb * lda;
        if (vec) {
            int c = 0;
            for (; c + 8 <= nc; c += 8) {
                double2 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldg(reinterpret_cast<const double2*>(Ap + (long long)(c + u) * lda));
#pragma unroll
                for (int u = 0; u < 8; ++u) {
#pragma unroll
                    for (int j = 0; j < K; ++j) {
                        const double xv = xs[c + u][j];
                        a0[j] = fma(v[u].x, xv, a0[j]);
                        a1[j] = fma(v[u].y, xv, a1[j]);
                    }
                    if (kAbs) { s0 += fabs(v[u].x); s1 += fabs(v[u].y); }
                }
            }
            for (; c < nc; ++c) {
                const double2 v = __ldg(reinterpret_cast<const double2*>(Ap + (long long)c * lda));
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    a0[j] = fma(v.x, xs[c][j], a0[j]);
                    a1[j] = fma(v.y, xs[c][j], a1[j]);
                }
                if (kAbs) { s0 += fabs(v.x); s1 += fabs(v.y); }
            }
        } else {
            for (int c = 0; c < nc; ++c) {
                const double v0 = __ldg(Ap + (long long)c * lda);
                const double v1 = (r0 + 1 < n) ? __ldg(Ap + 1 + (long long)c * lda) : 0.0;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    a0[j] = fma(v0, xs[c][j], a0[j]);
                    a1[j] = fma(v1, xs[c][j], a1[j]);
                }
                if (kAbs) { s0 += fabs(v0); s1 += fabs(v1); }
            }
        }
    }
    if (r0 >= n) return;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        if (j >= kc) break;
        double* p = partial + ((long long)blockIdx.y * kstride + j) * n + r0;
        p[0] = a0[j];
        if (r0 + 1 < n) p[1] = a1[j];
    }
    if (kAbs) {
        abs_partial[(long long)blockIdx.y * n + r0] = s0;
        if (r0 + 1 < n) abs_partial[(long long)blockIdx.y * n + r0 + 1] = s1;
    }
}

// column j = blockIdx.y: R(:,j) = B(:,j) - sum_chunks partial; norms[2j] = max|R(:,j)|, norms[2j+1] = max|X(:,j)|
// (zeroed by the launcher); abs_partial non-null: *anorm = max_row sum_chunks abs_partial (column 0's blocks do it)
__global__ void residual_block_finish_kernel(const double* __restrict__ partial, int n, int nchunk, int kstride,
                                             const double* __restrict__ B, long long ldb, const double* __restrict__ X,
                                             long long ldx, double* __restrict__ R, long long ldr, double* norms,
                                             const double* __restrict__ abs_partial, double* anorm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    const bool with_abs = abs_partial != nullptr && j == 0;
    double rv = 0.0, xv = 0.0, av = 0.0;
    if (i < n) {
        double s = 0.0;
        for (int c = 0; c < nchunk; ++c) s += partial[((long long)c * kstride + j) * n + i];
        if (with_abs)
            for (int c = 0; c < nchunk; ++c) av += abs_partial[(long long)c * n + i];
        rv = B[i + (long long)j * ldb] - s;
        R[i + (long long)j * ldr] = rv;
        rv = fabs(rv);
        xv = fabs(X[i + (long long)j * ldx]);
    }
    for (int o = 16; o > 0; o >>= 1) {  // a NaN must survive the reduction: it ends the refinement
        rv = nan_max(rv, __shfl_xor_sync(0xffffffffu, rv, o));
        xv = nan_max(xv, __shfl_xor_sync(0xffffffffu, xv, o));
        av = fmax(av, __shfl_xor_sync(0xffffffffu, av, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomic_max_double_nonneg(&norms[2 * j], rv);
        atomic_max_double_nonneg(&norms[2 * j + 1], xv);
        if (with_abs) atomic_max_double_nonneg(anorm, av);
    }
}

// out[j] = max_i |B(i,j)|   (zeroed by the launcher), grid (chunks, columns)
__global__ void column_absmax_kernel(const double* __restrict__ B, long long ldb, int n, double* out) {
    const int j = blockIdx.y;
    double m = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) m = nan_max(m, fabs(B[i + (long long)j * ldb]));
    for (int o = 16; o > 0; o >>= 1) m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomic_max_double_nonneg(&out[j], m);
}

__device__ __forceinline__ void st_relaxed_f4(float4* p, float4 v) {
    asm volatile("st.relaxed.gpu.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ bool has_nan(float4 v) { return (v.x != v.x) | (v.y != v.y) | (v.z != v.z) | (v.w != v.w); }

// Both triangular sweeps of L U D = R for kc <= TSB_K columns in one cooperative launch: lu_solve_kernel's steps (one
// 128-row block of one sweep, left-looking, steps complete in order, `ready` counts them, consumers poll the NaN-
// prefilled data and consult the counter every 64 polls), widened to a block of columns.  Every 128 x 128 factor tile
// of a block row is loaded once (4 rows x 16 columns per thread, double-buffered in registers, the diagonal block's
// inverse last) and multiplied into all columns.  The 128 x TSB_K solution blocks are too large for registers: the
// operand block of each tile is polled from L2 by all 256 threads (one float4 each) into shared memory and read from
// there as a warp-wide broadcast.  No DSMEM mailboxes: per step there is TSB_K times the arithmetic of the
// single-vector kernel, so the L2 hand-off latency weighs less on the chain.
// ysol / xsol: npad x TSB_K fp32, row-interleaved (entry (row, j) at row * TSB_K + j): a solved block is 4 KiB contiguous.
constexpr int TSB_K = kSolveBlock;
static_assert(DBS * TSB_K == 4 * TSV_THREADS, "one float4 of a solution block per thread");

__global__ void __launch_bounds__(TSV_THREADS)
lu_solve_block_kernel(const float* __restrict__ W, long long ldw, int n, int nblk, const float* __restrict__ Linv,
                      const float* __restrict__ Uinv, const double* __restrict__ rhs, long long ldr, int kc, float* ysol,
                      float* xsol, double* __restrict__ d_out, long long ldd, double* __restrict__ x_accum, long long ldxa,
                      unsigned* ready) {
    __shared__ __align__(16) float s_part[8][DBS][TSB_K];  // per-warp partial products of the block row
    __shared__ __align__(16) float s_op[2][DBS][TSB_K];    // operand block of the current tile (two buffers)
    __shared__ __align__(16) float s_acc[DBS][TSB_K];      // right-hand side minus the tile products
    const int tid = threadIdx.x;
    const int rg = tid & 31, cg = tid >> 5;          // tile layout: rows 4rg.., columns 16cg..
    const int orow = tid >> 1, oj = 4 * (tid & 1);   // owner layout: row orow, columns oj .. oj+3 of a block
    unsigned seen = 0;
    for (int s = blockIdx.x; s < 2 * nblk; s += gridDim.x) {
        const bool back = s >= nblk;
        const int t = back ? s - nblk : s;
        const int i = back ? nblk - 1 - t : t;
        const float* solv = back ? xsol : ysol;
        const float* inv = (back ? Uinv : Linv) + (long long)i * DBS * DBS;
        const int row = i * DBS + orow;
        float4 a_pre = make_float4(0.f, 0.f, 0.f, 0.f);
        if (back) {
            a_pre = ld_relaxed_f4(reinterpret_cast<const float4*>(ysol) + (long long)i * (DBS * TSB_K / 4) + tid);
        } else if (row < n) {
            float a[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) a[u] = (oj + u < kc) ? static_cast<float>(rhs[row + (long long)(oj + u) * ldr]) : 0.f;
            a_pre = make_float4(a[0], a[1], a[2], a[3]);
        }
        float acc[4][TSB_K];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int j = 0; j < TSB_K; ++j) acc[r][j] = 0.f;
        const float* wrow = W + (long long)i * DBS + 4 * rg;
        auto load_tile = [&](float4 (&v)[16], int tt) {
            if (tt < t) {
                const int j = back ? nblk - 1 - tt : tt;
                const float* wp = wrow + ((long long)j * DBS + 16 * cg) * ldw;
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = __ldcs(reinterpret_cast<const float4*>(wp + (long long)q * ldw));
            } else {
                const float* ip = inv + 4 * rg + 16 * cg * DBS;
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = __ldcs(reinterpret_cast<const float4*>(ip + q * DBS));
            }
        };
        // o[r][j] += sum_q v[q].r * blk[16 cg + q][j]
        auto multiply = [&](const float4 (&v)[16], const float (*blk)[TSB_K], float (&o)[4][TSB_K]) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const float4 lo = *reinterpret_cast<const float4*>(&blk[16 * cg + q][0]);
                const float4 hi = *reinterpret_cast<const float4*>(&blk[16 * cg + q][4]);
                const float sv[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
                const float w[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int j = 0; j < TSB_K; ++j) o[r][j] = fmaf(w[r], sv[j], o[r][j]);
            }
        };
        // wait for the solution block tile tt multiplies, stage it, accumulate
        auto consume = [&](const float4 (&v)[16], int tt) {
            const int j = back ? nblk - 1 - tt : tt;
            const unsigned need = (back ? nblk : 0) + tt + 1;
            const float4* sp = reinterpret_cast<const float4*>(solv) + (long long)j * (DBS * TSB_K / 4) + tid;
            float4 x4;
            for (int spin = 0;; ++spin) {
                x4 = ld_relaxed_f4(sp);
                if (!has_nan(x4) || seen >= need) break;
                if ((spin & 63) == 63) seen = ld_acquire_u32(ready);  // a NaN that is data, not "not yet written"
            }
            reinterpret_cast<float4*>(&s_op[tt & 1][0][0])[tid] = x4;
            __syncthreads();  // (the buffer written here was last read two tiles ago, before the previous barrier)
            multiply(v, s_op[tt & 1], acc);
        };
        // partial products of the 8 warps -> s_part; the owner of (row, oj..oj+3) adds (sign 1) or subtracts (sign -1)
        // them in warp order, the order of lu_solve_kernel
        auto reduce = [&](const float (&o)[4][TSB_K], float4 sum, float sign) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                float4* p = reinterpret_cast<float4*>(&s_part[cg][4 * rg + r][0]);
                p[0] = make_float4(o[r][0], o[r][1], o[r][2], o[r][3]);
                p[1] = make_float4(o[r][4], o[r][5], o[r][6], o[r][7]);
            }
            __syncthreads();
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                const float4 pg = reinterpret_cast<const float4*>(&s_part[g][0][0])[tid];
                sum.x += sign * pg.x; sum.y += sign * pg.y; sum.z += sign * pg.z; sum.w += sign * pg.w;
            }
            return sum;
        };
        auto finish = [&](const float4 (&vi)[16]) {
            float4 a = a_pre;
            if (back) {  // y of this block row, solved at forward step i of this launch (the prefetch may predate it)
                for (int spin = 0; has_nan(a); ++spin) {
                    a = ld_relaxed_f4(reinterpret_cast<const float4*>(ysol) + (long long)i * (DBS * TSB_K / 4) + tid);
                    if (!has_nan(a) || seen >= (unsigned)(i + 1)) break;  // read after the counter said so: final
                    if ((spin & 63) == 63) seen = ld_acquire_u32(ready);
                }
            }
            a = reduce(acc, a, -1.f);
            reinterpret_cast<float4*>(&s_acc[0][0])[tid] = a;
            __syncthreads();  // s_acc complete; every owner has read s_part
            float o[4][TSB_K];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int j = 0; j < TSB_K; ++j) o[r][j] = 0.f;
            multiply(vi, s_acc, o);
            const float4 v = reduce(o, make_float4(0.f, 0.f, 0.f, 0.f), 1.f);
            float* sol = back ? xsol : ysol;
            st_relaxed_f4(reinterpret_cast<float4*>(sol) + (long long)i * (DBS * TSB_K / 4) + tid, v);
            if (back && row < n) {
                const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (oj + u < kc) {
                        if (d_out) d_out[row + (long long)(oj + u) * ldd] = static_cast<double>(vv[u]);
                        if (x_accum) x_accum[row + (long long)(oj + u) * ldxa] += static_cast<double>(vv[u]);
                    }
            }
        };
        {
            float4 va[16], vb[16];
            load_tile(va, 0);
            for (int tt = 0; tt < t; tt += 2) {
                load_tile(vb, tt + 1);
                consume(va, tt);
                if (tt + 1 < t) {
                    load_tile(va, tt + 2);
                    consume(vb, tt + 1);
                }
            }
            if (t & 1) finish(vb); else finish(va);
        }
        __syncthreads();  // s_part / s_acc / s_op are free for the next step
        if (tid == 0) {
            __threadfence();
            st_release_u32(ready, (unsigned)(s + 1));
        }
    }
}

}  // namespace

int launch_residual(const double* A, long long lda, int n, const double* x, const double* b, double* r,
                    double* partial, int nchunk, double* norms, cudaStream_t st, double* abs_partial, double* anorm) {
    const int cols_per = (n + nchunk - 1) / nchunk;
    dim3 grid((n + 2 * RES_THREADS - 1) / (2 * RES_THREADS), nchunk);
    const bool with_abs = abs_partial != nullptr && anorm != nullptr;
    if (with_abs) {
        residual_partial_kernel<true><<<grid, RES_THREADS, cols_per * sizeof(double), st>>>(A, lda, n, x, partial, cols_per, abs_partial);
        cudaMemsetAsync(anorm, 0, sizeof(double), st);
    } else {
        residual_partial_kernel<false><<<grid, RES_THREADS, cols_per * sizeof(double), st>>>(A, lda, n, x, partial, cols_per, nullptr);
    }
    cudaMemsetAsync(norms, 0, 2 * sizeof(double), st);
    residual_finish_kernel<<<(n + 255) / 256, 256, 0, st>>>(partial, n, nchunk, b, x, r, norms, with_abs ? abs_partial : nullptr,
                                                            with_abs ? anorm : nullptr);
    return (int)cudaGetLastError();
}

namespace {
// step counter + NaN fill of what the sweep produces (consumers poll the data), one launch
__global__ void sweep_prep_kernel(unsigned* ready, unsigned v, float* y_fill, float* x_fill, int npad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *ready = v;
    if (i < npad) {
        if (y_fill) y_fill[i] = __int_as_float(0x7fffffff);
        if (x_fill) x_fill[i] = __int_as_float(0x7fffffff);
    }
}
}  // namespace

int launch_lu_solve(const float* W, long long ldw, int n, int npad, const float* Linv32, const float* Uinv32,
                    const double* rhs, float* y, double* d_out, double* x_accum, unsigned* ready, cudaStream_t st) {
    return launch_lu_sweep(W, ldw, n, npad, Linv32, Uinv32, rhs, y, y + npad, d_out, x_accum, ready, 0, st, nullptr, 0, nullptr);
}

int launch_lu_sweep(const float* W, long long ldw, int n, int npad, const float* Linv32, const float* Uinv32,
                    const double* rhs, float* ysol, float* xsol, double* d_out, double* x_accum, unsigned* ready,
                    int mode, cudaStream_t st, const float* sub, int flags, const SweepPx* px) {
    // the dynamic shared-memory opt-in and the co-residency limits are PER DEVICE: cached per device ordinal
    constexpr int kMaxDev = 64;
    static int s_max_grid[kMaxDev] = {}, s_max_grid_cl[kMaxDev] = {};
    static std::mutex s_mu;
    // CTAs per cluster (mailbox hand-offs stay inside a cluster): 8; MPLU_TSV_CLUSTER = 2 / 4 for experiments (more co-resident
    // CTAs -- 8-CTA clusters fill 120 of the 148 SMs -- against more hand-offs that cross a cluster boundary through L2)
    static const int CL = [] { const char* e = getenv("MPLU_TSV_CLUSTER"); const int v = e ? atoi(e) : 8; return (v == 2 || v == 4) ? v : 8; }();
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= kMaxDev) return (int)cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lock(s_mu);
    int& max_grid = s_max_grid[dev];
    int& max_grid_cl = s_max_grid_cl[dev];
    if (!max_grid) {
        cudaError_t e = cudaFuncSetAttribute(lu_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TSV_SMEM_BYTES);
        if (e != cudaSuccess) return (int)e;
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lu_solve_kernel, TSV_THREADS, TSV_SMEM_BYTES);
        if (e != cudaSuccess) return (int)e;
        if (per_sm < 1) return (int)cudaErrorLaunchOutOfResources;
        max_grid = sms * per_sm;
        // co-resident clusters of CL CTAs (the mailbox hand-off); 0 = not available, use the plain launch
        const char* env = getenv("MPLU_TSV_CLUSTER");
        if (!(env && env[0] == '0')) {
            cudaLaunchConfig_t q{};
            q.gridDim = dim3(CL); q.blockDim = dim3(TSV_THREADS); q.dynamicSmemBytes = TSV_SMEM_BYTES;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            q.attrs = at; q.numAttrs = 1;
            int ncl = 0;
            if (cudaOccupancyMaxActiveClusters(&ncl, lu_solve_kernel, &q) == cudaSuccess && ncl > 0) max_grid_cl = ncl * CL;
            else cudaGetLastError();
        }
    }
    int nblk = npad / DBS;
    int s_begin = mode == 2 ? nblk : 0, s_end = mode == 1 ? nblk : 2 * nblk;
    // NaN-fill what this launch produces: consumers poll the data (mode 2 takes its right-hand side in ysol)
    if (!(flags & SWEEP_PREPARED))
        sweep_prep_kernel<<<(npad + 255) / 256, 256, 0, st>>>(ready, (unsigned)s_begin, mode != 2 ? ysol : nullptr,
                                                             (mode != 1 && xsol) ? xsol : nullptr, npad);
    int use_mbox = 0;
    int grid = nblk < max_grid ? nblk : max_grid;
    if (max_grid_cl >= CL && nblk >= CL) {
        int g = nblk < max_grid_cl ? nblk : max_grid_cl;
        g -= g % CL;
        if (g >= CL) { grid = g; use_mbox = 1; }
    }
    const SweepPx pxv = px ? *px : SweepPx{nullptr, 0, 0, 0, 0};
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(TSV_THREADS);
    cfg.dynamicSmemBytes = TSV_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attrs[2];
    attrs[0].id = cudaLaunchAttributeCooperative;
    attrs[0].val.cooperative = 1;
    attrs[1].id = cudaLaunchAttributeClusterDimension;
    attrs[1].val.clusterDim.x = CL; attrs[1].val.clusterDim.y = 1; attrs[1].val.clusterDim.z = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = use_mbox ? 2 : 1;
    // SWEEP_PLAIN_LAUNCH (one sweep of a small tile, every step its own CTA, far fewer CTAs than SMs): no cooperative
    // attribute.  A CTA only ever waits for steps owned by CTAs of lower index, and the hardware dispatches CTAs (clusters) in
    // index order, so a waiting CTA never keeps the one it waits for off the machine.
    if ((flags & SWEEP_PLAIN_LAUNCH) && mode != 0 && grid == nblk && grid <= 32) {
        attrs[0] = attrs[1];
        cfg.numAttrs = use_mbox ? 1 : 0;
    }
    cudaError_t le = cudaLaunchKernelEx(&cfg, lu_solve_kernel, W, ldw, n, nblk, Linv32, Uinv32, rhs, ysol, xsol, d_out,
                                        x_accum, ready, s_begin, s_end, use_mbox, sub, pxv, TileChain{});
    if (le != cudaSuccess && use_mbox) {  // cooperative cluster launch not available: plain cooperative launch from now on
        cudaGetLastError();
        max_grid_cl = 0;
        use_mbox = 0;
        cfg.gridDim = dim3(nblk < max_grid ? nblk : max_grid);
        attrs[0].id = cudaLaunchAttributeCooperative;
        attrs[0].val.cooperative = 1;
        cfg.numAttrs = 1;
        le = cudaLaunchKernelEx(&cfg, lu_solve_kernel, W, ldw, n, nblk, Linv32, Uinv32, rhs, ysol, xsol, d_out, x_accum, ready,
                                s_begin, s_end, use_mbox, sub, pxv, TileChain{});
    }
    return (int)le;
}

namespace {
template <bool kAbs, int K>
void residual_block_partial(dim3 grid, cudaStream_t st, const double* A, long long lda, int n, const double* X, long long ldx,
                            int kc, double* partial, int cols_per, double* abs_partial) {
    residual_block_partial_kernel<kAbs, K><<<grid, RB_THREADS, 0, st>>>(A, lda, n, X, ldx, kc, partial, kc, cols_per,
                                                                        abs_partial);
}
template <bool kAbs>
void residual_block_partial_k(dim3 grid, cudaStream_t st, const double* A, long long lda, int n, const double* X,
                              long long ldx, int kc, double* partial, int cols_per, double* abs_partial) {
    // the narrowest instantiation that holds kc columns (a column's sums do not depend on it)
    if (kc <= 2) residual_block_partial<kAbs, 2>(grid, st, A, lda, n, X, ldx, kc, partial, cols_per, abs_partial);
    else if (kc <= 4) residual_block_partial<kAbs, 4>(grid, st, A, lda, n, X, ldx, kc, partial, cols_per, abs_partial);
    else if (kc <= 8) residual_block_partial<kAbs, 8>(grid, st, A, lda, n, X, ldx, kc, partial, cols_per, abs_partial);
    else residual_block_partial<kAbs, 16>(grid, st, A, lda, n, X, ldx, kc, partial, cols_per, abs_partial);
}
}  // namespace

int launch_residual_block(const double* A, long long lda, int n, const double* X, long long ldx, const double* B,
                          long long ldb, double* R, long long ldr, int kc, double* partial, double* norms, cudaStream_t st,
                          double* abs_partial, double* anorm) {
    if (kc < 1 || kc > kResidualBlock) return (int)cudaErrorInvalidValue;
    const int nchunk = kResidualChunks;
    const int cols_per = (n + nchunk - 1) / nchunk;
    const dim3 grid((n + 2 * RB_THREADS - 1) / (2 * RB_THREADS), nchunk);
    const bool with_abs = abs_partial != nullptr && anorm != nullptr;
    if (with_abs) {
        residual_block_partial_k<true>(grid, st, A, lda, n, X, ldx, kc, partial, cols_per, abs_partial);
        cudaMemsetAsync(anorm, 0, sizeof(double), st);
    } else {
        residual_block_partial_k<false>(grid, st, A, lda, n, X, ldx, kc, partial, cols_per, nullptr);
    }
    cudaMemsetAsync(norms, 0, 2 * kc * sizeof(double), st);
    residual_block_finish_kernel<<<dim3((n + 255) / 256, kc), 256, 0, st>>>(partial, n, nchunk, kc, B, ldb, X, ldx,
                                                                           R, ldr, norms, with_abs ? abs_partial : nullptr,
                                                                           with_abs ? anorm : nullptr);
    return (int)cudaGetLastError();
}

int launch_column_absmax(const double* B, long long ldb, int n, int ncols, double* out, cudaStream_t st) {
    cudaMemsetAsync(out, 0, ncols * sizeof(double), st);
    const int chunks = (n + 255) / 256 < 32 ? (n + 255) / 256 : 32;
    column_absmax_kernel<<<dim3(chunks, ncols), 256, 0, st>>>(B, ldb, n, out);
    return (int)cudaGetLastError();
}

int launch_lu_solve_block(const float* W, long long ldw, int n, int npad, const float* Linv32, const float* Uinv32,
                          const double* rhs, long long ldr, int kc, float* work, double* d_out, long long ldd,
                          double* x_accum, long long ldxa, unsigned* ready, cudaStream_t st) {
    if (kc < 1 || kc > TSB_K) return (int)cudaErrorInvalidValue;
    constexpr int kMaxDev = 64;
    static int s_max_grid[kMaxDev] = {};
    static std::mutex s_mu;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= kMaxDev) return (int)cudaErrorInvalidDevice;
    int max_grid;
    {
        std::lock_guard<std::mutex> lock(s_mu);
        if (!s_max_grid[dev]) {  // every CTA must be resident: consumers spin on steps owned by other CTAs
            int sms = 0, per_sm = 0;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lu_solve_block_kernel, TSV_THREADS, 0);
            if (e != cudaSuccess) return (int)e;
            if (per_sm < 1) return (int)cudaErrorLaunchOutOfResources;
            s_max_grid[dev] = sms * per_sm;
        }
        max_grid = s_max_grid[dev];
    }
    const int nblk = npad / DBS;
    const long long nw = (long long)npad * TSB_K;
    float* ysol = work;
    float* xsol = work + nw;
    sweep_prep_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>(ready, 0u, ysol, xsol, (int)nw);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(nblk < max_grid ? nblk : max_grid);
    cfg.blockDim = dim3(TSV_THREADS);
    cfg.stream = st;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeCooperative;
    attrs[0].val.cooperative = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = 1;
    return (int)cudaLaunchKernelEx(&cfg, lu_solve_block_kernel, W, ldw, n, nblk, Linv32, Uinv32, rhs, ldr, kc, ysol, xsol,
                                   d_out, ldd, x_accum, ldxa, ready);
}

// every tile sweep of a block-cyclic solve in one launch: nb/128 CTAs (one step of each tile sweep per CTA) in clusters of 8,
// resident for the whole solve; see TileChain
int launch_tile_chain(const TileChain& tc, cudaStream_t st) {
    constexpr int CL = 8;
    const int nblk = tc.nb / DBS;
    if (tc.count <= 0 || nblk <= 0 || nblk > 64 || tc.nb % DBS) return (int)cudaErrorInvalidValue;
    const int use_mbox = (nblk % CL == 0) ? 1 : 0;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(nblk);
    cfg.blockDim = dim3(TSV_THREADS);
    cfg.dynamicSmemBytes = TSV_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeClusterDimension;
    attrs[0].val.clusterDim.x = CL; attrs[0].val.clusterDim.y = 1; attrs[0].val.clusterDim.z = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = use_mbox ? 1 : 0;
    return (int)cudaLaunchKernelEx(&cfg, lu_solve_kernel, (const float*)nullptr, (long long)tc.nb, tc.nb, nblk, (const float*)nullptr,
                                   (const float*)nullptr, (const double*)nullptr, (float*)nullptr, (float*)nullptr, (double*)nullptr,
                                   (double*)nullptr, (unsigned*)nullptr, 0, 0, use_mbox, (const float*)nullptr,
                                   SweepPx{nullptr, 0, 0, 0, 0}, tc);
}

}  // namespace mplu
