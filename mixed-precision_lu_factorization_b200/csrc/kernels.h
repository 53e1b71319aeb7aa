// Internal launch interface shared by the CUDA translation units of libmplu (not part of the public C ABI).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace mplu {

// indices into the device-resident scale table (all powers of two; 1 for bf16)
enum ScaleIdx : int {
    SC_A = 0,           // scale of matrix-magnitude (A / U type) 16-bit shadows
    SC_A_INV = 1,       // 1 / SC_A
    SC_L = 2,           // scale of multiplier (L type) shadows
    SC_L_INV = 3,       // 1 / SC_L
    SC_NEG_LA_INV = 4,  // -1 / (SC_L * SC_A): alpha of the Schur update
    SC_ONE = 5,
    SC_COUNT = 8
};

constexpr int kDiagBlock = 128;  // diagonal block / base panel width

// panel.cu
int panel_init();  // per-device kernel attributes; call before the first launch / graph capture
// rscale / cscale non-null (equilibration): W = fp32(diag(rscale) A diag(cscale)), amax of that; ||A||_inf of A itself
int launch_first_touch(const double* A, long long lda, int n, float* W, long long ldw, int npad, float* amax,
                       double* rowsum_part, int nchunk, double* anorm, cudaStream_t st, const double* rscale = nullptr,
                       const double* cscale = nullptr);
// the same first touch for the columns [cb, ce) only (amax accumulates, not reset; row sums into slots
// [slot0, slot0 + nslots) of rowsum_part), and the final ||A||_inf over the first nslots slots
int launch_first_touch_cols(const double* A, long long lda, int n, float* W, long long ldw, int npad, int cb, int ce,
                            float* amax, double* rowsum_part, int slot0, int nslots, cudaStream_t st);
// the same for rows [0, rows) of the columns [cb, ce) only, without row sums (lazy first touch: first block row)
int launch_first_touch_block(const double* A, long long lda, int n, float* W, long long ldw, int npad, int rows, int cb, int ce,
                             float* amax, cudaStream_t st);
int launch_anorm(const double* rowsum_part, int n, int nslots, double* anorm, cudaStream_t st);
int launch_scales(const float* amax, float* scales, int target_exp_a, int exp_l, int bf16, cudaStream_t st);
int launch_shadow_cast(const float* W, long long ldw, void* H, long long ldh, int rows, int cols, const float* scale,
                       int bf16, int* status, cudaStream_t st);
// No-pivot LU of the 128x128 block at W(k0,k0) + its explicit inverses.  Linv16/Uinv16 point at the block's origin
// inside the 16-bit inverse bands (leading dimension ld16); Linv32/Uinv32 are the fp32 copies for the triangular
// solves, indexed by blk.  tile_scales[0..3] = {s_Linv, 1/s_Linv, s_Uinv, 1/s_Uinv} of the enclosing diagonal tile:
// written when first_in_tile, read otherwise.
int launch_diag_lu(float* W, long long ldw, int k0, void* Linv16, void* Uinv16, long long ld16, float* Linv32,
                   float* Uinv32, float* tile_scales, int first_in_tile, int blk, int bf16, int* status, cudaStream_t st,
                   long long* dbg_clk = nullptr,  // optional device array of phase time stamps (clock64)
                   int pdl = 0,                   // 1 = programmatic dependent launch
                   int valid = kDiagBlock);       // rows/columns of the block that belong to the matrix (the rest is identity padding)

// equil.cu: dgeequb scales + dlaqge decision.  eq: EQ_WORDS device words; the non-negative doubles are kept as bit patterns.
enum EquilWord : int { EQ_RMIN = 0, EQ_CMIN = 1, EQ_RMAX = 2, EQ_CMAX = 3, EQ_BAD = 4, EQ_EQUED = 5, EQ_WORDS = 8 };
// r (n), c (n) = the scales of the applied sides, 1 elsewhere; eq[EQ_EQUED] = EQUED (bit 0 rows, bit 1 columns; 0 after a
// zero row / column or a non-finite entry).  part: nchunk * n doubles of workspace.  Four launches.
int launch_equilibrate(const double* A, long long lda, int n, double* part, int nchunk, double* r, double* c,
                       unsigned long long* eq, cudaStream_t st);
// out(:, j) = s o in(:, j) (accumulate: out(:, j) += s o in(:, j)) for k columns; in may be out
int launch_diag_scale(const double* s, int n, int k, const double* in, long long ldi, double* out, long long ldo,
                      int accumulate, cudaStream_t st);

// ir.cu
// r = b - A*x (fp64), ||r||_inf and ||x||_inf into norms[0], norms[1]
// abs_partial (nchunk * n doubles) / anorm non-null: the same pass also forms the row sums of |A| and ||A||_inf
int launch_residual(const double* A, long long lda, int n, const double* x, const double* b, double* r,
                    double* partial, int nchunk, double* norms, cudaStream_t st, double* abs_partial = nullptr,
                    double* anorm = nullptr);
// solve L U d = r with the fp32 factors in W (unit-lower L, U), blocked by kDiagBlock with the fp32 inverses of the
// diagonal blocks; y (fp32 work vectors, 2*npad floats); ready = one device word (step counter of the sweep).  d_out (fp64) = solution; if x_accum != null, x_accum += d.
int launch_lu_solve(const float* W, long long ldw, int n, int npad, const float* Linv32, const float* Uinv32,
                    const double* rhs, float* y, double* d_out, double* x_accum, unsigned* ready, cudaStream_t st);

// Several right-hand sides (column-major blocks).  A column's arithmetic does not depend on its position in the block,
// on the block's width or on the other columns.
constexpr int kResidualBlock = 16;  // columns per residual launch (A is streamed once for all of them)
constexpr int kResidualChunks = 16; // column chunks of A summed separately: workspace kResidualChunks * kc * n
constexpr int kSolveBlock = 8;      // columns per triangular-solve launch (the factors are streamed once for all of them)
// R(:, 0..kc) = B - A X in fp64 for kc <= kResidualBlock columns; norms[2j] = ||R(:,j)||_inf, norms[2j+1] = ||X(:,j)||_inf.
// partial: kResidualChunks * kc * n doubles.  abs_partial (kResidualChunks * n) / anorm non-null: the same pass
// also forms the row sums of |A| and ||A||_inf
int launch_residual_block(const double* A, long long lda, int n, const double* X, long long ldx, const double* B,
                          long long ldb, double* R, long long ldr, int kc, double* partial, double* norms, cudaStream_t st,
                          double* abs_partial = nullptr, double* anorm = nullptr);
// out[j] = ||B(:,j)||_inf for ncols columns
int launch_column_absmax(const double* B, long long ldb, int n, int ncols, double* out, cudaStream_t st);
// L U D = rhs for kc <= kSolveBlock columns (the arithmetic of launch_lu_solve, column by column); work: 2 * npad *
// kSolveBlock floats; D (fp64) -> d_out and / or x_accum += D, each column-major with its leading dimension
int launch_lu_solve_block(const float* W, long long ldw, int n, int npad, const float* Linv32, const float* Uinv32,
                          const double* rhs, long long ldr, int kc, float* work, double* d_out, long long ldd,
                          double* x_accum, long long ldxa, unsigned* ready, cudaStream_t st);

// Partial sums that arrive from peer GPUs (block-cyclic solver, csrc/dist.cu): `base` = this rank's exchange buffer (kPxFlagWords
// flag words, then slots of nb floats); the sweep waits until the Q flags slot0 .. slot0+Q-1 hold `epoch` and subtracts the sum
// of those slots from its right-hand side.  The launch is already resident (its tile loads under way) when the data lands.
constexpr unsigned long long kPxFlagWords = 16384;
struct SweepPx {
    const float* base;
    unsigned long long slot0;
    int Q, nb;
    unsigned epoch;
};

// All tile sweeps of one block-cyclic solve in ONE persistent launch (csrc/dist.cu, MPLU_DIST_TILE_CHAIN=1 with the peer
// exchange): count = 2 T tile sweeps, forward over the replicated diagonal tiles k = 0 .. T-1, then backward k = T-1 .. 0; tile
// sweep (sweep, k) takes its right-hand side from rhs + k nb (forward) / yv + k nb (backward) minus the partial sums that arrive
// in the exchange slots ((sweep T + k) Q ..) -- except the first tile of each sweep, which has none --, writes yv / xv + k nb
// and counts its steps in ready[sweep T + k] (final value nb/128 forward, 2 nb/128 backward: what the GEMV kernels of the step
// wait for on the device).  dbg: bit 0 is set when a wait for the exchange slots timed out.
struct TileChain {
    int count, T, nb;
    const float *Dw, *Dl32, *Du32;
    const double* rhs;
    float *yv, *xv;
    unsigned* ready;
    const float* px_base;
    int Q;
    unsigned epoch;
    unsigned* dbg;
    unsigned* started;  // host-visible counter (may be null): every CTA adds 1 once it is resident -- the host enqueues the
                        // kernels that wait for this launch on the device only after all of them are, so that their
                        // blocks cannot take its SMs first
};
int launch_tile_chain(const TileChain& tc, cudaStream_t st);

// One sweep only: mode 0 = both (as launch_lu_solve), 1 = forward (L y = rhs, y -> ysol), 2 = backward (U x = ysol,
// x -> xsol); used tile by tile by the block-cyclic solver.  sub (fp32, npad entries, may be null) is subtracted from the
// right-hand side: what the other tile columns already contributed.
int launch_lu_sweep(const float* W, long long ldw, int n, int npad, const float* Linv32, const float* Uinv32,
                    const double* rhs, float* ysol, float* xsol, double* d_out, double* x_accum, unsigned* ready,
                    int mode, cudaStream_t st, const float* sub = nullptr, int flags = 0, const struct SweepPx* px = nullptr);
// flags: SWEEP_PREPARED = the caller has set *ready to the first step (0 forward / npad/128 backward) and filled what the sweep
// produces with NaN (consumers poll the data); SWEEP_PLAIN_LAUNCH = small one-sweep launches without the cooperative attribute
enum { SWEEP_PREPARED = 1, SWEEP_PLAIN_LAUNCH = 2 };

}  // namespace mplu
