/* mplu.h -- thin C ABI of the B200-native mixed-precision LU + iterative-refinement solver.
 *
 * The reference (Keyteer/Mixed-precision_LU_Factorization) exposes exactly one host entry point,
 *     void MPF(double *h_A, int N, int r, int *IPIV);            -- /root/reference/MPF.h:3, MPF.cu:66-256
 * with C++ linkage, no status and no solve path.  That symbol is kept byte-compatible in include/MPF.h.  This header
 * is the C-ABI layer BASELINE.json's north_star asks for on top of it: plain pointers and sizes, explicit status
 * codes, device-resident and host-buffer variants of factor / solve / gesv.  Every function returns 0 on success,
 * a positive cudaError_t value for CUDA failures, or a negative MPLU_E_* code.
 *
 * Layout conventions are the reference's: matrices are column-major (benchmark.cpp:19 prints mat[j*n+i]), leading
 * dimension in elements, fp64 on the interface.
 */
#ifndef MPLU_H
#define MPLU_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mplu_context mplu_context;

enum {
    MPLU_OK = 0,
    MPLU_E_ARG = -1,        /* bad argument */
    MPLU_E_NODEVICE = -2,   /* no CUDA device (the reference prints and returns: MPF.cu:72-75) */
    MPLU_E_NOTFACTORED = -3,
    MPLU_E_TMAP = -4,       /* TMA descriptor encoding failed */
    MPLU_E_OVERFLOW = -5,   /* a 16-bit panel value left the fp16 range (factorization unusable) */
    MPLU_E_ZEROPIVOT = -6,  /* exact zero pivot met without pivoting */
    MPLU_E_NOCONV = -7,     /* refinement did not reach the tolerance in max_iters (x holds the last iterate) */
    MPLU_E_NCCL = -8        /* NCCL missing (dlopen of libnccl.so.2 failed) or an NCCL call failed */
};

enum { MPLU_FP16 = 0, MPLU_BF16 = 1 };
enum { MPLU_GEMM_AUTO = -1, MPLU_GEMM_CG1 = 0, MPLU_GEMM_CG2 = 1 };
enum { MPLU_REFINE_CLASSIC = 0, MPLU_REFINE_GMRES = 1 };
enum { MPLU_SCHED_RIGHT = 0, MPLU_SCHED_LEFT = 1 };

typedef struct mplu_options {
    int precision;    /* MPLU_FP16 (default) or MPLU_BF16: panel/operand storage type; accumulation is fp32 */
    int nb;           /* outer (trailing-update) block size, multiple of 128; 0 (default) = by n: 2048 / 1024 / 512 */
    int max_iters;    /* refinement iteration cap, default 30 (LAPACK dsgesv ITERMAX) */
    double tol;       /* <= 0: dsgesv rule ||r||_inf <= ||x||_inf ||A||_inf eps sqrt(n); else relative to ||A|| ||x|| */
    int gemm_variant; /* MPLU_GEMM_AUTO / CG1 (128x256 tiles) / CG2 (CTA-pair 256x256 tiles) */
    int max_sms;      /* 0 = all SMs */
    int a_exp;        /* fp16 only: A-type shadows are scaled so max|A| maps into (2^(a_exp-1), 2^a_exp]; default 11 */
    int l_exp;        /* fp16 only: multipliers are scaled by 2^l_exp; default 11 */
    int lookahead;    /* 1 (default): factor panel k+1 on a second stream while the rest of update k runs */
    int side_sms;     /* MPLU_SCHED_RIGHT: SMs of the chain lane (diagonal-tile GETRF + next-tile solves), default 40 */
    int use_graph;    /* 1 (default): capture the factorization schedule once per (n, options) into a CUDA graph */
    int pdl;          /* 1: programmatic dependent launches along each stream's kernel chain (default 0: measured slower,
                         pre-launched CTAs take SMs from the other lane); 2: on the chain lane only */
    int group;        /* 1 (default): independent L-side / U-side products of a recursion node share one launch */
    int refinement;   /* MPLU_REFINE_CLASSIC (default): d = (LU)^-1 r;  MPLU_REFINE_GMRES: GMRES on (LU)^-1 A d = (LU)^-1 r */
    int gmres_restart;/* Krylov steps per correction at most (default 50) */
    double gmres_tol; /* relative reduction of the preconditioned residual that ends a correction (default 1e-6) */
    int bf16_fallback;/* 1 (default): an fp16 factorization whose scaled values left the fp16 range is redone in bf16 */
    int tile_ws;      /* 1: diagonal tiles are factored in a compact nb x nb workspace, copied in / out (default 0: measured
                         neutral, 43.3 vs 43.0 ms at n=32768) */
    int cg2_min_elems;/* MPLU_GEMM_AUTO: products with M*N below this use single-CTA tiles even when M > 128 */
    int side_sms_early; /* chain-lane SMs while more than early_pct % of the columns are still trailing (0 = side_sms) */
    int early_pct;
    int tri_skip;     /* 1 (default): products with an explicit triangular inverse skip the zero half of their K range */
    int late_pct;     /* once at most late_pct % of the columns are trailing, both lanes may use every SM */
    int l2_persist;   /* 1: with tile_ws, pin that workspace in L2 through an access-policy window on the chain lane's
                         stream (default 0: measured much slower, 62.6 ms -- the carve-out starves the trailing GEMM) */
    int stream_host;  /* mplu_gesv_host only.  1 (default): A is copied block column by block column and factored
                         left-looking as it arrives, so the factorization hides behind the PCIe transfer (same factors
                         bit for bit); 0: copy everything, then run the device schedule.  Not with equilibrate = 1: the
                         row scales need every column of A before the first cast, so A is copied first */
    int schedule;     /* device-resident input: MPLU_SCHED_LEFT (default) = left-looking block columns with look-ahead and
                         eager updates, MPLU_SCHED_RIGHT = right-looking trailing updates with depth-1 look-ahead
                         (same factors bit for bit; n=32768: 35.8 vs 38.3 ms) */
    int eager;        /* MPLU_SCHED_LEFT: 1 (default) = the bulk lane spends each step's share of the remaining update work
                         ahead of need on the columns further right (balances the lanes); 0 = strictly left-looking */
    int side_sms_left;/* MPLU_SCHED_LEFT: SMs of the chain lane (default 16; side_sms / side_sms_early are the right-looking
                         schedule's) */
    int stream_c;     /* 1 (default): the tall rank-nb updates load / store their fp32 C and 16-bit shadow with the streaming
                         (evict-first) cache policy: that traffic is touched once per launch and far larger than L2 */
    int early_scale;  /* MPLU_SCHED_LEFT, mplu_gesv_device: 1 = the first touch of A overlaps the first diagonal tile's
                         GETRF; the fp16 scale then comes from the first block column and an overflow that spoils the
                         solve is redone with the global scale.  Default 0: measured neutral (35.5 vs 35.9 ms and 37.1
                         vs 37.0 ms on two boxes) -- the bandwidth-bound cast slows the latency-bound tile as much as
                         the overlap saves */
    int fuse_w;       /* GETRF of a diagonal block of at most fuse_w columns (multiple of 128) runs as ONE persistent launch
                         (leaves + every product between them, grid barriers instead of kernel boundaries); same factors
                         bit for bit among fused widths.  Default 512 (measured best at n = 32768: the products above that width run faster as
                         launches of the big GEMM kernel on the chain lane's SMs); 0 = one launch per leaf / product group */
    int fuse_ctas;    /* CTAs (= SMs) of that launch, even, default 8 */
    int lazy_touch;   /* MPLU_SCHED_LEFT, n a multiple of 128: 1 (default) = no separate fp64 -> fp32 cast pass over A.  Only the
                         first block column / block row are cast up front (the fp16 scale comes from them); every other
                         tile's first Schur update takes its addend straight from the caller's fp64 matrix (the cast is fused
                         into the GEMM epilogue's loads) and ||A||_inf is formed by the first residual pass.  An entry that
                         leaves the fp16 range under that scale is detected and the factorization redone the eager way */
    int flow_w;       /* GETRF of a diagonal block of at most flow_w columns (128 * a power of two) runs as ONE dataflow launch
                         (csrc/getrf_flow.cu): right-looking at 128-block granularity, two CTAs run leaf after leaf, the others
                         pull 128x128 tile products from a priority-ordered task list and hand results over through counters
                         in global memory -- no grid barriers, no merged inverse between two leaves.  Takes precedence over
                         fuse_w for the widths it covers; default 2048, 0 = off.  Factors agree with the other paths to rounding level
                         (the Schur updates are summed in rank-128 pieces) */
    int flow_ctas;    /* CTAs (= SMs) of that launch, even, >= 4 (2 leaf CTAs + helpers), default 16 */
    int fp64_fallback;/* 1 (default), mplu_gesv_device / mplu_gesv_host: like LAPACK dsgesv, a solve the low-precision factors cannot
                         deliver (16-bit overflow in fp16 and bf16, exact zero pivot, refinement stalled) is redone with an fp64
                         LU with row pivoting (the reference's MPF algorithm on the device) + fp64 solves; reported through
                         mplu_stats::fp64_fallback / dsgesv_iter.  0: return MPLU_E_OVERFLOW / _ZEROPIVOT / _NOCONV instead */
    int edge_nb;      /* MPLU_SCHED_LEFT, device-resident input: width of the FIRST and LAST block column (multiple of 128, < nb;
                         0 = nb, the default).  Nothing overlaps the first diagonal tile's GETRF and the last one's, so narrower
                         tiles there shorten the two stretches in which most SMs idle -- measured neutral at n = 32768 (33.4 vs
                         33.3 ms): the chain lane is the critical resource in EVERY step, and its 256 leaves do not get fewer */
    int pair_ts;      /* MPLU_SCHED_LEFT, two lanes: 1 = the bulk lane's small panel solves U(k, cols) share a grouped launch with the
                         previous op's tall update when their column ranges are disjoint (fills that launch's tail instead of a
                         one-wave launch of their own); same products, same factors */
    int update_pair;  /* MPLU_SCHED_LEFT, two lanes: 1 = when two consecutive updates k, k+1 of a block-column range are both
                         available the bulk lane applies them in ONE pass (K = both panels' widths: half the fp32 C traffic per
                         flop of an L2-bound kernel).  Same products; the two partial sums are added in TMEM instead of through
                         C, so factors agree with update_pair = 0 to fp32 rounding, not bit for bit.  Measured: 2-3 % faster at
                         n = 32768 (with side_sms_left = flow_ctas = 20), 4 % at n = 65536, same iteration counts up to kappa = 1e6;
                         default 0 because the twice as long fp32 accumulation in the tensor core costs GMRES-IR up to 5x more
                         Krylov steps on the kappa >= 1e7 systems of the condition-number sweep (DESIGN.md section 4) */
    int flow_merge_ctas; /* helpers that take inverse-merge tasks before main-list tasks; -1 (default) = a quarter of them */
    int equilibrate;  /* factor / gesv entry points (not the block-cyclic solver, which returns MPLU_E_ARG for anything but 0).
                         0 (default): off.  1: like LAPACK dgesvx with FACT = 'E': the power-of-two row and column scales r, c
                         of dgeequb are computed on the device and applied by dlaqge's rule (rows if ROWCND < 0.1 or AMAX
                         outside [SMALL, LARGE], columns if COLCND < 0.1; nothing after a zero row / column or a non-finite
                         entry).  With scales applied, diag(r) A diag(c) is factored (exactly: powers of two) and the
                         refinement runs against the ORIGINAL A with x = C (LU)^-1 R b corrections, so backward errors, the
                         stopping rule and the fp64 fallback keep their meaning.  Keeps matrices with widely different row or
                         column magnitudes inside the fp16 range.  Costs two HBM passes over A; when scales are applied the
                         cast of A is an eager pass (lazy_touch does not apply) and mplu_gesv_host copies A before
                         factoring (stream_host does not apply).  When no scale is applied, everything after the two passes
                         is the equilibrate = 0 computation, bit for bit.  See mplu_get_equilibration. */
} mplu_options;

typedef struct mplu_stats {
    int n;
    int iters;              /* refinement (correction) solves performed */
    int converged;          /* 1 if the stopping rule was met */
    int status_bits;        /* bit0 fp16 overflow, bit1 zero pivot, bit2 non-finite inverse */
    double anorm_inf;       /* ||A||_inf */
    double bnorm_inf;       /* ||b||_inf */
    double xnorm_inf;       /* ||x||_inf */
    double rnorm_inf;       /* ||b - A x||_inf, fp64 */
    double backward_error;  /* rnorm / (anorm*xnorm + bnorm) */
    double first_backward_error; /* same quantity after the un-refined first solve */
    float factor_ms;        /* device time of the factorization (CUDA events) */
    float solve_ms;         /* device time of first solve + refinement */
    float total_ms;         /* factor + solve (+ copies for the host variant) */
    float h2d_ms, d2h_ms;   /* host variant only */
    int gemm_launches;      /* tcgen05 GEMM launches in the factorization */
    int kernel_launches;    /* all kernel launches (factor + solve) */
    int trailing_launches;  /* rank-nb trailing updates among them (the dominant kernel) */
    float trailing_ms;      /* summed device time of those launches (CUDA events on the launching stream) */
    double trailing_flops;  /* their algorithmic flops, 2*M*N*K each */
    double trailing_bytes;  /* their algorithmic C traffic, 8*M*N bytes each (fp32 read + write) */
    int gmres_iters;        /* MPLU_REFINE_GMRES: Krylov steps summed over the refinement iterations */
    int precision_used;     /* MPLU_FP16 / MPLU_BF16: differs from the request after a bf16 fallback */
    int fp64_fallback;      /* 1: the solution comes from the full-precision fallback (opts.fp64_fallback) */
    int dsgesv_iter;        /* LAPACK dsgesv's ITER: >= 0 refinement iterations of a successful mixed-precision solve; < 0 the
                               fallback ran: -2 low-precision overflow, -3 low-precision factorization unusable (zero pivot),
                               -(max_iters + 1) refinement did not converge */
    int equed;              /* opts.equilibrate: LAPACK's EQUED of the mixed-precision factorization, 0 N (no scaling), 1 R (rows),
                               2 C (columns), 3 B (both); reported also when the fp64 fallback then solved the original system */
} mplu_stats;

void mplu_default_options(mplu_options *opts);
/* sizeof(mplu_options) / sizeof(mplu_stats) of the library, for bindings that mirror the structs */
int mplu_sizeof_options(void);
int mplu_sizeof_stats(void);

int mplu_create(mplu_context **ctx, int device);
void mplu_destroy(mplu_context *ctx);

/* Factor the n x n fp64 matrix dA (device memory, column-major, lda) without pivoting: blocked right-looking LU,
 * fp16/bf16 operands, fp32 accumulation and fp32 factor storage inside the context.  dA is not modified.
 * Replaces the panel loop of MPF (MPF.cu:100-241) for the no-pivot case. */
int mplu_factor_device(mplu_context *ctx, int n, const double *dA, long long lda, const mplu_options *opts);

/* Solve A x = b with the stored factors and fp64 iterative refinement against the ORIGINAL dA. */
int mplu_solve_device(mplu_context *ctx, const double *dA, long long lda, const double *db, double *dx,
                      mplu_stats *stats);

/* factor + solve, device-resident inputs (the headline metric's timed region). */
int mplu_gesv_device(mplu_context *ctx, int n, const double *dA, long long lda, const double *db, double *dx,
                     const mplu_options *opts, mplu_stats *stats);

/* factor + solve from HOST buffers (pageable or pinned): H2D of A and b, D2H of x inside the call. */
int mplu_gesv_host(mplu_context *ctx, int n, const double *hA, long long lda, const double *hb, double *hx,
                   const mplu_options *opts, mplu_stats *stats);

/* ---- several right-hand sides: A X = B (LAPACK dsgesv's NRHS / B / LDB / X / LDX) ----
 * B and X are column-major n x nrhs (leading dimensions ldb, ldx >= n) in the memory space of the variant.  B is not
 * modified; rows n .. ldx-1 of X are not written.  The regions spanned by B and X must not overlap (MPLU_E_ARG).
 * Refinement runs over the block like dsgesv: every column is refined until all columns meet the stopping rule of the
 * single-vector solve (or max_iters).  A column's result does not depend on its position in B or on the other columns;
 * the columns share only the iteration count.  A and the factors are streamed once per block of columns.
 * opts.refinement = MPLU_REFINE_GMRES runs the Krylov correction column by column (not batched).
 * nrhs = 1 is exactly mplu_solve_device / mplu_gesv_device / mplu_gesv_host.
 * berr: null, or a host array of nrhs doubles receiving each column's backward error ||r_j|| / (||A|| ||x_j|| + ||b_j||)
 * (infinity norms; 0 for a column solved exactly, e.g. a zero column).
 * mplu_stats for nrhs > 1: iters is shared by all columns; converged = every column converged; backward_error and
 * first_backward_error are maxima over the columns; rnorm_inf, xnorm_inf and bnorm_inf are those of the worst column. */
int mplu_solve_device_nrhs(mplu_context *ctx, int nrhs, const double *dA, long long lda, const double *dB, long long ldb,
                           double *dX, long long ldx, double *berr, mplu_stats *stats);
int mplu_gesv_device_nrhs(mplu_context *ctx, int n, int nrhs, const double *dA, long long lda, const double *dB,
                          long long ldb, double *dX, long long ldx, const mplu_options *opts, double *berr,
                          mplu_stats *stats);
/* B is copied to the device alongside A (block column by block column with opts.stream_host), X is copied back */
int mplu_gesv_host_nrhs(mplu_context *ctx, int n, int nrhs, const double *hA, long long lda, const double *hB,
                        long long ldb, double *hX, long long ldx, const mplu_options *opts, double *berr,
                        mplu_stats *stats);

/* Copy the fp32 L\U factors (unit-lower L below the diagonal, U on/above: the dgetrf layout MPF returns) widened
 * to fp64 into a column-major n x n array; `on_device` selects the destination memory space.  After an equilibrated
 * factorization these are the factors of diag(r) A diag(c) (mplu_get_equilibration). */
int mplu_get_factors(mplu_context *ctx, double *LU, long long ldlu, int on_device);

/* The equilibration of the last factorization (opts.equilibrate): *equed (may be null) = 0 N / 1 R / 2 C / 3 B, and the
 * row / column scales r, c (n doubles each, may be null; `on_device` selects their memory space).  A side that was not
 * applied reads as ones, so the factors are always those of diag(r) A diag(c).  MPLU_E_NOTFACTORED before any
 * factorization. */
int mplu_get_equilibration(mplu_context *ctx, int *equed, double *r, double *c, int on_device);

/* The stream all work of this context is enqueued on (a cudaStream_t). */
void *mplu_stream(mplu_context *ctx);

/* ---- kernel-level entry points (used by the parity tests and by callers that bring their own orchestration) ---- */

/* C(MxN, fp32, col-major) = beta*C + alpha * A(MxK) * B(KxN); A,B 16-bit column-major device arrays.
 * variant: 0 CG1, 1 CG2 (A column-major), 2/3 same with A passed as its transpose (K x M column-major).
 * H (optional) receives the 16-bit copy of the result scaled by hscale. */
int mplu_gemm16(int variant, int bf16, int M, int N, int K, float alpha, const void *dA, long long lda,
                const void *dB, long long ldb, float beta, float *dC, long long ldc, void *dH, long long ldh,
                float hscale, int max_sms, void *stream);

/* No-pivot LU of one 128x128 fp32 block in place + explicit inverses (fp32, column-major 128x128 each). */
int mplu_diag_lu128(float *dW, long long ldw, float *dLinv, float *dUinv, void *stream);

/* Host logic of the left-looking schedule (no device needed): the bulk lane's update plan for an n x n matrix tiled
 * by nb as (step, k, m0, m1, mandatory) quintuples -- update k applied to block columns [m0, m1) during step `step`.
 * Returns the number of ops; at most `max` are written to out[0 .. 5*max). */
int mplu_debug_plan_left(int n, int nb, int eager, int *out, int max);
int mplu_debug_tile_bounds(int n, int nb, int edge_nb, int *out, int max);
int mplu_debug_plan_left_edge(int n, int nb, int edge_nb, int eager, int *out, int max);

/* Dry run of the device factorization schedule (host logic only, no device needed): every launch with the lane it
 * runs on and the array regions it reads / writes, and every cross-lane event record / wait, serialised as ints (see
 * csrc/lu.cu).  Returns the number of ints of the full trace; at most `max` are written.  tests/test_schedule_trace.py
 * replays it with vector clocks to prove the schedule free of read-after-write / write-after-read races. */
int mplu_debug_trace(int n, int nb, const mplu_options *opts, int *out, int max);

/* r = b - A x in fp64; norms[0] = ||r||_inf, norms[1] = ||x||_inf (device array of 2 doubles). */
int mplu_residual(int n, const double *dA, long long lda, const double *dx, const double *db, double *dr,
                  double *dnorms, void *stream);

/* Cooperative launches of the drop-in kernels HGETF2_kernel / dgetf2_native_npv (include/hgetf2_kernel.h,
 * include/dgetf2_native_npv.h) with the reference caller's geometry, on device-resident column-major panels. */
int mplu_hgetf2(void *d_panel_fp16, int ld, int rows, int cols, int *d_ipiv_panel, void *stream);
int mplu_dgetf2_npv(int m, int n, double *d_panel, int ld, void *stream);

/* Synthetic input in device memory: a(i,j) = (splitmix64(seed<<40 | i<<20 | j) % 100) / 10 -- the value set of the
 * reference generator (matrix_generator.cpp:66) -- with, if `dominant`, the diagonal replaced by the column's
 * off-diagonal sum + 1.  db (optional) receives b = A * ones. */
int mplu_generate(int n, unsigned long long seed, int dominant, double *dA, long long lda, double *db, void *stream);

/* Device memory for callers that do not link the CUDA runtime themselves (drivers/benchmark.cpp --gen): plain cudaMalloc /
 * cudaFree / synchronous device-to-host cudaMemcpy on the current device. */
int mplu_device_alloc(void **ptr, unsigned long long bytes);
int mplu_device_free(void *ptr);
int mplu_device_to_host(void *dst, const void *src, unsigned long long bytes);

/* ---- 2D block-cyclic solver across the GPUs of one box (SURVEY.md section 8e; the reference is single-GPU,
 * MPF.cu:77).  The n x n matrix is cut into nb x nb tiles, tile (I,J) lives on process (I mod P, J mod Q) of a
 * P x Q grid, each process stores its tiles in ScaLAPACK local order (column-major mloc x nloc).  One process per
 * GPU, NCCL over NVLink for the panel broadcasts and the refinement's reductions (libnccl.so.2 is loaded with dlopen
 * on first use; single-GPU users never need it). */
typedef struct mplu_dist mplu_dist;

/* rank 0 creates the 128-byte NCCL unique id; the host program hands it to every rank (any transport) */
int mplu_dist_unique_id(void *id128);
/* this process becomes rank `rank` = p*Q + q of nranks = P*Q, computing on `device` */
int mplu_dist_create(mplu_dist **out, int device, int rank, int nranks, int P, int Q, const void *id128);
/* all P*Q logical ranks inside this process on one device, collectives as device copies (tests; no NCCL needed) */
int mplu_dist_create_local(mplu_dist **out, int device, int P, int Q);
void mplu_dist_destroy(mplu_dist *d);
/* number of logical ranks hosted by this process (1 with NCCL, P*Q in local mode) */
int mplu_dist_num_local(const mplu_dist *d);
/* grid coordinates and local extents of logical rank i of this process for an n x n matrix tiled by nb */
int mplu_dist_local_shape(const mplu_dist *d, int i, int n, int nb, int *p, int *q, long long *mloc, long long *nloc);
/* factor + solve: dA[i] / lda[i] = local fp64 tiles of logical rank i (device), db[i] / dx[i] = FULL-length right-hand
 * side and solution (device, replicated on every rank).  Requires n % nb == 0 and nb % 128 == 0. */
int mplu_dist_gesv(mplu_dist *d, int n, int nb, const double *const *dA, const long long *lda,
                   const double *const *db, double *const *dx, const mplu_options *opts, mplu_stats *stats);
/* the same solve from HOST buffers (local tiles hA[i], full hb[i]; full hx[i] out): H2D / D2H inside the call */
int mplu_dist_gesv_host(mplu_dist *d, int n, int nb, const double *const *hA, const long long *lda,
                        const double *const *hb, double *const *hx, const mplu_options *opts, mplu_stats *stats);
void mplu_dist_release_staging(mplu_dist *d);
/* local fp32 L\U factors of logical rank i widened to fp64 (device, column-major mloc x nloc, leading dimension ld) */
int mplu_dist_get_local_factors(mplu_dist *d, int i, double *dLU, long long ld);
/* local tiles of the synthetic dominant system of mplu_generate for process (p,q), and the full b = A*1 */
int mplu_generate_local(int n, unsigned long long seed, int nb, int P, int Q, int p, int q, double *dA_loc,
                        long long lda, double *db_full, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MPLU_H */
