// Internal declarations shared by lu.cu (single-GPU schedule, C ABI) and dist.cu (2D block-cyclic schedule).
// Not part of the public interface (include/mplu.h).
#pragma once
#include "../../include/mplu.h"
#include "gemm_tc.h"
#include "getrf_fused.h"
#include "kernels.h"

#include <functional>
#include <vector>

// dry-run trace of a schedule (lu.cu: trace_*; tests/test_schedule_trace.py)
struct TraceRegion { int arr, r0, r1, c0, c1, write; };
struct TraceOp { int kind, stream, ev, group; std::vector<TraceRegion> regs; };

struct mplu_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int n = 0, npad = 0, cap_npad = 0;
    bool factored = false;
    mplu_options opts{};
    // working storage
    float* W = nullptr;       // npad x npad fp32, column-major (ld = npad): becomes L\U
    uint16_t* Wh = nullptr;   // npad x npad 16-bit shadow of the not yet factored (trailing) part, A-type scale
    uint16_t* Fh = nullptr;   // npad x npad 16-bit shadow of the FACTORS: L part scaled SC_L, U part scaled SC_A
    uint16_t* Linv16 = nullptr;  // nbcap x npad band: inverse of the L factor of tile [T, T+nb) at rows [0,nb), cols [T,T+nb)
    uint16_t* Uinv16 = nullptr;
    uint16_t* Tb1 = nullptr;     // nbcap x nbcap scratch of the inverse merges (L side, U side)
    uint16_t* Tb2 = nullptr;
    int cap_nb = 0;
    void* slab = nullptr;        // the single allocation behind W .. inv_scales
    size_t slab_bytes = 0;
    mplu_context* tile = nullptr;  // nb x nb workspace context in which diagonal tiles are factored (L2-resident)
    float* Linv32 = nullptr;
    float* Uinv32 = nullptr;
    float* inv_scales = nullptr;  // 4 per diagonal block
    float* scales = nullptr;      // SC_COUNT
    float* amax = nullptr;
    double* anorm = nullptr;      // ||A||inf
    double* rowsum_part = nullptr;
    int* status = nullptr;
    unsigned* ready = nullptr;    // step counter of the cooperative triangular-solve kernel
    // refinement
    double* r = nullptr;
    double* partial = nullptr;
    double* norms = nullptr;  // [0] ||r||, [1] ||x||, [2] ||b|| (the layout of RefineOps::norms for one column)
    float* y = nullptr;       // 2*npad
    int nchunk = 64;
    // several right-hand sides (mplu_*_nrhs): allocated on the first call with nrhs > 1, freed with the other work arrays
    double* rb_R = nullptr;        // n x nrhs residual block (ld n)
    double* rb_partial = nullptr;  // kResidualChunks * kResidualBlock * n
    double* rb_norms = nullptr;    // per column ||r||, ||x||, then ||b|| per column
    float* rb_y = nullptr;         // 2 * npad * kSolveBlock (the batched solve's fp32 work blocks)
    int rb_cap_n = 0, rb_cap_npad = 0, rb_cap_nrhs = 0;
    // equilibration (opts.equilibrate, equil.cu): the scales of the stored factors (W holds diag(eq_r) A diag(eq_c)) and
    // EQUED (bit 0 rows, bit 1 columns applied); eq_D = n x eq_cap_k correction scratch, allocated on first use
    int equed = 0;
    double* eq_r = nullptr; double* eq_c = nullptr;
    unsigned long long* eq_words = nullptr;
    int eq_cap_n = 0;
    double* eq_D = nullptr;
    size_t eq_D_cap = 0;
    // GMRES-IR workspace (gmres.cu)
    double* gm_V = nullptr; double* gm_w = nullptr; double* gm_h = nullptr; double* gm_zero = nullptr;
    int gm_cap_n = 0, gm_cap_m = 0;
    // staging for the host variant
    double* dA_stage = nullptr; size_t dA_cap = 0;
    double* db_stage = nullptr; double* dx_stage = nullptr; size_t dv_cap = 0;
    // streamed host variant: copy stream, one event per block column (ev_copy[copy_last] = last byte arrived)
    cudaStream_t copy = nullptr;
    cudaEvent_t ev_copy[512] = {};
    int copy_last = 0;
    // left-looking prologue (first touch overlapped with the first diagonal tile)
    cudaEvent_t ev_pro[2] = {nullptr, nullptr};
    bool prologue_done = false, used_early_scale = false, allow_early = true;
    // lazy first touch (left-looking schedule): only the first block column / block row of A are cast up front, every
    // other tile takes the addend of its FIRST update from the original fp64 matrix (aref: device copy of {A, lda});
    // ||A||_inf is then formed by the first residual pass (anorm_pending)
    mplu::ARef* aref = nullptr;
    bool lazy = false, anorm_pending = false;
    // dry run: non-null = record the schedule instead of launching it
    std::vector<TraceOp>* trace = nullptr;
    int trace_group = 0;
    // fused GETRF (getrf_fused.cu): step programs of the diagonal blocks, recorded once per (geometry, options) by running
    // the recursion with `rec` set, kept on the device; one barrier word per fused launch of a factorization
    struct FusedProg { int T, c0, w; size_t offset; int num_steps, num_problems; };
    struct FusedRecorder { std::vector<mplu::FusedStep> steps; std::vector<mplu::FusedProblem> problems; bool unsupported = false; };
    std::vector<FusedProg> fprogs;
    std::vector<unsigned char> fprog_host;
    std::vector<long long> fprog_key;
    unsigned char* fprog_dev = nullptr;
    size_t fprog_cap = 0, fprog_uploaded = 0;
    FusedRecorder* rec = nullptr;
    unsigned* fbar = nullptr;
    int fbar_cap = 0, fbar_next = 0;
    // development aid (mplu_debug_fused_profile): per fused launch of the last factorization, which program it ran and
    // a slice of kFusedProfSlots time stamps
    static constexpr int kFusedProfSlots = 640;
    long long* fprof = nullptr;
    bool fprof_on = false, fprof_sub = false;
    std::vector<int> fprof_prog;  // launch index -> index into fprogs
    mplu::FusedMaps fmaps;
    // dataflow GETRF (getrf_flow.cu): per diagonal block one blob [FlowLeaf ...][FusedProblem ...][FlowTask ...], built once
    // per (geometry, options) and kept on the device; every launch of a factorization takes its own slice of zeroed counters
    struct FlowProg { int T, c0, w; size_t off_leaves, off_problems, off_tasks; int num_leaves, num_problems, num_tasks, num_main, num_counters; };
    std::vector<FlowProg> flow_progs;
    std::vector<unsigned char> flow_host;
    std::vector<long long> flow_key;
    unsigned char* flow_dev = nullptr;
    size_t flow_cap = 0, flow_uploaded = 0;
    unsigned* fctr = nullptr;
    int fctr_cap = 0, fctr_next = 0;
    // development aid (mplu_debug_flow_profile): %globaltimer stamps of ONE dataflow launch of the last factorization
    long long* flow_prof = nullptr;
    size_t flow_prof_cap = 0;
    int flow_prof_launch = -1, flow_launch_count = 0, flow_prof_prog = -1;
    // GEMM operand views (tensor maps) of the 16-bit arrays
    struct Operand16 {
        uint16_t* base = nullptr;
        long long ld = 0;
        CUtensorMap mapA, mapB1, mapB2;  // as A operand (64x64 boxes), as B operand for 1-CTA / CTA-pair tiles
    } opWh, opFh, opLinv, opUinv, opT1, opT2;
    int gemm_launches = 0, kernel_launches = 0;
    // look-ahead / graph
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    static constexpr int kMaxSteps = 512;
    cudaEvent_t ev_step[4 * kMaxSteps] = {};  // per step: GETRF done, next-tile TRSM done, b2 done, b3a done
    cudaGraphExec_t graph_exec = nullptr;
    std::vector<long long> gkey;  // what the cached graph was captured for (factor_impl)
    int g_gemm_launches = 0, g_kernel_launches = 0, g_trail_count = 0;
    double g_trail_flops = 0, g_trail_bytes = 0;
    bool capturing = false;
    int num_sms = 0;
    // per-launch timing of the trailing updates (events are cheap: <= npad/nb pairs per factorization)
    static constexpr int kMaxTrail = 1024;
    cudaEvent_t trail_ev[2 * kMaxTrail] = {};
    int trail_count = 0;
    double trail_flops = 0, trail_bytes = 0;
    // optional timeline marks (development aid, mplu_debug_timeline): tag + event
    static constexpr int kMaxMarks = 4096;
    cudaEvent_t mark_ev[kMaxMarks] = {};
    int mark_tag[kMaxMarks] = {};
    int mark_count = 0;
    bool marks_on = false;
};

namespace mplu_detail {

#define CK(expr)                                  \
    do {                                          \
        cudaError_t _e = (expr);                  \
        if (_e != cudaSuccess) return (int)_e;    \
    } while (0)
#define CKI(expr)                  \
    do {                           \
        int _e = (expr);           \
        if (_e != 0) return _e;    \
    } while (0)

using Operand16 = mplu_context::Operand16;

struct GemmCall {
    const Operand16* A; int a_r0, a_c0;  // A block origin inside its parent (row m0, col k0)
    const Operand16* B; int b_r0, b_c0;  // B block origin inside its parent (row k0, col n0)
    int M, N, K;
    float* C; long long ldc;             // fp32 output (null: none), already offset to the block origin
    bool accumulate;                     // out = C + alpha*acc (else alpha*acc)
    uint16_t* H; long long ldh;          // 16-bit output (null: none), already offset
    int h_rows, h_cols;                  // H is written where (m < h_rows || n < h_cols)
    float alpha;                         // static factor times *alpha_p1 times *alpha_p2 (device, null = 1)
    const float* alpha_p1;
    const float* alpha_p2;
    const float* hscale_p;               // H = cvt16(out * *hscale_p)
    int tri = 0;                         // GemmTri: which operand is triangular (its zero part of K is skipped)
    bool stream_c = false;               // C / H are far larger than L2 and touched once: streaming cache policy
    bool from_a = false;                 // accumulate onto the ORIGINAL fp64 matrix (a tile's first update) instead of C
};

// Where a piece of the schedule runs: stream + SM budget (0 = all SMs).
struct Lane {
    cudaStream_t st;
    int sms;
    bool pdl = false;  // chain lane: opts.pdl == 2 launches its kernels programmatically
};


int make_operand(Operand16* o, uint16_t* base, uint64_t rows, uint64_t cols, uint64_t ld);
// launch one product / two independent products (grouped) on a lane of context c
int run_gemm(mplu_context* c, const Lane& ln, const mplu_detail::GemmCall& g);
int run_gemm_pair(mplu_context* c, const Lane& ln, const GemmCall& g0, const GemmCall& g1);
// GETRF of the nb x nb matrix already resident in c->W (fp32, ld = c->npad = nb): casts the shadow with the scales in
// c->scales, factors the tile recursively and leaves L\U in c->W, the merged 16-bit inverses in c->Linv16 /
// c->Uinv16 (nb x nb, ld = c->cap_nb), their scales in c->inv_scales[0..3] and the fp32 128-block inverses in
// c->Linv32 / c->Uinv32.  Everything is enqueued on `st`.
int getrf_resident_tile(mplu_context* c, cudaStream_t st, int w);
int ensure_work(mplu_context* c, int n);
// GMRES-IR: solve A d = r (n doubles on the device) by GMRES preconditioned with the stored factors, x += d (gmres.cu)
int gmres_correction(mplu_context* c, const double* dA, long long lda, const double* r, double* dx, int* inner);
// eq_D holds at least `elems` doubles
int ensure_equil_scratch(mplu_context* c, size_t elems);
// dsgesv-style full-precision redo of a solve the low-precision factors could not deliver (fp64_fallback.cu); `why` is the
// MPLU_E_* code the mixed-precision path ended with.  nrhs column-major right-hand sides (B, ldb) and solutions (X, ldx):
// one fp64 factorization, then every column is solved and refined on its own; berr (host, may be null) receives each
// column's backward error, stats the worst column's figures
int fp64_fallback_solve(mplu_context* c, int n, const double* dA, long long lda, int nrhs, const double* dB, long long ldb,
                        double* dX, long long ldx, int why, double* berr, mplu_stats* stats);
// the per-column backward error ||r|| / (||A|| ||x|| + ||b||) (0 for r = 0: a zero column is solved exactly)
inline double backward_error(double rn, double an, double xn, double bn) { return rn == 0.0 ? 0.0 : rn / (an * xn + bn); }

// LAPACK dsgesv's iterative refinement of k columns that share the iteration count (refine, lu.cu).  The caller enqueues
// the device work; refine reads the norms back, applies the stopping rule and counts.  Every operation returns 0 or an
// error code.
struct RefineOps {
    // device norms, read back on st: [2j] ||r_j||_inf, [2j+1] ||x_j||_inf, [2k+j] ||b_j||_inf; and ||A||_inf
    const double* norms;
    const double* anorm;
    cudaStream_t st;
    std::function<int()> first_solve;                 // the ||b_j|| and X = (LU)^-1 B
    std::function<int(bool* formed_anorm)> residual;  // R = B - A X and its norms; *formed_anorm: this pass also formed ||A||
    std::function<int(int* krylov_steps)> correct;    // X += the correction computed from R
    std::function<int()> wait;                        // until the norms have arrived on the host
};
struct RefineColumn { double rnorm, xnorm, bnorm, berr, first_berr; };
struct RefineResult {
    std::vector<RefineColumn> col;
    double anorm = 0.0;
    int iters = 0, converged = 0, gmres_iters = 0;
};
// max_iters <= 0: dsgesv's 30.  tol <= 0: ||r_j|| <= ||x_j|| ||A|| eps sqrt(n), else ||r_j|| <= tol ||A|| ||x_j||
int refine(const RefineOps& ops, int n, int k, int max_iters, double tol, RefineResult* res);
// berr (host, may be null) = every column's backward error; the refinement fields of stats (may be null) = those of the
// worst column (the largest backward error, the first NaN), first_backward_error = the largest first-solve one
void refine_stats(const RefineResult& res, int n, double* berr, mplu_stats* stats);
// 0 when converged, else what the status bits of the factorization explain, else MPLU_E_NOCONV
int refine_rc(int converged, int status_bits);
// LAPACK dsgesv's ITER for a mixed-precision solve that ended with rc after iters corrections
int dsgesv_iter(int rc, int iters);

}  // namespace mplu_detail
