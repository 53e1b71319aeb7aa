// Host orchestration of the blocked right-looking no-pivot LU + fp64 iterative refinement, and the C ABI of
// include/mplu.h.  This is the B200-native counterpart of the panel loop in /root/reference/MPF.cu:100-241:
//   reference per panel (r = 32):  gather -> fp16 pivot search -> LASWP -> fp64 panel LU -> Dtrsm -> rank-32 Dgemm
//   here per diagonal tile (nb = 1024..2048), all products on the tcgen05 GEMM with 16-bit operands, fp32 accumulate:
//     GETRF   the nb x nb diagonal tile, recursively, CARRYING EXPLICIT INVERSES: a 128x128 leaf (diag_lu) returns
//             L11\U11, inv(L11), inv(U11); a node of width w = 2h does  U12 = inv(La) A12,  L21 = A21 inv(Ua),
//             A22 -= L21 U12, recurses, then merges  inv(L) = [inv(La) 0; -inv(Lb) L21 inv(La), inv(Lb)]  (same for U)
//     TRSM    L panel = A21 inv(U11) and U panel = inv(L11) A12: ONE GEMM each with the tile's nb x nb inverse
//             (replaces cublasDtrsm, MPF.cu:215-225, and the 2*nb/128-1 dependent launches of a recursive TRSM)
//     GEMM    A22 -= L21 U12 (replaces cublasDgemm, MPF.cu:230-239)
// Two lanes (streams with disjoint SM budgets), depth-1 look-ahead:
//   chain lane: TRSM of the NEXT tile's rows/columns -> update of the next diagonal tile -> GETRF of it   (critical path)
//   bulk lane:  TRSM of the remaining rows/columns -> update of the next block column/row -> rest of the trailing matrix
// The whole schedule is captured once into a CUDA graph per (n, options) and replayed.
// No host<->device round trips inside the loop (the reference does one per panel, MPF.cu:146,158).
#include "lu_internal.h"
#include "../../include/mplu_debug.h"

#include <algorithm>
#include <cstring>
#include <functional>
#include <vector>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

using namespace mplu;
using namespace mplu_detail;

namespace mplu_detail {

void free_work(mplu_context* c) {
    if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
    cudaFree(c->slab);
    cudaFree(c->rowsum_part); cudaFree(c->r); cudaFree(c->partial); cudaFree(c->y);
    cudaFree(c->fprog_dev); cudaFree(c->fbar); cudaFree(c->fprof);
    cudaFree(c->flow_dev); cudaFree(c->fctr); cudaFree(c->flow_prof);
    c->flow_dev = nullptr; c->flow_cap = 0; c->flow_uploaded = 0; c->fctr = nullptr; c->fctr_cap = 0;
    c->flow_prof = nullptr; c->flow_prof_cap = 0;
    c->flow_progs.clear(); c->flow_host.clear(); c->flow_key.clear();
    c->fprof = nullptr;
    c->fprog_dev = nullptr; c->fprog_cap = 0; c->fbar = nullptr; c->fbar_cap = 0;
    c->fprogs.clear(); c->fprog_host.clear(); c->fprog_key.clear(); c->fprog_uploaded = 0;
    c->slab = nullptr; c->slab_bytes = 0;
    c->W = nullptr; c->Wh = c->Fh = nullptr; c->Linv16 = c->Uinv16 = c->Tb1 = c->Tb2 = nullptr;
    c->Linv32 = c->Uinv32 = nullptr; c->cap_nb = 0;
    c->inv_scales = nullptr; c->rowsum_part = nullptr; c->r = c->partial = nullptr; c->y = nullptr;
    c->cap_npad = 0;
    cudaFree(c->rb_R); cudaFree(c->rb_partial); cudaFree(c->rb_norms); cudaFree(c->rb_y);
    c->rb_R = c->rb_partial = c->rb_norms = nullptr; c->rb_y = nullptr;
    c->rb_cap_n = c->rb_cap_npad = c->rb_cap_nrhs = 0;
}

// workspaces of the multi-column solve, sized for the factored n and nrhs columns (kept and grown across calls)
int ensure_rhs_work(mplu_context* c, int nrhs) {
    if (c->rb_R && c->n <= c->rb_cap_n && c->npad <= c->rb_cap_npad && nrhs <= c->rb_cap_nrhs) return 0;
    const int cap_n = std::max(c->n, c->rb_cap_n), cap_npad = std::max(c->npad, c->rb_cap_npad),
              cap_nrhs = std::max(nrhs, c->rb_cap_nrhs);
    cudaFree(c->rb_R); cudaFree(c->rb_partial); cudaFree(c->rb_norms); cudaFree(c->rb_y);
    c->rb_R = c->rb_partial = c->rb_norms = nullptr; c->rb_y = nullptr;
    c->rb_cap_n = c->rb_cap_npad = c->rb_cap_nrhs = 0;
    const size_t kb = (size_t)std::min(cap_nrhs, kResidualBlock);
    CK(cudaMalloc(&c->rb_R, (size_t)cap_n * cap_nrhs * sizeof(double)));
    CK(cudaMalloc(&c->rb_partial, (size_t)kResidualChunks * kb * cap_n * sizeof(double)));
    CK(cudaMalloc(&c->rb_norms, 3 * (size_t)cap_nrhs * sizeof(double)));
    CK(cudaMalloc(&c->rb_y, 2 * (size_t)cap_npad * kSolveBlock * sizeof(float)));
    c->rb_cap_n = cap_n; c->rb_cap_npad = cap_npad; c->rb_cap_nrhs = cap_nrhs;
    return 0;
}

int ensure_equil_scratch(mplu_context* c, size_t elems) {
    if (elems <= c->eq_D_cap) return 0;
    cudaFree(c->eq_D);
    c->eq_D = nullptr; c->eq_D_cap = 0;
    CK(cudaMalloc(&c->eq_D, elems * sizeof(double)));
    c->eq_D_cap = elems;
    return 0;
}

// opts.equilibrate = 1: dgeequb's scales of A into c->eq_r / c->eq_c and dlaqge's EQUED into c->equed.  The host needs
// EQUED to choose the first touch, so it is read back here (one synchronisation, before any graph launch).
int equilibrate(mplu_context* c, const double* dA, long long lda) {
    const int n = c->n;
    cudaStream_t st = c->stream;
    if (n > c->eq_cap_n) {
        cudaFree(c->eq_r); cudaFree(c->eq_c);
        c->eq_r = c->eq_c = nullptr; c->eq_cap_n = 0;
        CK(cudaMalloc(&c->eq_r, (size_t)n * sizeof(double)));
        CK(cudaMalloc(&c->eq_c, (size_t)n * sizeof(double)));
        c->eq_cap_n = n;
    }
    if (!c->eq_words) CK(cudaMalloc(&c->eq_words, EQ_WORDS * sizeof(unsigned long long)));
    // rowsum_part (nchunk x npad) is free until the first touch: the row pass keeps its per-chunk maxima there
    CKI(launch_equilibrate(dA, lda, n, c->rowsum_part, c->nchunk, c->eq_r, c->eq_c, c->eq_words, st));
    unsigned long long equed = 0;
    CK(cudaMemcpyAsync(&equed, c->eq_words + EQ_EQUED, sizeof(equed), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    c->equed = (int)equed;
    return 0;
}

int effective_nb(const mplu_context* c, int npad) {
    int NB = c->opts.nb;
    if (NB < kDiagBlock) NB = kDiagBlock;
    NB = (NB / kDiagBlock) * kDiagBlock;
    return NB > npad ? npad : NB;
}

int make_operand(Operand16* o, uint16_t* base, uint64_t rows, uint64_t cols, uint64_t ld) {
    o->base = base;
    o->ld = (long long)ld;
    if (make_tmap_16bit(&o->mapA, base, rows, cols, ld, 64, 64)) return MPLU_E_TMAP;
    if (make_tmap_16bit(&o->mapB1, base, rows, cols, ld, 64, 256)) return MPLU_E_TMAP;
    if (make_tmap_16bit(&o->mapB2, base, rows, cols, ld, 64, 128)) return MPLU_E_TMAP;
    return 0;
}

int ensure_work(mplu_context* c, int n) {
    const int npad = ((n + kDiagBlock - 1) / kDiagBlock) * kDiagBlock;
    c->n = n;
    c->npad = npad;
    const int NB = effective_nb(c, npad);
    if (npad > c->cap_npad || NB > c->cap_nb) {
        free_work(c);
        const size_t np = (size_t)npad, nb = (size_t)NB;
        // every array the GEMMs and diag_lu touch lives in ONE allocation, so that a diagonal tile's whole working set
        // can be named by a single L2 access-policy window (see tile workspace below)
        auto up = [](size_t b) { return (b + 1023) & ~(size_t)1023; };
        const size_t szW = up(np * np * sizeof(float)), sz16 = up(np * np * sizeof(uint16_t)), szI = up(np * nb * sizeof(uint16_t)),
                     szT = up(nb * nb * sizeof(uint16_t)), sz32 = up(np * kDiagBlock * sizeof(float)),
                     szS = up(4 * (np / kDiagBlock) * sizeof(float));
        c->slab_bytes = szW + 2 * sz16 + 2 * szI + 2 * szT + 2 * sz32 + szS;
        CK(cudaMalloc(&c->slab, c->slab_bytes));
        char* q = reinterpret_cast<char*>(c->slab);
        c->W = reinterpret_cast<float*>(q); q += szW;
        c->Wh = reinterpret_cast<uint16_t*>(q); q += sz16;
        c->Fh = reinterpret_cast<uint16_t*>(q); q += sz16;
        c->Linv16 = reinterpret_cast<uint16_t*>(q); q += szI;
        c->Uinv16 = reinterpret_cast<uint16_t*>(q); q += szI;
        c->Tb1 = reinterpret_cast<uint16_t*>(q); q += szT;
        c->Tb2 = reinterpret_cast<uint16_t*>(q); q += szT;
        c->Linv32 = reinterpret_cast<float*>(q); q += sz32;
        c->Uinv32 = reinterpret_cast<float*>(q); q += sz32;
        c->inv_scales = reinterpret_cast<float*>(q);
        // diag_lu only stores the triangles of the fp32 inverses: the other halves stay zero from here on
        CK(cudaMemset(c->Linv32, 0, np * kDiagBlock * sizeof(float)));
        CK(cudaMemset(c->Uinv32, 0, np * kDiagBlock * sizeof(float)));
        CK(cudaMalloc(&c->rowsum_part, (size_t)c->nchunk * np * sizeof(double)));
        CK(cudaMalloc(&c->r, np * sizeof(double)));
        CK(cudaMalloc(&c->partial, (size_t)c->nchunk * np * sizeof(double)));
        CK(cudaMalloc(&c->y, 2 * np * sizeof(float)));
        // fused GETRF: step programs (a leaf costs 48 bytes, a recursion node < 1.2 KiB) and one barrier word per launch
        c->fprog_cap = (np / kDiagBlock) * 1536 + 65536;
        CK(cudaMalloc(&c->fprog_dev, c->fprog_cap));
        c->fbar_cap = (int)(np / kDiagBlock) + 16;
        CK(cudaMalloc(&c->fbar, c->fbar_cap * sizeof(unsigned)));
        CK(cudaMemset(c->fbar, 0, c->fbar_cap * sizeof(unsigned)));
        {   // dataflow GETRF: task lists (a block of b 128-blocks has ~b^3/3 tile tasks of 32 bytes) and dependency counters
            const size_t b = nb / kDiagBlock, tiles = np / nb + 1;
            c->flow_cap = tiles * (32 * (b * b * b / 3 + 4 * b * b + 16) + 1024 * b) + 65536;
            CK(cudaMalloc(&c->flow_dev, c->flow_cap));
            c->fctr_cap = (int)(tiles * (3 * b * b + 8 * b + 16)) + 64;
            CK(cudaMalloc(&c->fctr, (size_t)c->fctr_cap * sizeof(unsigned)));
            CK(cudaMemset(c->fctr, 0, (size_t)c->fctr_cap * sizeof(unsigned)));
        }
        c->cap_npad = npad;
        c->cap_nb = NB;
    }
    // operand views over the parents (dims = allocation so that out-of-range boxes are zero filled)
    const uint64_t np = (uint64_t)npad, nbc = (uint64_t)c->cap_nb;
    CKI(make_operand(&c->opWh, c->Wh, np, np, np));
    CKI(make_operand(&c->opFh, c->Fh, np, np, np));
    CKI(make_operand(&c->opLinv, c->Linv16, nbc, np, nbc));
    CKI(make_operand(&c->opUinv, c->Uinv16, nbc, np, nbc));
    CKI(make_operand(&c->opT1, c->Tb1, nbc, nbc, nbc));
    CKI(make_operand(&c->opT2, c->Tb2, nbc, nbc, nbc));
    const Operand16* ops[FM_COUNT] = {&c->opWh, &c->opFh, &c->opLinv, &c->opUinv, &c->opT1, &c->opT2};
    for (int i = 0; i < FM_COUNT; ++i) {
        c->fmaps.a[i] = ops[i]->mapA;
        c->fmaps.b[i] = ops[i]->mapB2;
        const bool band = i == FM_LINV || i == FM_UINV, scratch = i == FM_T1 || i == FM_T2;
        if (make_tmap_plain(&c->fmaps.h[i], ops[i]->base, 2, band || scratch ? nbc : np, scratch ? nbc : np, (uint64_t)ops[i]->ld,
                            kDiagBlock, kDiagBlock)) return MPLU_E_TMAP;
    }
    if (make_tmap_plain(&c->fmaps.c, c->W, 4, np, np, np, kDiagBlock, kDiagBlock)) return MPLU_E_TMAP;
    return 0;
}

void resolve_options(mplu_context* c, int n) {
    if (c->opts.nb <= 0) c->opts.nb = n >= 12288 ? 2048 : (n >= 4096 ? 1024 : 512);
}

// c->opts is the caller's REQUEST.  What a call resolves for itself (the nb chosen for this n, the bf16 fallback after an
// fp16 overflow) lives in c->opts only for the duration of that call; the precision actually used is reported through
// mplu_stats::precision_used.
struct OptionsScope {
    mplu_context* c;
    mplu_options requested;
    explicit OptionsScope(mplu_context* ctx) : c(ctx), requested(ctx->opts) {}
    ~OptionsScope() { c->opts = requested; }
};

// ---- dry-run trace (mplu_debug_trace): with c->trace set, the schedule functions record what they WOULD launch --
// every GEMM problem / leaf / cast with the array regions it reads and writes, every event record / wait -- instead of
// launching it.  tests/test_schedule_trace.py replays the trace with vector clocks and checks that every access
// happens-after the accesses it conflicts with: a missing or mis-ordered cross-lane event shows up on the CPU, without
// having to lose a timing-dependent race on a GPU first.
enum TraceKind : int { TK_GEMM = 0, TK_LEAF = 1, TK_RECORD = 2, TK_WAIT = 3, TK_CAST = 4, TK_MEMSET = 5 };
enum TraceArray : int { TA_W = 0, TA_WH = 1, TA_FH = 2, TA_LINV = 3, TA_UINV = 4, TA_T1 = 5, TA_T2 = 6 };

int trace_stream(const mplu_context* c, cudaStream_t st) { return st == c->stream ? 0 : 1; }

void trace_push(mplu_context* c, int kind, cudaStream_t st, int ev, int group, const std::vector<TraceRegion>& regs) {
    TraceOp op;
    op.kind = kind; op.stream = trace_stream(c, st); op.ev = ev; op.group = group; op.regs = regs;
    c->trace->push_back(op);
}

// which 16-bit array a (fake, dry-run) pointer lies in, and its (row, col) there for leading dimension ld
bool trace_locate16(const mplu_context* c, const void* p, long long ld, int* arr, int* r, int* col) {
    struct { const uint16_t* base; int id; size_t elems; } tab[] = {
        {c->Wh, TA_WH, (size_t)c->npad * c->npad}, {c->Fh, TA_FH, (size_t)c->npad * c->npad},
        {c->Linv16, TA_LINV, (size_t)c->cap_nb * c->npad}, {c->Uinv16, TA_UINV, (size_t)c->cap_nb * c->npad},
        {c->Tb1, TA_T1, (size_t)c->cap_nb * c->cap_nb}, {c->Tb2, TA_T2, (size_t)c->cap_nb * c->cap_nb}};
    const uint16_t* q = reinterpret_cast<const uint16_t*>(p);
    for (auto& t : tab)
        if (q >= t.base && q < t.base + t.elems) {
            const long long off = q - t.base;
            *arr = t.id; *r = (int)(off % ld); *col = (int)(off / ld);
            return true;
        }
    return false;
}

int trace_operand(const mplu_context* c, const Operand16* o) {
    if (o == &c->opWh) return TA_WH;
    if (o == &c->opFh) return TA_FH;
    if (o == &c->opLinv) return TA_LINV;
    if (o == &c->opUinv) return TA_UINV;
    if (o == &c->opT1) return TA_T1;
    return TA_T2;
}

void trace_gemm(mplu_context* c, const Lane& ln, const GemmCall& g, int group) {
    if (g.M <= 0 || g.N <= 0 || g.K <= 0) return;
    std::vector<TraceRegion> regs;
    regs.push_back({trace_operand(c, g.A), g.a_r0, g.a_r0 + g.M, g.a_c0, g.a_c0 + g.K, 0});
    regs.push_back({trace_operand(c, g.B), g.b_r0, g.b_r0 + g.K, g.b_c0, g.b_c0 + g.N, 0});
    if (g.C) {
        const long long off = g.C - c->W;
        const int r = (int)(off % g.ldc), col = (int)(off / g.ldc);
        if (g.accumulate) regs.push_back({TA_W, r, r + g.M, col, col + g.N, 0});
        regs.push_back({TA_W, r, r + g.M, col, col + g.N, 1});
    }
    if (g.H) {
        int arr = 0, r = 0, col = 0;
        if (trace_locate16(c, g.H, g.ldh, &arr, &r, &col)) {
            const int hr = g.h_rows < g.M ? g.h_rows : g.M, hc = g.h_cols < g.N ? g.h_cols : g.N;
            if (hr > 0) regs.push_back({arr, r, r + hr, col, col + g.N, 1});
            if (hc > 0 && hr < g.M) regs.push_back({arr, r + hr, r + g.M, col, col + hc, 1});
        }
    }
    trace_push(c, TK_GEMM, ln.st, -1, group, regs);
}

// event handles of a dry run are just numbers; real runs go to CUDA
int ev_record(mplu_context* c, cudaEvent_t ev, cudaStream_t st) {
    if (c->trace) { trace_push(c, TK_RECORD, st, (int)(uintptr_t)ev, -1, {}); return 0; }
    return (int)cudaEventRecord(ev, st);
}
int ev_wait(mplu_context* c, cudaStream_t st, cudaEvent_t ev) {
    if (c->trace) { trace_push(c, TK_WAIT, st, (int)(uintptr_t)ev, -1, {}); return 0; }
    return (int)cudaStreamWaitEvent(st, ev, 0);
}
int traced_cast(mplu_context* c, int r0, int c0, int rows, int cols, cudaStream_t st) {  // Wh block <- W block
    const long long ld = c->npad;
    if (c->trace) {
        if (rows > 0 && cols > 0)
            trace_push(c, TK_CAST, st, -1, -1, {{TA_W, r0, r0 + rows, c0, c0 + cols, 0}, {TA_WH, r0, r0 + rows, c0, c0 + cols, 1}});
        return 0;
    }
    return launch_shadow_cast(c->W + r0 + c0 * ld, ld, c->Wh + r0 + c0 * ld, ld, rows, cols, c->scales + SC_A,
                              c->opts.precision == MPLU_BF16, c->status, st);
}
// the fused GETRF launches of one factorization take their barrier words in order from a zeroed array
int reset_fused_barriers(mplu_context* c, cudaStream_t st) {
    c->fbar_next = 0;
    if (c->fbar) CK(cudaMemsetAsync(c->fbar, 0, (size_t)c->fbar_cap * sizeof(unsigned), st));
    c->fctr_next = 0;
    c->flow_launch_count = 0;
    if (c->fctr) CK(cudaMemsetAsync(c->fctr, 0, (size_t)c->fctr_cap * sizeof(unsigned), st));
    return 0;
}
int traced_clear_bands(mplu_context* c, cudaStream_t st) {
    if (c->trace) {
        trace_push(c, TK_MEMSET, st, -1, -1, {{TA_LINV, 0, c->cap_nb, 0, c->npad, 1}, {TA_UINV, 0, c->cap_nb, 0, c->npad, 1}});
        return 0;
    }
    CK(cudaMemsetAsync(c->Linv16, 0, (size_t)c->cap_nb * c->npad * sizeof(uint16_t), st));
    CK(cudaMemsetAsync(c->Uinv16, 0, (size_t)c->cap_nb * c->npad * sizeof(uint16_t), st));
    return reset_fused_barriers(c, st);
}

// programmatic dependent launch: everywhere (opts.pdl == 1) or on the chain lane only (opts.pdl == 2)
inline int lane_pdl(const mplu_context* c, const Lane& ln) { return c->opts.pdl == 1 || (c->opts.pdl == 2 && ln.pdl); }

GemmParams gemm_params(const mplu_context* c, const GemmCall& g, const Lane& ln) {
    GemmParams p{};
    p.M = g.M; p.N = g.N; p.K = g.K;
    p.a_r0 = g.a_r0; p.a_c0 = g.a_c0; p.b_r0 = g.b_r0; p.b_c0 = g.b_c0;
    p.C = g.C; p.ldc = g.ldc;
    p.Cin = g.accumulate ? g.C : nullptr; p.ldcin = g.ldc;
    if (g.accumulate && g.from_a) {  // the tile's first update: addend = fp32(A) of the same block, cast in the epilogue
        const long long off = g.C - c->W;
        p.Cin = nullptr;
        p.cin64 = c->aref;
        p.cin64_r0 = (int)(off % g.ldc);
        p.cin64_c0 = (int)(off / g.ldc);
    }
    p.H = g.H; p.ldh = g.ldh;
    p.h_rows = g.h_rows; p.h_cols = g.h_cols;
    p.alpha = g.alpha; p.alpha_p1 = g.alpha_p1; p.alpha_p2 = g.alpha_p2;
    p.hscale = 1.f; p.hscale_p = g.hscale_p;
    p.bf16 = c->opts.precision == MPLU_BF16;
    p.status = c->status;
    p.pdl = lane_pdl(c, ln);
    p.tri = c->opts.tri_skip ? g.tri : TRI_NONE;
    p.stream_c = (c->opts.stream_c && g.stream_c) ? 1 : 0;
    return p;
}

int pick_variant(const mplu_context* c, const GemmCall& g) {
    if (c->opts.gemm_variant == MPLU_GEMM_CG1) return GEMM_CG1_AMN;
    if (c->opts.gemm_variant == MPLU_GEMM_CG2) return (g.M > 128) ? GEMM_CG2_AMN : GEMM_CG1_AMN;
    // AUTO: CTA pairs (256x256 tiles) pay off once there is enough work to amortise the cluster set-up; the small
    // products inside a diagonal tile's GETRF run as single-CTA 128x256 tiles
    const long long cg2_min = c->opts.cg2_min_elems > 0 ? c->opts.cg2_min_elems : (1ll << 62);
    return (g.M > 128 && (long long)g.M * g.N >= cg2_min) ? GEMM_CG2_AMN : GEMM_CG1_AMN;
}

int lane_sms(const mplu_context* c, const Lane& ln) {
    int sms = ln.sms > 0 ? ln.sms : c->num_sms;
    if (c->opts.max_sms > 0 && c->opts.max_sms < sms) sms = c->opts.max_sms;
    return sms;
}

// ---- fused GETRF: with c->rec set, the recursion records its products / leaves as steps of a program instead of
// launching them (getrf_fused.cu interprets the program in one persistent launch)
int fused_map_of(const mplu_context* c, const Operand16* o) {
    if (o == &c->opWh) return FM_WH;
    if (o == &c->opFh) return FM_FH;
    if (o == &c->opLinv) return FM_LINV;
    if (o == &c->opUinv) return FM_UINV;
    if (o == &c->opT1) return FM_T1;
    return FM_T2;
}

// one product as the descriptor the persistent GETRF kernels interpret; false: a shape they cannot express
bool to_fused_problem(const mplu_context* c, const GemmCall& g, FusedProblem* out) {
    bool ok = true;
    FusedProblem p{};
    p.M = g.M; p.N = g.N; p.K = g.K;
    p.a_map = fused_map_of(c, g.A); p.a_r0 = g.a_r0; p.a_c0 = g.a_c0;
    p.b_map = fused_map_of(c, g.B); p.b_r0 = g.b_r0; p.b_c0 = g.b_c0;
    p.tri = c->opts.tri_skip ? g.tri : TRI_NONE;
    p.accumulate = g.accumulate ? 1 : 0;
    p.alpha = g.alpha; p.alpha_p1 = g.alpha_p1; p.alpha_p2 = g.alpha_p2; p.hscale_p = g.hscale_p;
    p.c_r0 = p.c_c0 = -1;
    if (g.C) {  // the fp32 result always lives in W
        const long long off = g.C - c->W;
        p.c_r0 = (int)(off % g.ldc); p.c_c0 = (int)(off / g.ldc);
        if (g.ldc != c->npad) ok = false;
    }
    p.h_map = -1;
    if (g.H) {  // the 16-bit copy is a whole-tile store: inside a GETRF every product shadows all of its result
        int arr = 0, hr = 0, hc = 0;
        if (trace_locate16(c, g.H, g.ldh, &arr, &hr, &hc) && (g.h_rows >= g.M || g.h_cols >= g.N)) {
            p.h_map = arr - TA_WH; p.h_r0 = hr; p.h_c0 = hc;
        } else {
            ok = false;
        }
    }
    if (g.accumulate && !g.C) ok = false;
    *out = p;
    return ok;
}

void rec_gemm_step(mplu_context* c, const GemmCall* calls, int count) {
    FusedStep st{};
    st.kind = FS_GEMM;
    st.first_problem = (int)c->rec->problems.size();
    int tiles = 0;
    for (int i = 0; i < count; ++i) {
        const GemmCall& g = calls[i];
        if (g.M <= 0 || g.N <= 0 || g.K <= 0) continue;
        FusedProblem p{};
        if (!to_fused_problem(c, g, &p)) c->rec->unsupported = true;
        c->rec->problems.push_back(p);
        tiles += (g.M / kDiagBlock) * (g.N / kDiagBlock);
        st.tile_end[st.num_problems++] = tiles;
    }
    if (st.num_problems > 0) c->rec->steps.push_back(st);
}

int run_gemm(mplu_context* c, const Lane& ln, const GemmCall& g) {
    if (g.M <= 0 || g.N <= 0 || g.K <= 0) return 0;
    if (c->rec) { rec_gemm_step(c, &g, 1); return 0; }
    if (c->trace) { trace_gemm(c, ln, g, c->trace_group++); c->gemm_launches++; c->kernel_launches++; return 0; }
    const int variant = pick_variant(c, g);
    const bool cg2 = (variant == GEMM_CG2_AMN);
    const GemmParams p = gemm_params(c, g, ln);
    c->gemm_launches++;
    c->kernel_launches++;
    return launch_gemm_tc(variant, &g.A->mapA, cg2 ? &g.B->mapB2 : &g.B->mapB1, p, lane_sms(c, ln), ln.st);
}

// Two independent products in ONE launch (grouped GEMM) when they use the same tile variant, else two launches.
int run_gemm_pair(mplu_context* c, const Lane& ln, const GemmCall& g0, const GemmCall& g1) {
    const bool e0 = g0.M <= 0 || g0.N <= 0 || g0.K <= 0, e1 = g1.M <= 0 || g1.N <= 0 || g1.K <= 0;
    if (e0) return e1 ? 0 : run_gemm(c, ln, g1);
    if (e1) return run_gemm(c, ln, g0);
    if (c->rec && c->opts.group) { const GemmCall both[2] = {g0, g1}; rec_gemm_step(c, both, 2); return 0; }
    if (c->trace && c->opts.group && pick_variant(c, g0) == pick_variant(c, g1)) {  // one launch: the two are concurrent
        const int grp = c->trace_group++;
        trace_gemm(c, ln, g0, grp); trace_gemm(c, ln, g1, grp);
        c->gemm_launches++; c->kernel_launches++;
        return 0;
    }
    const int variant = pick_variant(c, g0);
    if (!c->opts.group || variant != pick_variant(c, g1)) {
        CKI(run_gemm(c, ln, g0));
        return run_gemm(c, ln, g1);
    }
    const bool cg2 = (variant == GEMM_CG2_AMN);
    const GemmParams p0 = gemm_params(c, g0, ln), p1 = gemm_params(c, g1, ln);
    c->gemm_launches++;
    c->kernel_launches++;
    return launch_gemm_tc2(variant, &g0.A->mapA, cg2 ? &g0.B->mapB2 : &g0.B->mapB1, p0, &g1.A->mapA,
                           cg2 ? &g1.B->mapB2 : &g1.B->mapB1, &p1, lane_sms(c, ln), ln.st);
}

// Up to kMaxGroup independent products in ONE launch; falls back to separate launches when their tile variants differ.
int run_gemm_group(mplu_context* c, const Lane& ln, const GemmCall* calls, int count) {
    if (c->rec && c->opts.group) { rec_gemm_step(c, calls, count); return 0; }
    GemmGroup g;
    g.count = 0;
    int variant = -1;
    bool uniform = c->opts.group != 0;
    for (int i = 0; i < count; ++i) {
        if (calls[i].M <= 0 || calls[i].N <= 0 || calls[i].K <= 0) continue;
        const int v = pick_variant(c, calls[i]);
        if (variant < 0) variant = v;
        if (v != variant) uniform = false;
    }
    if (variant < 0) return 0;
    if (!uniform) {
        for (int i = 0; i < count; ++i) CKI(run_gemm(c, ln, calls[i]));
        return 0;
    }
    if (c->trace) {  // one launch: its problems are concurrent
        const int grp = c->trace_group++;
        for (int i = 0; i < count; ++i) trace_gemm(c, ln, calls[i], grp);
        c->gemm_launches++; c->kernel_launches++;
        return 0;
    }
    const bool cg2 = (variant == GEMM_CG2_AMN);
    for (int i = 0; i < count; ++i) {
        if (calls[i].M <= 0 || calls[i].N <= 0 || calls[i].K <= 0) continue;
        g.tmA[g.count] = calls[i].A->mapA;
        g.tmB[g.count] = cg2 ? calls[i].B->mapB2 : calls[i].B->mapB1;
        g.p[g.count] = gemm_params(c, calls[i], ln);
        g.count++;
    }
    c->gemm_launches++;
    c->kernel_launches++;
    return launch_gemm_group(variant, g, lane_sms(c, ln), ln.st);
}

int mark(mplu_context* c, int tag, cudaStream_t st);

// step programs recorded since the last upload -> device (pageable source: staged before the call returns)
int upload_fused_programs(mplu_context* c, cudaStream_t st) {
    const size_t have = c->fprog_host.size();
    if (have > c->fprog_uploaded) {
        CK(cudaMemcpyAsync(c->fprog_dev + c->fprog_uploaded, c->fprog_host.data() + c->fprog_uploaded, have - c->fprog_uploaded,
                           cudaMemcpyHostToDevice, st));
        c->fprog_uploaded = have;
    }
    const size_t fhave = c->flow_host.size();
    if (fhave > c->flow_uploaded) {
        CK(cudaMemcpyAsync(c->flow_dev + c->flow_uploaded, c->flow_host.data() + c->flow_uploaded, fhave - c->flow_uploaded,
                           cudaMemcpyHostToDevice, st));
        c->flow_uploaded = fhave;
    }
    return 0;
}

inline int split_width(int w) { return kDiagBlock * ((w / kDiagBlock + 1) / 2); }

struct Sched {
    mplu_context* c;
    long long ld;   // npad
    long long ldi;  // leading dimension of the inverse bands and merge scratch (cap_nb)
    float* Wp(int r, int col) const { return c->W + r + (long long)col * ld; }
    uint16_t* Whp(int r, int col) const { return c->Wh + r + (long long)col * ld; }
    uint16_t* Fhp(int r, int col) const { return c->Fh + r + (long long)col * ld; }
    const float* sc(int i) const { return c->scales + i; }
    // scales of the diagonal tile starting at column T: {s_Linv, 1/s_Linv, s_Uinv, 1/s_Uinv}
    float* ts(int T) const { return c->inv_scales + 4 * (T / kDiagBlock); }

    // A[r0:r1, c0:c1) -= L[r0:r1, k0:k1) * U[k0:k1, c0:c1): operands from the factor shadow Fh, result in W and,
    // where asked, in the trailing shadow Wh (the reference's cublasDgemm, MPF.cu:230-239)
    GemmCall schur_call(int r0, int r1, int c0, int c1, int k0, int k1, int h_rows, int h_cols, bool first = false) const {
        GemmCall g{&c->opFh, r0, k0, &c->opFh, k0, c0, r1 - r0, c1 - c0, k1 - k0, Wp(r0, c0), ld, true,
                   Whp(r0, c0), ld, h_rows, h_cols, 1.f, sc(SC_NEG_LA_INV), nullptr, sc(SC_A)};
        g.from_a = first && c->lazy;  // update 0 of a block that the lazy first touch left in the caller's fp64 matrix
        // updates much larger than a diagonal tile: their C / shadow traffic is touched once per launch and exceeds L2,
        // so it goes through the streaming cache policy (the tile-sized updates of the chain lane stay cacheable)
        g.stream_c = (long long)(r1 - r0) * (c1 - c0) >= (8ll << 20);
        return g;
    }
    int schur(const Lane& ln, int r0, int r1, int c0, int c1, int k0, int k1, int h_rows, int h_cols, bool first = false) const {
        return run_gemm(c, ln, schur_call(r0, r1, c0, c1, k0, k1, h_rows, h_cols, first));
    }
    // U[k0:k0+w, c0:c1) = inv(L[k0:k0+w)) * A[k0:k0+w, c0:c1)   (inverse of the block inside tile T, one GEMM)
    GemmCall trsm_u_call(int T, int k0, int w, int c0, int c1) const {
        return GemmCall{&c->opLinv, k0 - T, k0, &c->opWh, k0, c0, w, c1 - c0, w, Wp(k0, c0), ld, false,
                        Fhp(k0, c0), ld, w, c1 - c0, 1.f, ts(T) + 1, sc(SC_A_INV), sc(SC_A), TRI_A_LOWER};
    }
    int trsm_u(const Lane& ln, int T, int k0, int w, int c0, int c1) const {
        return run_gemm(c, ln, trsm_u_call(T, k0, w, c0, c1));
    }
    // L[r0:r1, k0:k0+w) = A[r0:r1, k0:k0+w) * inv(U[k0:k0+w))
    GemmCall trsm_l_call(int T, int k0, int w, int r0, int r1) const {
        return GemmCall{&c->opWh, r0, k0, &c->opUinv, k0 - T, k0, r1 - r0, w, w, Wp(r0, k0), ld, false,
                        Fhp(r0, k0), ld, r1 - r0, w, 1.f, sc(SC_A_INV), ts(T) + 3, sc(SC_L), TRI_B_UPPER};
    }
    int trsm_l(const Lane& ln, int T, int k0, int w, int r0, int r1) const {
        return run_gemm(c, ln, trsm_l_call(T, k0, w, r0, r1));
    }
    // both panel solves of one step in a single grouped launch
    int trsm_lu(const Lane& ln, int T, int k0, int w, int lo, int hi) const {
        return run_gemm_pair(c, ln, trsm_l_call(T, k0, w, lo, hi), trsm_u_call(T, k0, w, lo, hi));
    }
    // GETRF of the diagonal block [c0, c0+w)^2 inside tile T, leaving inv(L), inv(U) of the block in the bands.
    // One persistent launch for the whole recursion below this block (getrf_fused.cu).
    bool fuse(int w) const {
        return !c->trace && !c->rec && c->opts.fuse_w > kDiagBlock && w > kDiagBlock && w <= c->opts.fuse_w &&
               w % kDiagBlock == 0 && c->npad % kDiagBlock == 0;
    }
    int getrf_fused(const Lane& ln, int T, int c0, int w) const {
        // programs depend on the geometry, the arrays and the options that shape the products
        const std::vector<long long> key = {c->npad, c->cap_nb, ldi, c->n, c->opts.precision, c->opts.tri_skip, c->opts.group, c->opts.nb,
                                            c->opts.edge_nb, c->opts.fuse_w, c->opts.flow_w, c->opts.schedule,
                                            (long long)reinterpret_cast<uintptr_t>(c->W)};
        if (key != c->fprog_key) {
            c->fprogs.clear(); c->fprog_host.clear(); c->fprog_uploaded = 0;
            c->fprog_key = key;
        }
        const mplu_context::FusedProg* fp = nullptr;
        for (const auto& f : c->fprogs) if (f.T == T && f.c0 == c0 && f.w == w) { fp = &f; break; }
        if (!fp) {
            mplu_context::FusedRecorder r;
            c->rec = &r;
            const int rc = getrf(ln, T, c0, w);
            c->rec = nullptr;
            if (rc) return rc;
            if (r.unsupported) return MPLU_E_ARG;
            const size_t sb = r.steps.size() * sizeof(FusedStep), pb = r.problems.size() * sizeof(FusedProblem);
            const size_t off = c->fprog_host.size();
            if (off + sb + pb > c->fprog_cap) return MPLU_E_ARG;
            c->fprog_host.resize(off + sb + pb);
            memcpy(c->fprog_host.data() + off, r.steps.data(), sb);
            memcpy(c->fprog_host.data() + off + sb, r.problems.data(), pb);
            c->fprogs.push_back({T, c0, w, off, (int)r.steps.size(), (int)r.problems.size()});
            fp = &c->fprogs.back();
        }
        // new programs reach the device before the launch: here when launching directly, after the capture otherwise
        if (!c->capturing) CKI(upload_fused_programs(c, ln.st));
        if (c->fbar_next >= c->fbar_cap) return MPLU_E_ARG;
        FusedArgs a{};
        a.program = c->fprog_dev + fp->offset;
        a.num_steps = fp->num_steps; a.num_problems = fp->num_problems;
        a.barrier = c->fbar + c->fbar_next++;
        a.W = c->W; a.ldw = ld;
        a.Linv16 = c->Linv16; a.Uinv16 = c->Uinv16; a.ld16 = ldi;
        a.Linv32 = c->Linv32; a.Uinv32 = c->Uinv32;
        a.inv_scales = c->inv_scales;
        a.bf16 = c->opts.precision == MPLU_BF16;
        a.status = c->status;
        if (c->fprof_on && c->fprof && fp->num_steps + 3 <= mplu_context::kFusedProfSlots) {
            const int li = (int)(a.barrier - c->fbar);
            a.dbg_clk = c->fprof + (size_t)li * mplu_context::kFusedProfSlots;
            if ((int)c->fprof_prog.size() <= li) c->fprof_prog.resize(li + 1, -1);
            c->fprof_prog[li] = (int)(fp - c->fprogs.data());
        }
        int G = c->opts.fuse_ctas > 0 ? c->opts.fuse_ctas : 8;
        const int budget = lane_sms(c, ln);
        if (G > budget) G = budget;
        G -= G % 2;
        if (G < 2) G = 2;
        c->gemm_launches++;
        c->kernel_launches++;
        return launch_getrf_fused(c->fmaps, a, G, ln.st);
    }
    // ---- dataflow GETRF (getrf_flow.cu): the block as a right-looking task list with explicit dependency counters
    bool flow(int w) const {
        const int b = w / kDiagBlock;
        return !c->trace && !c->rec && c->opts.flow_w > kDiagBlock && w > kDiagBlock && w <= c->opts.flow_w && w % kDiagBlock == 0 &&
               (b & (b - 1)) == 0 && c->npad % kDiagBlock == 0 && b <= 128;
    }
    struct FlowBuild {
        std::vector<FlowLeaf> leaves;
        std::vector<FusedProblem> problems;
        std::vector<FlowTask> tasks;
        int num_main = 0;  // tasks [0, num_main): main list, the rest: inverse merges
        int nctr = 2;      // counters 0 / 1 are the queue heads of the two lists
        bool unsupported = false;
    };
    enum FlowKind : int { FK_PL = 0, FK_PU = 1, FK_S = 2, FK_T1 = 3, FK_T2 = 4, FK_X = 5, FK_Y = 6 };
    // Task list of GETRF([c0, c0+w)^2) inside tile T.  Counters: LD[i] leaf i done (2 = both CTAs); LR[j][i] / UR[i][k] panel
    // tile final; V[j][k] rank-128 updates applied to tile (j,k); per merge node: NL / NU (panel tiles of its off-diagonal
    // block final), MT1 / MT2 (first merge products), MX / MY (merged inverse of the node complete).
    // Two lists, each in priority order and each a topological order (a helper may hold an entry and wait: the earliest
    // unfinished entry of a list can always run; main entries never wait for merges):
    //   main:    A_0 B_0 | A_1 C_0 B_1 | A_2 C_1 B_2 | ...
    //     A_i: L(i+1,i), U(i,i+1), the update of D_{i+1}: all that separates leaf i+1 from leaf i
    //     B_i: the other panel tiles of step i, then the updates of the three tiles step i+1's A-group reads
    //     C_i: the rest of update i, tiles of row / column i+1 first
    //   merges:  M_0 M_1 ...   M_i: merge products whose inputs exist after step i.  The second product of a merge,
    //     X21 = -inv(Lb) T1, waits per tile ROW for that row of inv(Lb) (per column of inv(Ub) on the U side), so after the
    //     last leaf only one row of tiles per level is left instead of four whole levels.
    void build_flow(int T, int c0, int w, FlowBuild& fb) const {
        const int nblk = w / kDiagBlock, end = c0 + w;
        auto newc = [&]() { return fb.nctr++; };
        std::vector<int> LD(nblk), LR(nblk * nblk, -1), UR(nblk * nblk, -1), V(nblk * nblk, -1), NLc(nblk * nblk, -1), NUc(nblk * nblk, -1);
        for (int i = 0; i < nblk; ++i) LD[i] = newc();
        for (int i = 0; i < nblk; ++i)
            for (int j = i + 1; j < nblk; ++j) { LR[j * nblk + i] = newc(); UR[i * nblk + j] = newc(); }
        for (int j = 1; j < nblk; ++j)
            for (int k = 1; k < nblk; ++k) V[j * nblk + k] = newc();
        std::vector<std::vector<FlowTask>> A(nblk), Bp(nblk), Bs(nblk), Cs(nblk), Cm(nblk);
        auto add_problem = [&](const GemmCall& g) {
            FusedProblem p{};
            if (!to_fused_problem(c, g, &p)) fb.unsupported = true;
            fb.problems.push_back(p);
            return (int)fb.problems.size() - 1;
        };
        auto mk = [&](int prob, int mt, int nt, int kind, int step) {
            const FusedProblem& p = fb.problems[prob];
            int k0 = 0, k1 = p.K;
            const int mlo = mt * kDiagBlock, mhi = mlo + kDiagBlock, nlo = nt * kDiagBlock, nhi = nlo + kDiagBlock;
            if (p.tri == TRI_A_LOWER) k1 = std::min(p.K, mhi);
            else if (p.tri == TRI_A_UPPER) k0 = std::min(mlo, p.K - 64);
            else if (p.tri == TRI_B_UPPER) k1 = std::min(p.K, nhi);
            else if (p.tri == TRI_B_LOWER) k0 = std::min(nlo, p.K - 64);
            FlowTask t{};
            t.problem = (uint16_t)prob; t.mt = (uint8_t)mt; t.nt = (uint8_t)nt;
            t.kb0 = (uint8_t)(k0 / 64); t.kb1 = (uint8_t)((k1 + 63) / 64);
            for (int i = 0; i < 4; ++i) { t.wait_ctr[i] = 0xFFFF; t.wait_val[i] = 0; }
            for (int i = 0; i < 3; ++i) t.sig_ctr[i] = 0xFFFF;
            t.pad_[0] = (uint16_t)kind; t.pad_[1] = (uint16_t)step;
            if (prob > 0xFFFE || mt > 255 || nt > 255 || (k1 + 63) / 64 > 255) fb.unsupported = true;
            return t;
        };
        auto wait = [&](FlowTask& t, int ctr, int val) {
            for (int i = 0; i < 4; ++i)
                if (t.wait_ctr[i] == 0xFFFF) { t.wait_ctr[i] = (uint16_t)ctr; t.wait_val[i] = (uint16_t)val; return; }
            fb.unsupported = true;
        };
        auto sig = [&](FlowTask& t, int ctr) {
            if (ctr < 0) return;
            for (int i = 0; i < 3; ++i)
                if (t.sig_ctr[i] == 0xFFFF) { t.sig_ctr[i] = (uint16_t)ctr; return; }
            fb.unsupported = true;
        };
        // ---- merge tree (the recursion of getrf() below, its products as tile tasks)
        typedef std::pair<int, int> Dep;  // counter, target
        // "inv(L) / inv(U) of this block is complete": as a whole, per block row of inv(L), per block column of inv(U)
        struct Merged { Dep lx, ux; std::vector<Dep> lrow, ucol; };
        struct Prev { bool have = false; Dep lx, ux; };
        std::vector<Prev> prev(nblk + 1);  // last node of each width (in 128-blocks): its scratch slice is reused
        std::function<Merged(int, int)> merge = [&](int n0, int nw) -> Merged {
            if (nw <= kDiagBlock) {
                const Dep d{LD[(n0 - c0) / kDiagBlock], 2};
                return Merged{d, d, {d}, {d}};
            }
            const int h = split_width(nw), g = nw - h, n1 = n0 + h;
            const Merged left = merge(n0, h), right = merge(n1, g);
            const int ia0 = (n0 - c0) / kDiagBlock, ia1 = (n1 - c0) / kDiagBlock, ib1 = (n0 + nw - c0) / kDiagBlock;  // a = [ia0, ia1), b = [ia1, ib1)
            const int NL = newc(), NU = newc(), MT1 = newc(), MT2 = newc(), MX = newc(), MY = newc();
            for (int j = ia1; j < ib1; ++j)
                for (int i = ia0; i < ia1; ++i) { NLc[j * nblk + i] = NL; NUc[i * nblk + j] = NU; }
            const int gt = g / kDiagBlock, ht = h / kDiagBlock, tiles = gt * ht;
            const long long off = ldi - nw;
            const int p1 = add_problem(GemmCall{&c->opFh, n1, n0, &c->opLinv, n0 - T, n0, g, h, h, nullptr, 0, false,
                                                c->Tb1 + off * ldi, ldi, g, h, 1.f, sc(SC_L_INV), ts(T) + 1, sc(SC_L), TRI_B_LOWER});
            const int p2 = add_problem(GemmCall{&c->opUinv, n0 - T, n0, &c->opFh, n0, n1, h, g, h, nullptr, 0, false,
                                                c->Tb2 + off * ldi, ldi, h, g, 1.f, ts(T) + 3, sc(SC_A_INV), sc(SC_L), TRI_A_UPPER});
            const int px = add_problem(GemmCall{&c->opLinv, n1 - T, n1, &c->opT1, 0, (int)off, g, h, g, nullptr, 0, false,
                                                c->Linv16 + (n1 - T) + (long long)n0 * ldi, ldi, g, h, -1.f, ts(T) + 1, sc(SC_L_INV), ts(T) + 0, TRI_A_LOWER});
            const int py = add_problem(GemmCall{&c->opT2, 0, (int)off, &c->opUinv, n1 - T, n1, h, g, g, nullptr, 0, false,
                                                c->Uinv16 + (n0 - T) + (long long)n1 * ldi, ldi, h, g, -1.f, sc(SC_L_INV), ts(T) + 3, ts(T) + 2, TRI_B_UPPER});
            const Prev pv = prev[nw / kDiagBlock];
            for (int nt = 0; nt < ht; ++nt)
                for (int mt = 0; mt < gt; ++mt) {
                    FlowTask t = mk(p1, mt, nt, FK_T1, ia1 - 1);
                    wait(t, NL, tiles); wait(t, left.lx.first, left.lx.second);
                    if (pv.have) wait(t, pv.lx.first, pv.lx.second);  // the previous node of this width has read the scratch slice
                    sig(t, MT1);
                    Cm[ia1 - 1].push_back(t);
                    FlowTask u = mk(p2, nt, mt, FK_T2, ia1 - 1);
                    wait(u, NU, tiles); wait(u, left.ux.first, left.ux.second);
                    if (pv.have) wait(u, pv.ux.first, pv.ux.second);
                    sig(u, MT2);
                    Cm[ia1 - 1].push_back(u);
                }
            Merged me{Dep{MX, tiles}, Dep{MY, tiles}, left.lrow, left.ucol};
            // rows (columns) of the b part become final one by one, in the order their leaves end
            for (int r = 0; r < gt; ++r) {
                const int XR = newc(), YC = newc();
                for (int q = 0; q < ht; ++q) {
                    FlowTask t = mk(px, r, q, FK_X, ia1 + r);
                    wait(t, MT1, tiles); wait(t, right.lrow[r].first, right.lrow[r].second);
                    sig(t, XR); sig(t, MX);
                    Cm[ia1 + r].push_back(t);
                    FlowTask u = mk(py, q, r, FK_Y, ia1 + r);
                    wait(u, MT2, tiles); wait(u, right.ucol[r].first, right.ucol[r].second);
                    sig(u, YC); sig(u, MY);
                    Cm[ia1 + r].push_back(u);
                }
                me.lrow.push_back(Dep{XR, ht});
                me.ucol.push_back(Dep{YC, ht});
            }
            prev[nw / kDiagBlock].have = true;
            prev[nw / kDiagBlock].lx = me.lx;
            prev[nw / kDiagBlock].ux = me.ux;
            return me;
        };
        merge(c0, w);
        // ---- leaves, panel solves, rank-128 updates
        for (int i = 0; i < nblk; ++i) {
            const int b = c0 + i * kDiagBlock, b1 = b + kDiagBlock;
            FlowLeaf lf{};
            lf.k0 = b; lf.blk = b / kDiagBlock; lf.first_in_tile = b == T; lf.T = T;
            lf.valid = c->n - b < kDiagBlock ? c->n - b : kDiagBlock;
            lf.wait_ctr = i > 0 ? (uint16_t)V[i * nblk + i] : 0xFFFF;
            lf.wait_val = (uint16_t)i;
            lf.sig_ctr = (uint16_t)LD[i];
            fb.leaves.push_back(lf);
            if (b1 >= end) break;
            const int pl = add_problem(trsm_l_call(T, b, kDiagBlock, b1, end));
            const int pu = add_problem(trsm_u_call(T, b, kDiagBlock, b1, end));
            const int ps = add_problem(schur_call(b1, end, b1, end, b, b1, end - b1, end - b1));
            for (int j = i + 1; j < nblk; ++j) {
                FlowTask tl = mk(pl, j - i - 1, 0, FK_PL, i);
                wait(tl, LD[i], 2);
                if (i > 0) wait(tl, V[j * nblk + i], i);
                sig(tl, LR[j * nblk + i]); sig(tl, NLc[j * nblk + i]);
                FlowTask tu = mk(pu, 0, j - i - 1, FK_PU, i);
                wait(tu, LD[i], 2);
                if (i > 0) wait(tu, V[i * nblk + j], i);
                sig(tu, UR[i * nblk + j]); sig(tu, NUc[i * nblk + j]);
                auto& grp = j == i + 1 ? A[i] : Bp[i];
                grp.push_back(tl); grp.push_back(tu);
            }
            std::vector<std::pair<int, FlowTask>> rest;
            for (int j = i + 1; j < nblk; ++j)
                for (int k = i + 1; k < nblk; ++k) {
                    FlowTask t = mk(ps, j - i - 1, k - i - 1, FK_S, i);
                    wait(t, LR[j * nblk + i], 1); wait(t, UR[i * nblk + k], 1);
                    if (i > 0) wait(t, V[j * nblk + k], i);
                    sig(t, V[j * nblk + k]);
                    if (j == i + 1 && k == i + 1) A[i].push_back(t);
                    else if (j <= i + 2 && k <= i + 2) Bs[i].push_back(t);
                    else rest.push_back({std::min(j, k) * nblk + std::max(j, k), t});
                }
            std::stable_sort(rest.begin(), rest.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
            for (auto& r : rest) Cs[i].push_back(r.second);
        }
        auto put = [&](const std::vector<FlowTask>& v) { fb.tasks.insert(fb.tasks.end(), v.begin(), v.end()); };
        put(A[0]); put(Bp[0]); put(Bs[0]);
        for (int i = 0; i < nblk; ++i) {
            if (i + 1 < nblk) put(A[i + 1]);
            put(Cs[i]);
            if (i + 1 < nblk) { put(Bp[i + 1]); put(Bs[i + 1]); }
        }
        fb.num_main = (int)fb.tasks.size();
        for (int i = 0; i < nblk; ++i) put(Cm[i]);
        if (fb.nctr > 0xFFFE) fb.unsupported = true;
    }
    int getrf_flow(const Lane& ln, int T, int c0, int w) const {
        // programs depend on the geometry (incl. the tiling: a context that switches options must not pile programs of
        // different tilings into a buffer sized for one), the arrays and the options that shape the products
        const std::vector<long long> key = {c->npad, c->cap_nb, ldi, c->n, c->opts.precision, c->opts.tri_skip, c->opts.nb, c->opts.edge_nb,
                                            c->opts.flow_w, c->opts.schedule, (long long)reinterpret_cast<uintptr_t>(c->W)};
        if (key != c->flow_key) {
            c->flow_progs.clear(); c->flow_host.clear(); c->flow_uploaded = 0;
            c->flow_key = key;
        }
        int pi = -1;
        for (size_t i = 0; i < c->flow_progs.size(); ++i)
            if (c->flow_progs[i].T == T && c->flow_progs[i].c0 == c0 && c->flow_progs[i].w == w) { pi = (int)i; break; }
        if (pi < 0) {
            FlowBuild fb;
            build_flow(T, c0, w, fb);
            if (fb.unsupported) return MPLU_E_ARG;
            const size_t lb = fb.leaves.size() * sizeof(FlowLeaf), pb = fb.problems.size() * sizeof(FusedProblem),
                         tb = fb.tasks.size() * sizeof(FlowTask);
            const size_t off = c->flow_host.size();
            if (off + lb + pb + tb > c->flow_cap) return MPLU_E_ARG;
            c->flow_host.resize(off + lb + pb + tb);
            memcpy(c->flow_host.data() + off, fb.leaves.data(), lb);
            memcpy(c->flow_host.data() + off + lb, fb.problems.data(), pb);
            memcpy(c->flow_host.data() + off + lb + pb, fb.tasks.data(), tb);
            c->flow_progs.push_back({T, c0, w, off, off + lb, off + lb + pb, (int)fb.leaves.size(), (int)fb.problems.size(),
                                     (int)fb.tasks.size(), fb.num_main, fb.nctr});
            pi = (int)c->flow_progs.size() - 1;
        }
        const mplu_context::FlowProg& fp = c->flow_progs[pi];
        if (!c->capturing) CKI(upload_fused_programs(c, ln.st));
        if (c->fctr_next + fp.num_counters > c->fctr_cap) return MPLU_E_ARG;
        FlowArgs a{};
        a.leaves = reinterpret_cast<const FlowLeaf*>(c->flow_dev + fp.off_leaves); a.num_leaves = fp.num_leaves;
        a.problems = reinterpret_cast<const FusedProblem*>(c->flow_dev + fp.off_problems); a.num_problems = fp.num_problems;
        a.tasks = reinterpret_cast<const FlowTask*>(c->flow_dev + fp.off_tasks); a.num_tasks = fp.num_tasks;
        a.num_main = fp.num_main;
        a.counters = c->fctr + c->fctr_next;
        c->fctr_next += fp.num_counters;
        a.W = c->W; a.ldw = ld;
        a.Linv16 = c->Linv16; a.Uinv16 = c->Uinv16; a.ld16 = ldi;
        a.Linv32 = c->Linv32; a.Uinv32 = c->Uinv32;
        a.inv_scales = c->inv_scales;
        a.bf16 = c->opts.precision == MPLU_BF16;
        a.status = c->status;
        if (c->flow_prof && c->flow_launch_count == c->flow_prof_launch &&
            (size_t)(2 * fp.num_leaves + 4 * fp.num_tasks) * sizeof(long long) <= c->flow_prof_cap) {
            a.dbg = c->flow_prof;
            c->flow_prof_prog = pi;
        }
        c->flow_launch_count++;
        int G = c->opts.flow_ctas > 0 ? c->opts.flow_ctas : 16;
        const int budget = lane_sms(c, ln);
        if (G > budget) G = budget;
        G -= G % 2;
        if (G < 4) G = 4;
        // helpers that serve the inverse merges first: about a quarter of them (measured, tools/flow_profile.py)
        a.merge_ctas = c->opts.flow_merge_ctas >= 0 ? c->opts.flow_merge_ctas : (G - 2) / 4;
        if (a.merge_ctas > G - 3) a.merge_ctas = G - 3;
        c->gemm_launches++;
        c->kernel_launches++;
        return launch_getrf_flow(c->fmaps, a, G, ln.st);
    }
    int getrf(const Lane& ln, int T, int c0, int w) const {
        if (flow(w)) {
            // MPLU_E_ARG = "does not fit the task-list / counter buffers" (returned before anything is launched): the
            // block is then factored by the step program or the recursion below instead of failing the solve
            const int rc = getrf_flow(ln, T, c0, w);
            if (rc != MPLU_E_ARG) return rc;
        }
        if (fuse(w)) return getrf_fused(ln, T, c0, w);
        if (w <= kDiagBlock) {
            const int blk = c0 / kDiagBlock;
            if (c->rec) {
                FusedStep st{};
                st.kind = FS_LEAF;
                st.k0 = c0; st.blk = blk; st.first_in_tile = c0 == T; st.T = T;
                st.valid = c->n - c0 < kDiagBlock ? c->n - c0 : kDiagBlock;
                c->rec->steps.push_back(st);
                return 0;
            }
            uint16_t* l16 = c->Linv16 + (c0 - T) + (long long)c0 * ldi;
            uint16_t* u16 = c->Uinv16 + (c0 - T) + (long long)c0 * ldi;
            if (c->trace) {  // reads and rewrites its W block, writes its triangles of the two inverse bands
                trace_push(c, TK_LEAF, ln.st, -1, -1,
                           {{TA_W, c0, c0 + kDiagBlock, c0, c0 + kDiagBlock, 0}, {TA_W, c0, c0 + kDiagBlock, c0, c0 + kDiagBlock, 1},
                            {TA_LINV, c0 - T, c0 - T + kDiagBlock, c0, c0 + kDiagBlock, 1},
                            {TA_UINV, c0 - T, c0 - T + kDiagBlock, c0, c0 + kDiagBlock, 1}});
                c->kernel_launches++;
                return 0;
            }
            CKI(mark(c, 8000 + blk, ln.st));  // development aid (mplu_debug_marks_enable): leaf start / end
            CKI(launch_diag_lu(c->W, ld, c0, l16, u16, ldi, c->Linv32, c->Uinv32, ts(T), c0 == T, blk,
                               c->opts.precision == MPLU_BF16, c->status, ln.st, nullptr, lane_pdl(c, ln),
                               c->n - c0 < kDiagBlock ? c->n - c0 : kDiagBlock));
            c->kernel_launches++;
            return mark(c, 9000 + blk, ln.st);
        }
        const int h = split_width(w), g = w - h, c1 = c0 + h;
        CKI(getrf(ln, T, c0, h));
        CKI(trsm_lu(ln, T, c0, h, c1, c0 + w));
        // The Schur update and the first products of the inverse merge,
        //     inv(L)21 = -inv(Lb) * (L21 * inv(La)),   inv(U)12 = -(inv(Ua) * U12) * inv(Ub),
        // only need the panel solves' results: one grouped launch.  The parked products live in a per-width slice of
        // the scratch (columns [cap - w, cap - w + w/2)): the right child's own merges use slices further right.
        const long long off = ldi - w;
        GemmCall first[3] = {
            schur_call(c1, c0 + w, c1, c0 + w, c0, c1, g, g),
            GemmCall{&c->opFh, c1, c0, &c->opLinv, c0 - T, c0, g, h, h, nullptr, 0, false,
                     c->Tb1 + off * ldi, ldi, g, h, 1.f, sc(SC_L_INV), ts(T) + 1, sc(SC_L), TRI_B_LOWER},
            GemmCall{&c->opUinv, c0 - T, c0, &c->opFh, c0, c1, h, g, h, nullptr, 0, false,
                     c->Tb2 + off * ldi, ldi, h, g, 1.f, ts(T) + 3, sc(SC_A_INV), sc(SC_L), TRI_A_UPPER}};
        CKI(run_gemm_group(c, ln, first, 3));
        CKI(getrf(ln, T, c1, g));
        GemmCall x{&c->opLinv, c1 - T, c1, &c->opT1, 0, (int)off, g, h, g, nullptr, 0, false,
                   c->Linv16 + (c1 - T) + (long long)c0 * ldi, ldi, g, h, -1.f, ts(T) + 1, sc(SC_L_INV), ts(T) + 0, TRI_A_LOWER};
        GemmCall y{&c->opT2, 0, (int)off, &c->opUinv, c1 - T, c1, h, g, g, nullptr, 0, false,
                   c->Uinv16 + (c0 - T) + (long long)c1 * ldi, ldi, h, g, -1.f, sc(SC_L_INV), ts(T) + 3, ts(T) + 2, TRI_B_UPPER};
        return run_gemm_pair(c, ln, x, y);
    }
};

int getrf_resident_tile(mplu_context* c, cudaStream_t st, int w) {
    const long long ld = c->npad;  // the workspace's leading dimension (its allocation), w <= npad is the tile width
    const int bf16 = c->opts.precision == MPLU_BF16;
    const Lane ln{st, c->opts.max_sms};
    CKI(launch_shadow_cast(c->W, ld, c->Wh, ld, w, w, c->scales + SC_A, bf16, c->status, st));
    CK(cudaMemsetAsync(c->Linv16, 0, (size_t)c->cap_nb * w * sizeof(uint16_t), st));
    CK(cudaMemsetAsync(c->Uinv16, 0, (size_t)c->cap_nb * w * sizeof(uint16_t), st));
    CKI(reset_fused_barriers(c, st));
    const Sched S{c, ld, (long long)c->cap_nb};
    return S.getrf(ln, 0, 0, w);
}

// GETRF of the diagonal tile [T, T+w)^2 of context c in the compact workspace context c->tile (its arrays are one slab
// that the chain lane keeps resident in L2 with an access-policy window while the bulk lane streams the trailing matrix
// through the cache): copy the tile in, factor it there, copy L\U, the 16-bit inverses (into the bands), the fp32 block
// inverses and the tile's scales back.
int getrf_in_workspace(mplu_context* c, const Lane& ln, int T, int w) {
    mplu_context* t = c->tile;
    const long long ld = c->npad, tld = t->npad;
    cudaStream_t st = ln.st;
    const size_t wb = (size_t)w;
    t->opts.max_sms = lane_sms(c, ln);
    t->opts.precision = c->opts.precision;
    int* own_status = t->status;
    t->status = c->status;  // the tile's kernels report into the caller's status word
    t->capturing = c->capturing;  // fused step programs recorded during a capture are uploaded after it (factor_impl)
    CK(cudaMemcpy2DAsync(t->W, (size_t)tld * sizeof(float), c->W + T + (long long)T * ld, (size_t)ld * sizeof(float),
                         wb * sizeof(float), wb, cudaMemcpyDeviceToDevice, st));
    t->gemm_launches = t->kernel_launches = 0;
    int rc = getrf_resident_tile(t, st, w);
    t->status = own_status;
    if (rc) return rc;
    c->gemm_launches += t->gemm_launches;
    c->kernel_launches += t->kernel_launches + 1;
    CK(cudaMemcpy2DAsync(c->W + T + (long long)T * ld, (size_t)ld * sizeof(float), t->W, (size_t)tld * sizeof(float),
                         wb * sizeof(float), wb, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpy2DAsync(c->Linv16 + (long long)T * c->cap_nb, (size_t)c->cap_nb * 2, t->Linv16, (size_t)t->cap_nb * 2, wb * 2, wb,
                         cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpy2DAsync(c->Uinv16 + (long long)T * c->cap_nb, (size_t)c->cap_nb * 2, t->Uinv16, (size_t)t->cap_nb * 2, wb * 2, wb,
                         cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(c->Linv32 + (size_t)T * kDiagBlock, t->Linv32, wb * kDiagBlock * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(c->Uinv32 + (size_t)T * kDiagBlock, t->Uinv32, wb * kDiagBlock * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(c->inv_scales + 4 * (T / kDiagBlock), t->inv_scales, 4 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

// Create / size the tile workspace and pin it in L2 for the stream the diagonal tiles are factored on.
int prepare_tile_workspace(mplu_context* c, int NB, cudaStream_t getrf_stream) {
    if (!c->tile) CKI(mplu_create(&c->tile, c->device));
    mplu_context* t = c->tile;
    t->opts = c->opts;
    t->opts.nb = NB;
    t->opts.lookahead = 0;
    t->opts.use_graph = 0;
    CKI(ensure_work(t, NB));
    if (c->opts.l2_persist) {
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, c->device));
        size_t want = t->slab_bytes;
        if (prop.persistingL2CacheMaxSize > 0 && prop.accessPolicyMaxWindowSize > 0) {
            const size_t carve = want < (size_t)prop.persistingL2CacheMaxSize ? want : (size_t)prop.persistingL2CacheMaxSize;
            CK(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve));
            cudaStreamAttrValue attr{};
            attr.accessPolicyWindow.base_ptr = t->slab;
            attr.accessPolicyWindow.num_bytes = want < (size_t)prop.accessPolicyMaxWindowSize ? want : (size_t)prop.accessPolicyMaxWindowSize;
            attr.accessPolicyWindow.hitRatio = (float)((double)carve / (double)attr.accessPolicyWindow.num_bytes);
            if (attr.accessPolicyWindow.hitRatio > 1.f) attr.accessPolicyWindow.hitRatio = 1.f;
            attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            CK(cudaStreamSetAttribute(getrf_stream, cudaStreamAttributeAccessPolicyWindow, &attr));
        }
    }
    return 0;
}

int record_event(mplu_context* c, cudaEvent_t ev, cudaStream_t st) {
    if (c->trace) return 0;
    return (int)cudaEventRecordWithFlags(ev, st, c->capturing ? cudaEventRecordExternal : cudaEventRecordDefault);
}

// timeline mark: tag = 1000*kind + step; kinds: 1 chain: next-tile TRSM start, 2 chain: GETRF start, 3 chain: GETRF end,
// 4 bulk: TRSM start, 5 bulk: block column/row update start, 6 bulk: rest start, 7 bulk: rest end
int mark(mplu_context* c, int tag, cudaStream_t st) {
    if (c->trace) return 0;
    if (!c->marks_on || c->mark_count >= mplu_context::kMaxMarks) return 0;
    cudaEvent_t& e = c->mark_ev[c->mark_count];
    if (!e) CK(cudaEventCreate(&e));
    c->mark_tag[c->mark_count++] = tag;
    return record_event(c, e, st);
}

int step_event(mplu_context* c, int step, int kind, cudaEvent_t* out) {
    if (step >= mplu_context::kMaxSteps) return MPLU_E_ARG;
    if (c->trace) { *out = (cudaEvent_t)(uintptr_t)(1000 + 4 * step + kind); return 0; }
    cudaEvent_t& e = c->ev_step[4 * step + kind];
    if (!e) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    *out = e;
    return 0;
}

// Everything after the first touch: scales, shadows of the first block column / block row, the tile loop.
int enqueue_factorization(mplu_context* c) {
    const int npad = c->npad;
    const long long ld = npad;
    const int bf16 = c->opts.precision == MPLU_BF16;
    const int NB = effective_nb(c, npad);
    if ((npad + NB - 1) / NB >= mplu_context::kMaxSteps) return MPLU_E_ARG;
    cudaStream_t st = c->stream;
    int side_sms = c->opts.side_sms > 0 ? c->opts.side_sms : 40;
    side_sms -= side_sms % 2;
    const bool two = c->opts.lookahead != 0 && side_sms >= 2 && side_sms <= c->num_sms - 16 && npad > 2 * NB;
    const Lane all{st, 0};
    Lane bulk = two ? Lane{st, c->num_sms - side_sms} : all;
    Lane chain = two ? Lane{c->side, side_sms, true} : all;
    // While the trailing matrix is large the schedule is bound by the bulk lane (the chain lane waits for it), so the
    // chain gets fewer SMs there: side_sms_early while more than early_frac of the columns remain.
    int side_early = c->opts.side_sms_early > 0 ? c->opts.side_sms_early : side_sms;
    side_early -= side_early % 2;
    if (side_early < 2 || side_early > side_sms) side_early = side_sms;
    const Sched S{c, ld, (long long)c->cap_nb};
    enum { EV_GETRF = 0, EV_NEXT = 1, EV_B2 = 2, EV_B3A = 3 };
    cudaEvent_t ev = nullptr;

    if (!c->trace) CKI(launch_scales(c->amax, c->scales, c->opts.a_exp, c->opts.l_exp, bf16, st));
    CKI(traced_cast(c, 0, 0, npad, NB, st));
    if (npad > NB)
        CKI(traced_cast(c, 0, NB, NB, npad - NB, st));
    c->kernel_launches += 3;
    // the inverse bands are only ever written inside the diagonal tiles' triangles: everything else must read 0
    CKI(traced_clear_bands(c, st));

    const bool ws = c->opts.tile_ws != 0 && npad > NB;
    if (ws) CK(cudaMemcpyAsync(c->tile->scales, c->scales, SC_COUNT * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (ws) CKI(getrf_in_workspace(c, all, 0, NB)); else CKI(S.getrf(all, 0, 0, NB));
    if (two) {
        CKI(ev_record(c, c->ev_fork, st));
        CKI(ev_wait(c, c->side, c->ev_fork));
    }
    int step = 0;
    for (int k0 = 0; k0 + NB < npad; k0 += NB, ++step) {
        const int k1 = k0 + NB;
        const int k2 = (k1 + NB < npad) ? k1 + NB : npad;
        const int nbn = k2 - k1;
        if (two) {
            const long long rem100 = (npad - k2) * 100ll;
            const int sd = rem100 > (long long)npad * c->opts.early_pct ? side_early : side_sms;
            bulk.sms = c->num_sms - sd;
            chain.sms = sd;
            if (rem100 <= (long long)npad * c->opts.late_pct) {
                // the trailing matrix is small: the bulk lane idles most of the step, both lanes may use every SM
                bulk.sms = 0;
                chain.sms = 0;
            }
        }
        // ---- chain lane: panel solves restricted to the next tile, its Schur update, its GETRF
        if (two && step > 0) {  // tile rows/columns k1.. of block column/row k were updated by the bulk lane
            CKI(step_event(c, step - 1, EV_B2, &ev));
            CKI(ev_wait(c, chain.st, ev));
        }
        CKI(mark(c, 1000 + step, chain.st));
        CKI(S.trsm_lu(chain, k0, k0, NB, k1, k2));
        if (two) { CKI(step_event(c, step, EV_NEXT, &ev)); CKI(ev_record(c, ev, chain.st)); }
        if (two && step > 0) {  // the next diagonal tile has received update step-1 (first piece of the bulk's rest)
            CKI(step_event(c, step - 1, EV_B3A, &ev));
            CKI(ev_wait(c, chain.st, ev));
        }
        CKI(S.schur(chain, k1, k2, k1, k2, k0, k1, nbn, nbn));
        CKI(mark(c, 2000 + step, chain.st));
        if (ws) CKI(getrf_in_workspace(c, chain, k1, nbn)); else CKI(S.getrf(chain, k1, k1, nbn));
        CKI(mark(c, 3000 + step, chain.st));
        if (two) { CKI(step_event(c, step + 1, EV_GETRF, &ev)); CKI(ev_record(c, ev, chain.st)); }
        // ---- bulk lane: the other rows/columns of the panels, then the trailing update
        if (k2 >= npad) continue;
        if (two && step > 0) {  // GETRF of tile k (its inverses) came from the chain lane
            CKI(step_event(c, step, EV_GETRF, &ev));
            CKI(ev_wait(c, bulk.st, ev));
        }
        CKI(mark(c, 4000 + step, bulk.st));
        CKI(S.trsm_lu(bulk, k0, k0, NB, k2, npad));
        if (two) { CKI(step_event(c, step, EV_NEXT, &ev)); CKI(ev_wait(c, bulk.st, ev)); }
        CKI(mark(c, 5000 + step, bulk.st));
        // next block column and next block row (full shadows), one grouped launch
        CKI(run_gemm_pair(c, bulk, S.schur_call(k2, npad, k1, k2, k0, k1, npad - k2, nbn),
                          S.schur_call(k1, k2, k2, npad, k0, k1, nbn, npad - k2)));
        if (two) { CKI(step_event(c, step, EV_B2, &ev)); CKI(ev_record(c, ev, bulk.st)); }
        // the rest of the trailing matrix (no shadow), block column k2.. first: the chain lane's next Schur update
        // only needs the diagonal tile inside it
        const int k3 = (k2 + NB < npad) ? k2 + NB : npad;
        CKI(S.schur(bulk, k2, npad, k2, k3, k0, k1, 0, 0));
        if (two) { CKI(step_event(c, step, EV_B3A, &ev)); CKI(ev_record(c, ev, bulk.st)); }
        if (k3 >= npad) continue;
        const int Mt = npad - k2, Nt = npad - k3;
        const bool timed = !c->trace && c->trail_count < mplu_context::kMaxTrail;
        if (timed) {
            cudaEvent_t& e0 = c->trail_ev[2 * c->trail_count];
            if (!e0) { CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&c->trail_ev[2 * c->trail_count + 1])); }
            CKI(record_event(c, e0, bulk.st));
        }
        CKI(mark(c, 6000 + step, bulk.st));
        CKI(S.schur(bulk, k2, npad, k3, npad, k0, k1, 0, 0));
        CKI(mark(c, 7000 + step, bulk.st));
        if (timed) {
            CKI(record_event(c, c->trail_ev[2 * c->trail_count + 1], bulk.st));
            c->trail_count++;
            c->trail_flops += 2.0 * Mt * (double)Nt * NB;
            c->trail_bytes += 8.0 * Mt * (double)Nt;
        }
    }
    if (two) {
        CKI(ev_record(c, c->ev_join, c->side));
        CKI(ev_wait(c, st, c->ev_join));
    }
    return 0;
}

// Bulk-lane plan of the left-looking schedule (pure host logic; mplu_debug_plan_left exposes it to the CPU tests).
// Block column m (m >= 2) must receive the updates k = 0 .. m-2 in increasing k before step m, and update k can only be
// applied from step k+1 on (its L panel is complete then).  Step j first brings block column j+1 up to date
// (mandatory), then spends the rest of its share of the remaining update flops on the columns further right, nearest
// first, one op per run of equally advanced columns.  An op applies update k to block columns [m0, m1).
struct LeftOp { int step, k, m0, m1, mandatory, kn = 1; };  // kn: consecutive updates k .. k+kn-1 applied in one pass

// Block-column boundaries of the left-looking schedule: nb-wide, except that with opts.edge_nb the first and the last one are
// narrower.  While the first diagonal tile is factored nothing else can run, and the last one has nothing left to overlap
// with: 2 x 1.25 ms of the n = 32768 factorization with ~130 SMs idle; a 1024-wide tile there takes half as long.
std::vector<int> tile_bounds(int npad, int NB, int edge) {
    std::vector<int> tb{0};
    edge = (edge / kDiagBlock) * kDiagBlock;
    if (edge > 0 && edge < NB && npad >= 4 * NB) {
        int pos = edge;
        tb.push_back(pos);
        while (npad - pos > NB + edge) { pos += NB; tb.push_back(pos); }
        if (npad - pos > edge) tb.push_back(npad - edge);  // what is left: (rest - edge) <= NB, then the narrow last tile
    } else {
        for (int pos = NB; pos < npad; pos += NB) tb.push_back(pos);
    }
    tb.push_back(npad);
    return tb;
}

// pair: an op may apply TWO consecutive updates (k, k+1) in one pass over the block columns (K = both panels' widths: the
// tall update is bound by L2 traffic and its fp32 C read + write is a fifth of that at K = 2048, a tenth at 4096)
std::vector<LeftOp> plan_left(const std::vector<int>& tb, bool eager, bool pair = false) {
    const int nt = (int)tb.size() - 1, npad = tb[nt];
    std::vector<LeftOp> ops;
    std::vector<int> done(nt > 0 ? nt : 1, 0);  // done[m]: block column m has received the updates k < done[m]
    auto colb = [&](int m) { return tb[m < nt ? m : nt]; };
    auto cost = [&](int k, int m0, int m1) {  // flops of update k on block columns [m0, m1): panel solve + Schur update
        const double N = colb(m1) - colb(m0), wk = tb[k + 1] - tb[k];
        return 2.0 * (npad - tb[k + 1]) * N * wk + wk * wk * N;
    };
    double remaining = 0.0;
    for (int m = 2; m < nt; ++m)
        for (int k = 0; k + 2 <= m; ++k) remaining += cost(k, m, m + 1);
    for (int j = 1; j + 1 < nt; ++j) {
        double spent = 0.0;
        for (int k = done[j + 1]; k < j; ++k) {
            const int kn = (pair && k + 1 < j) ? 2 : 1;
            ops.push_back({j, k, j + 1, j + 2, 1, kn});
            spent += cost(k, j + 1, j + 2);
            if (kn == 2) { ++k; spent += cost(k, j + 1, j + 2); }
        }
        done[j + 1] = j;
        const double share = eager ? remaining / (double)(nt - 1 - j) : 0.0;
        while (spent < share) {
            int m = j + 2;
            while (m < nt && done[m] >= j) ++m;
            if (m >= nt) break;
            const int d = done[m];
            int m1 = m + 1;
            while (m1 < nt && done[m1] == d) ++m1;
            const int kn = (pair && d + 1 < j) ? 2 : 1;  // update d+1 is available too (its L panel is complete)
            const double c1 = cost(d, m, m + 1) + (kn == 2 ? cost(d + 1, m, m + 1) : 0.0);
            const int fit = (int)((share - spent) / c1 + 0.5);
            if (m1 - m > fit) m1 = m + (fit > 1 ? fit : 1);
            ops.push_back({j, d, m, m1, 0, kn});
            spent += cost(d, m, m1) + (kn == 2 ? cost(d + 1, m, m1) : 0.0);
            for (int i = m; i < m1; ++i) done[i] = d + kn;
        }
        remaining -= spent;
    }
    return ops;
}

// opts.schedule == MPLU_SCHED_LEFT: left-looking by nb-wide block columns with look-ahead.
// The right-looking schedule above front-loads the tensor-core work (step k updates the whole trailing matrix), so its
// first steps are bound by the bulk lane and its last ~10 by the latency-bound GETRF chain with the bulk lane idle.
// Left-looking, block column j receives all of its updates k < j just before its turn; the amount of update work per
// step GROWS with j instead of shrinking, and every step has less of it than one GETRF takes: the chain lane never
// waits for more than the two-tile update it does itself, and the bulk lane's rank-nb updates (tall (n - k nb) x nb
// products, the best-shaped GEMMs of the factorization) hide behind the chain.  Per tile the same products are
// formed in the same order: the factors are bit-identical to the right-looking schedule's.
//   chain, step j:  U(j-1,j) = inv(L(j-1,j-1)) A(j-1,j);  tile (j,j) -= L(j,j-1) U(j-1,j);  GETRF(D_j);
//                   L(j+1,j) = A(j+1,j) inv(U(j,j))
//   bulk,  step j:  rows below tile j of column j -= L(.,j-1) U(j-1,j);   column j+1: updates k = 0..j-1;
//                   L(j+2:,j) = A(j+2:,j) inv(U(j,j))
int enqueue_factorization_left(mplu_context* c) {
    const int npad = c->npad;
    const long long ld = npad;
    const int bf16 = c->opts.precision == MPLU_BF16;
    const int NB = effective_nb(c, npad);
    const std::vector<int> tb = tile_bounds(npad, NB, c->opts.edge_nb);  // block column m = [tb[m], tb[m+1])
    const int nt = (int)tb.size() - 1;
    const int w0 = tb[1];
    if (nt >= mplu_context::kMaxSteps) return MPLU_E_ARG;
    cudaStream_t st = c->stream;
    int side_sms = c->opts.side_sms_left > 0 ? c->opts.side_sms_left : 16;
    side_sms -= side_sms % 2;
    const bool two = c->opts.lookahead != 0 && side_sms >= 2 && side_sms <= c->num_sms - 16 && nt > 2;
    const Lane all{st, 0};
    const Lane bulk = two ? Lane{st, c->num_sms - side_sms} : all;
    const Lane chain = two ? Lane{c->side, side_sms, true} : all;
    const Sched S{c, ld, (long long)c->cap_nb};
    // chain: U(j-1,j) ready, GETRF(D_j) done; bulk: column j has its updates k < j-1, rows below tile j of column j have update j-1
    enum { EV_U = 0, EV_G = 1, EV_COL = 2, EV_B1 = 3 };
    cudaEvent_t ev = nullptr;

    if (!c->prologue_done) {  // else prologue_left() has done this part, overlapped with the first touch
        if (!c->trace) CKI(launch_scales(c->amax, c->scales, c->opts.a_exp, c->opts.l_exp, bf16, st));
        CKI(traced_cast(c, 0, 0, npad, w0, st));
        if (npad > w0)
            CKI(traced_cast(c, 0, w0, w0, npad - w0, st));
        c->kernel_launches += 3;
        CKI(traced_clear_bands(c, st));
        CKI(S.getrf(all, 0, 0, w0));
        if (w0 < npad) CKI(S.trsm_l(all, 0, 0, w0, w0, npad));
    }
    // Two lanes: U(j, j+1), the first thing step j+1 needs, rides in the launch that ends step j on the chain lane
    // (it is independent of that step's L(j+1, j)); here for j = 0.
    bool u_done = false;
    if (two) {
        CKI(S.trsm_u(all, 0, 0, w0, tb[1], tb[2]));
        CKI(step_event(c, 1, EV_U, &ev));
        CKI(ev_record(c, ev, st));
        u_done = true;
        CKI(ev_record(c, c->ev_fork, st));
        CKI(ev_wait(c, c->side, c->ev_fork));
    }
    // the bulk lane's tall updates: rows r0.. of block columns [c0, c1), full shadow
    // `last`: this is the block columns' final update (k = column - 1): everything below gets its 16-bit shadow (the
    // GETRF / L-panel solve read it); an intermediate update only shadows tile row k+1, which the next panel solve
    // U(k+1,.) reads -- the rest would be overwritten by update k+1 anyway, and the full-shadow epilogue costs the
    // tall update a fifth of its rate (855 vs 1109 TFLOP/s at 30720 x 30720 x 2048)
    auto big_schur = [&](const Lane& ln, int r0, int c0, int c1, int k0, int k1, bool last, int next_rows) -> int {
        return S.schur(ln, r0, npad, c0, c1, k0, k1, last ? npad - r0 : next_rows, last ? c1 - c0 : 0, k0 == 0);
    };
    auto timed_schur = [&](const Lane& ln, int r0, int c0, int c1, int k0, int k1, int next_rows) -> int {
        // every rank-nb update of the bulk lane is timed with its own event pair for the roofline figure
        const bool timed = !c->trace && c->trail_count < mplu_context::kMaxTrail;
        if (timed) {
            cudaEvent_t& e0 = c->trail_ev[2 * c->trail_count];
            if (!e0) { CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&c->trail_ev[2 * c->trail_count + 1])); }
            CKI(record_event(c, e0, ln.st));
        }
        CKI(big_schur(ln, r0, c0, c1, k0, k1, false, next_rows));
        if (timed) {
            CKI(record_event(c, c->trail_ev[2 * c->trail_count + 1], ln.st));
            c->trail_count++;
            c->trail_flops += 2.0 * (npad - r0) * (double)(c1 - c0) * (k1 - k0);
            c->trail_bytes += 8.0 * (npad - r0) * (double)(c1 - c0);
        }
        return 0;
    };
    auto colb = [&](int m) { return tb[m < nt ? m : nt]; };
    // Bulk lane, opts.pair_ts: the panel solve U(k, cols) of an op is a one-wave launch with a triangular operand (K per
    // tile uneven: ~35 % of the lane's rate) -- it rides in the launch of the PREVIOUS op's tall update when their column
    // ranges are disjoint (then the two products touch disjoint data), filling that launch's tail instead of standing
    // alone.  `pend` = an update that has been formed but not launched yet; events that must follow it wait in `pend_ev`.
    struct Pending { bool have = false; GemmCall g{}; int c0 = 0, c1 = 0; bool timed = false; double flops = 0, bytes = 0; } pend;
    std::vector<cudaEvent_t> pend_ev;
    const bool pair_ts = two && c->opts.pair_ts != 0 && c->opts.group != 0;
    // launch the pending update, optionally together with the independent panel solve `t`
    auto launch_pending = [&](const GemmCall* t, double t_flops) -> int {
        if (!pend.have) return t ? run_gemm(c, bulk, *t) : 0;
        const bool timed = pend.timed && !c->trace && c->trail_count < mplu_context::kMaxTrail;
        if (timed) {
            cudaEvent_t& e0 = c->trail_ev[2 * c->trail_count];
            if (!e0) { CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&c->trail_ev[2 * c->trail_count + 1])); }
            CKI(record_event(c, e0, bulk.st));
        }
        if (t) { const GemmCall both[2] = {pend.g, *t}; CKI(run_gemm_group(c, bulk, both, 2)); }
        else CKI(run_gemm(c, bulk, pend.g));
        if (timed) {
            CKI(record_event(c, c->trail_ev[2 * c->trail_count + 1], bulk.st));
            c->trail_count++;
            c->trail_flops += pend.flops + (t ? t_flops : 0.0);
            c->trail_bytes += pend.bytes;
        }
        pend.have = false;
        for (cudaEvent_t e : pend_ev) CKI(ev_record(c, e, bulk.st));
        pend_ev.clear();
        return 0;
    };
    auto record_after_pending = [&](cudaEvent_t e) -> int {
        if (pend.have) { pend_ev.push_back(e); return 0; }
        return ev_record(c, e, bulk.st);
    };
    auto apply = [&](int k, int m0, int m1, int kn = 1) -> int {
        const int k0 = tb[k], k1 = tb[k + 1], d0 = colb(m0), d1 = colb(m1);
        const int next_rows = colb(k + 2) - k1;  // tile row k+1 is what the next panel solve reads
        if (kn == 2) {
            // updates k and k+1 in one pass: U(k,.) -> update k on tile row k+1 only (its U(k+1,.) solve reads it) -> U(k+1,.)
            // -> rows below tile row k+1 receive both updates from the two adjacent panels as ONE product with K = both widths
            const int k2 = colb(k + 2);
            CKI(launch_pending(nullptr, 0.0));
            CKI(S.trsm_u(bulk, k0, k0, k1 - k0, d0, d1));
            CKI(S.schur(bulk, k1, k2, d0, d1, k0, k1, k2 - k1, 0, k0 == 0));
            CKI(S.trsm_u(bulk, k1, k1, k2 - k1, d0, d1));
            if (k2 < npad) {
                const bool timed = !c->trace && c->trail_count < mplu_context::kMaxTrail;
                if (timed) {
                    cudaEvent_t& e0 = c->trail_ev[2 * c->trail_count];
                    if (!e0) { CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&c->trail_ev[2 * c->trail_count + 1])); }
                    CKI(record_event(c, e0, bulk.st));
                }
                CKI(S.schur(bulk, k2, npad, d0, d1, k0, k2, colb(k + 3) - k2, 0, k0 == 0));
                if (timed) {
                    CKI(record_event(c, c->trail_ev[2 * c->trail_count + 1], bulk.st));
                    c->trail_count++;
                    c->trail_flops += 2.0 * (npad - k2) * (double)(d1 - d0) * (k2 - k0);
                    c->trail_bytes += 8.0 * (npad - k2) * (double)(d1 - d0);
                }
            }
            return 0;
        }
        if (!pair_ts) {
            CKI(S.trsm_u(bulk, k0, k0, k1 - k0, d0, d1));
            return timed_schur(bulk, k1, d0, d1, k0, k1, next_rows);
        }
        const GemmCall t = S.trsm_u_call(k0, k0, k1 - k0, d0, d1);
        const bool indep = pend.have && (d1 <= pend.c0 || d0 >= pend.c1);
        if (indep) CKI(launch_pending(&t, (double)(k1 - k0) * (k1 - k0) * (d1 - d0)));
        else { CKI(launch_pending(nullptr, 0.0)); CKI(run_gemm(c, bulk, t)); }
        pend.have = true;
        pend.g = S.schur_call(k1, npad, d0, d1, k0, k1, next_rows, 0, k0 == 0);
        pend.c0 = d0; pend.c1 = d1; pend.timed = true;
        pend.flops = 2.0 * (npad - k1) * (double)(d1 - d0) * (k1 - k0);
        pend.bytes = 8.0 * (npad - k1) * (double)(d1 - d0);
        return 0;
    };
    const std::vector<LeftOp> plan = plan_left(tb, c->opts.eager != 0, two && c->opts.update_pair != 0);
    size_t pi = 0;
    for (int j = 1; j < nt; ++j) {
        const int c0 = tb[j], c1 = tb[j + 1], w = c1 - c0;
        const int c2 = colb(j + 2);  // end of tile row j+1
        const int kp = tb[j - 1];    // previous block column [kp, c0)
        // ---- chain lane
        if (!two)  // single lane: plain left-looking, column j receives its updates k < j-1 here
            for (int k = 0; k + 2 <= j; ++k) CKI(apply(k, j, j + 1));
        CKI(mark(c, 1000 + j, chain.st));
        if (!u_done) {
            if (two && j >= 2) {  // the bulk lane gave column j its updates k < j-1
                CKI(step_event(c, j, EV_COL, &ev));
                CKI(ev_wait(c, chain.st, ev));
            }
            CKI(S.trsm_u(chain, kp, kp, c0 - kp, c0, c1));
            if (two) { CKI(step_event(c, j, EV_U, &ev)); CKI(ev_record(c, ev, chain.st)); }
        }
        u_done = false;
        CKI(S.schur(chain, c0, two ? c1 : npad, c0, c1, kp, c0, (two ? c1 : npad) - c0, w, kp == 0));
        CKI(mark(c, 2000 + j, chain.st));
        CKI(S.getrf(chain, c0, c0, w));
        CKI(mark(c, 3000 + j, chain.st));
        if (two) { CKI(step_event(c, j, EV_G, &ev)); CKI(ev_record(c, ev, chain.st)); }
        if (!two) {
            if (c1 < npad) CKI(S.trsm_l(chain, c0, c0, w, c1, npad));
            continue;
        }
        // ---- bulk lane
        CKI(step_event(c, j, EV_U, &ev));
        CKI(ev_wait(c, bulk.st, ev));
        CKI(mark(c, 4000 + j, bulk.st));
        if (c1 < npad) {
            if (pair_ts) {  // column j's final update below its diagonal tile: may share its launch with the next op's panel solve
                pend.have = true;
                pend.g = S.schur_call(c1, npad, c0, c1, kp, c0, npad - c1, c1 - c0, kp == 0);
                pend.c0 = c0; pend.c1 = c1; pend.timed = false;
            } else {
                CKI(big_schur(bulk, c1, c0, c1, kp, c0, true, 0));
            }
            CKI(step_event(c, j, EV_B1, &ev));
            CKI(record_after_pending(ev));
        }
        CKI(mark(c, 5000 + j, bulk.st));
        if (j + 1 < nt) {
            // mandatory ops of this step (block column j+1 brought up to date), the event the chain lane's next step
            // waits for, then the eager ops (plan_left)
            for (; pi < plan.size() && plan[pi].step == j && plan[pi].mandatory; ++pi)
                CKI(apply(plan[pi].k, plan[pi].m0, plan[pi].m1, plan[pi].kn));
            CKI(step_event(c, j + 1, EV_COL, &ev));
            CKI(record_after_pending(ev));
            for (; pi < plan.size() && plan[pi].step == j; ++pi) CKI(apply(plan[pi].k, plan[pi].m0, plan[pi].m1, plan[pi].kn));
        }
        CKI(launch_pending(nullptr, 0.0));  // nothing stays pending across the wait for this step's GETRF
        CKI(mark(c, 6000 + j, bulk.st));
        if (c2 < npad) {
            CKI(step_event(c, j, EV_G, &ev));
            CKI(ev_wait(c, bulk.st, ev));
            CKI(S.trsm_l(bulk, c0, c0, w, c2, npad));
        }
        CKI(mark(c, 7000 + j, bulk.st));
        // ---- chain lane again (issued after the bulk lane's record of EV_B1: a wait must follow its record in host
        // order to be captured): tile j+1 of column j has received update j-1 from the bulk lane long before
        if (c1 < npad) {
            CKI(step_event(c, j, EV_B1, &ev));
            CKI(ev_wait(c, chain.st, ev));
            // ... and block column j+1 its updates k < j (recorded above, well before GETRF(D_j) ended): L(j+1,j) and
            // U(j,j+1) share one launch
            CKI(step_event(c, j + 1, EV_COL, &ev));
            CKI(ev_wait(c, chain.st, ev));
            CKI(run_gemm_pair(c, chain, S.trsm_l_call(c0, c0, w, c1, c2), S.trsm_u_call(c0, c0, w, c1, c2)));
            CKI(step_event(c, j + 1, EV_U, &ev));
            CKI(ev_record(c, ev, chain.st));
            u_done = true;
        }
    }
    if (two) {
        CKI(ev_record(c, c->ev_join, c->side));
        CKI(ev_wait(c, st, c->ev_join));
    }
    return 0;
}

// Left-looking schedule, first block column: the first touch of A (12 n^2 bytes, HBM bound, 2 ms at n = 32768) and the
// GETRF of the first diagonal tile (latency bound, 1.3 ms, 2-40 SMs) overlap instead of running back to back.  The
// first block column is cast first; the fp16 scale is fixed from ITS largest magnitude (it holds the first diagonal
// tile; bf16 has no scale); then the second stream factors tile 0 and solves the first L panel while this stream casts
// the other block columns.  A later block column that leaves the fp16 range under that scale raises the overflow bit
// and mplu_gesv_device redoes the factorization with the global scale (opts.early_scale = 0 asks for that directly).
// Direct launches, not part of the captured graph: they carry the caller's A pointer.
int prologue_left(mplu_context* c, const double* dA, long long lda) {
    const int n = c->n, npad = c->npad;
    const long long ld = npad;
    const int bf16 = c->opts.precision == MPLU_BF16;
    const std::vector<int> tb = tile_bounds(npad, effective_nb(c, npad), c->opts.edge_nb);
    const int NB = tb[1];  // the first block column
    const int nt = (int)tb.size() - 1;
    cudaStream_t st = c->stream;
    const int s0 = c->nchunk / nt > 0 ? c->nchunk / nt : 1;  // row-sum slots of the first block column
    if (!c->ev_pro[0]) { CK(cudaEventCreateWithFlags(&c->ev_pro[0], cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&c->ev_pro[1], cudaEventDisableTiming)); }
    CK(cudaMemsetAsync(c->amax, 0, sizeof(float), st));
    CKI(launch_first_touch_cols(dA, lda, n, c->W, ld, npad, 0, NB, c->amax, c->rowsum_part, 0, s0, st));
    CKI(launch_scales(c->amax, c->scales, c->opts.a_exp, c->opts.l_exp, bf16, st));
    CKI(launch_shadow_cast(c->W, ld, c->Wh, ld, npad, NB, c->scales + SC_A, bf16, c->status, st));
    CK(cudaMemsetAsync(c->Linv16, 0, (size_t)c->cap_nb * npad * sizeof(uint16_t), st));
    CK(cudaMemsetAsync(c->Uinv16, 0, (size_t)c->cap_nb * npad * sizeof(uint16_t), st));
    CKI(reset_fused_barriers(c, st));
    c->kernel_launches += 3;
    CK(cudaEventRecord(c->ev_pro[0], st));
    CK(cudaStreamWaitEvent(c->side, c->ev_pro[0], 0));
    {   // second stream: tile 0 and the first L panel, every SM it can get next to the bandwidth-bound cast
        const Sched S{c, ld, (long long)c->cap_nb};
        const Lane lane{c->side, 0};
        CKI(S.getrf(lane, 0, 0, NB));
        CKI(S.trsm_l(lane, 0, 0, NB, NB, npad));
        CK(cudaEventRecord(c->ev_pro[1], c->side));
    }
    // The cast of the other block columns must leave room on every SM for the second stream's CTAs (a GEMM CTA needs
    // 320 threads, diag_lu 512): about 5 blocks of 256 threads per SM instead of the 8 that would otherwise be resident
    // for the whole kernel -- with a full grid every one of tile 0's 61 dependent launches waited for a wave boundary
    // of the cast and the overlap gained nothing.  768 blocks x 256 threads x 4 loads in flight still saturate HBM.
    int s1 = (5 * c->num_sms) / ((npad + 255) / 256);
    if (s1 < 1) s1 = 1;
    if (s1 > c->nchunk - s0) s1 = c->nchunk - s0;
    CKI(launch_first_touch_cols(dA, lda, n, c->W, ld, npad, NB, npad, c->amax, c->rowsum_part, s0, s1, st));
    CKI(launch_shadow_cast(c->W + (long long)NB * ld, ld, c->Wh + (long long)NB * ld, ld, NB, npad - NB, c->scales + SC_A,
                           bf16, c->status, st));
    CKI(launch_anorm(c->rowsum_part, n, s0 + s1, c->anorm, st));
    c->kernel_launches += 3;
    CK(cudaStreamWaitEvent(st, c->ev_pro[1], 0));
    return 0;
}

int factor_impl(mplu_context* c, int n, const double* dA, long long lda) {
    CKI(ensure_work(c, n));
    const int npad = c->npad;
    cudaStream_t st = c->stream;
    CK(cudaMemsetAsync(c->status, 0, sizeof(int), st));
    // Equilibration: with scales to apply, W = diag(r) A diag(c) comes from the eager first touch (the lazy one and the
    // early-scale prologue read A itself); the captured schedule is the same.  EQUED = N changes nothing below.
    c->equed = 0;
    int eq_kern = 0;
    if (c->opts.equilibrate == 1) {
        CKI(equilibrate(c, dA, lda));
        eq_kern = 4;
    }
    const bool scaled = c->equed != 0;
    // left-looking schedule with at least two block columns: the first touch overlaps the first diagonal tile
    // Lazy first touch (left-looking schedule, order a multiple of 128, at least two block columns): only the first
    // block column and block row are cast here; every other tile's first update reads its addend from the fp64 matrix
    // itself (GemmParams::cin64), which removes the 12 n^2-byte cast pass.  The fp16 scale then comes from those two
    // panels; a later entry that leaves the fp16 range under it raises the overflow bit and the caller redoes the
    // factorization with the full first touch and the global scale (allow_early = false), like early_scale.
    const int NB0 = effective_nb(c, npad);
    const bool lazy = !scaled && c->opts.schedule == MPLU_SCHED_LEFT && c->opts.lazy_touch != 0 && c->allow_early &&
                      npad == n && npad > NB0 && c->opts.tile_ws == 0 && !c->trace;
    const bool early = !scaled && !lazy && c->opts.schedule == MPLU_SCHED_LEFT && c->opts.early_scale != 0 &&
                       c->allow_early && npad > NB0 && c->opts.tile_ws == 0;
    c->lazy = lazy;
    c->anorm_pending = lazy;
    c->prologue_done = early;
    c->used_early_scale = (early || lazy) && c->opts.precision != MPLU_BF16;
    int pro_gemm = 0, pro_kern = 0;
    if (lazy) {
        if (!c->aref) CK(cudaMalloc(&c->aref, sizeof(ARef)));
        const ARef href{dA, lda};
        CK(cudaMemcpyAsync(c->aref, &href, sizeof(href), cudaMemcpyHostToDevice, st));  // pageable source: staged at once
        CK(cudaMemsetAsync(c->amax, 0, sizeof(float), st));
        const int w0 = tile_bounds(npad, NB0, c->opts.edge_nb)[1];  // first block column / block row
        CKI(launch_first_touch_cols(dA, lda, n, c->W, npad, npad, 0, w0, c->amax, nullptr, 0, 64, st));
        CKI(launch_first_touch_block(dA, lda, n, c->W, npad, npad, w0, w0, npad, c->amax, st));
    } else if (early) {
        c->gemm_launches = c->kernel_launches = 0;
        CKI(prologue_left(c, dA, lda));
        pro_gemm = c->gemm_launches;
        pro_kern = c->kernel_launches;
    } else {
        CKI(launch_first_touch(dA, lda, n, c->W, npad, npad, c->amax, c->rowsum_part, c->nchunk, c->anorm, st,
                               scaled ? c->eq_r : nullptr, scaled ? c->eq_c : nullptr));
    }

    const bool use_graph = c->opts.use_graph != 0;
    {
        const int NB = effective_nb(c, npad);
        if (c->opts.tile_ws != 0 && npad > NB) {
            const bool two = c->opts.lookahead != 0 && npad > 2 * NB;
            CKI(prepare_tile_workspace(c, NB, two ? c->side : st));
        }
    }
    // every option and pointer the captured schedule depends on, one value per slot (no packing, no struct padding)
    const mplu_options& o = c->opts;
    const std::vector<long long> key = {
        n, npad, effective_nb(c, npad), o.precision, o.gemm_variant, o.max_sms, o.lookahead, o.side_sms, o.a_exp, o.l_exp,
        o.pdl, o.group, o.tile_ws, o.cg2_min_elems, o.side_sms_early, o.early_pct, o.late_pct, o.tri_skip, o.l2_persist,
        o.schedule, o.eager, o.side_sms_left, o.stream_c, o.fuse_w, o.fuse_ctas, o.flow_w, o.flow_ctas, o.flow_merge_ctas, o.edge_nb, o.pair_ts, o.update_pair, (long long)c->flow_prof_launch, (long long)early, (long long)lazy, (long long)c->marks_on,
        (long long)reinterpret_cast<uintptr_t>(c->W), (long long)reinterpret_cast<uintptr_t>(c->tile ? c->tile->W : nullptr)};
    const bool hit = use_graph && c->graph_exec && key == c->gkey;
    if (!hit) {
        c->gemm_launches = 0;
        c->kernel_launches = early ? 0 : 2;  // first touch + anorm (lazy: the two panel casts)
        c->trail_count = 0;
        c->trail_flops = c->trail_bytes = 0;
        c->mark_count = 0;
        if (use_graph) {
            if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
            CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
            c->capturing = true;
            int rc = c->opts.schedule == MPLU_SCHED_LEFT ? enqueue_factorization_left(c) : enqueue_factorization(c);
            c->capturing = false;
            cudaGraph_t graph = nullptr;
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            if (e != cudaSuccess) return (int)e;
            e = cudaGraphInstantiate(&c->graph_exec, graph, 0);
            cudaGraphDestroy(graph);
            if (e != cudaSuccess) { c->graph_exec = nullptr; return (int)e; }
            c->gkey = key;
            c->g_gemm_launches = c->gemm_launches; c->g_kernel_launches = c->kernel_launches;
            c->g_trail_count = c->trail_count; c->g_trail_flops = c->trail_flops; c->g_trail_bytes = c->trail_bytes;
        } else {
            CKI(c->opts.schedule == MPLU_SCHED_LEFT ? enqueue_factorization_left(c) : enqueue_factorization(c));
        }
    }
    if (use_graph) {
        CKI(upload_fused_programs(c, st));  // programs recorded during the capture (no-op on a cache hit)
        if (c->tile) CKI(upload_fused_programs(c->tile, st));
        c->gemm_launches = c->g_gemm_launches; c->kernel_launches = c->g_kernel_launches;
        c->trail_count = c->g_trail_count; c->trail_flops = c->g_trail_flops; c->trail_bytes = c->g_trail_bytes;
        CK(cudaGraphLaunch(c->graph_exec, st));
    }
    c->gemm_launches += pro_gemm;
    c->kernel_launches += pro_kern + eq_kern;
    c->factored = true;
    return 0;
}

// Host-resident input (mplu_gesv_host): the factorization runs LEFT-looking over nb-wide block columns so that it
// overlaps the PCIe transfer, which is 4x longer than the whole device-resident solve (8 n^2 bytes at ~55 GB/s).
// Block column j is copied on the copy stream; as soon as it has arrived the compute stream casts it (first touch),
// brings it up to date with the j block columns factored before it -- U_kj = inv(L_kk) A_kj, A_{k+1:,j} -= L_{k+1:,k} U_kj
// for k = 0..j-1, the reference's Dtrsm / Dgemm pair (MPF.cu:215-239) applied per arriving block column --, factors its
// diagonal tile and solves its L panel.  Every tile receives the same products in the same order as in the
// right-looking schedule, so the factors are bit-identical to mplu_factor_device's; what remains after the last
// byte has arrived is the last block column's update chain and one diagonal-tile GETRF.
// The fp16 scale has to be fixed before the first cast: it is taken from the first block column (which holds the
// first diagonal tile); a later block column that leaves the fp16 range under that scale sets the overflow bit and
// the caller redoes the solve from the (by then resident) device copy with the global scale.
// Equilibration (opts.equilibrate) is not streamed: a row scale needs every column of its row before the first cast,
// so with it gesv_host_impl copies A first and runs the device path.
bool streamed_supported(const mplu_context* c, int n) {
    const int npad = ((n + kDiagBlock - 1) / kDiagBlock) * kDiagBlock;
    const int NB = effective_nb(c, npad);
    const int nt = (npad + NB - 1) / NB;
    return nt >= 2 && nt <= c->nchunk && nt < mplu_context::kMaxSteps;
}

int factor_streamed(mplu_context* c, int n, const double* hA, long long lda, double* dA) {
    CKI(ensure_work(c, n));
    const int npad = c->npad;
    const long long ld = npad;
    const int bf16 = c->opts.precision == MPLU_BF16;
    const int NB = effective_nb(c, npad);
    const int nt = (npad + NB - 1) / NB;
    const int per = c->nchunk / nt;  // row-sum slots per block column
    if (per < 1 || nt >= mplu_context::kMaxSteps) return MPLU_E_ARG;
    c->equed = 0;  // equilibration needs all of A before the first cast: gesv_host_impl does not stream then
    cudaStream_t st = c->stream, cp = c->copy;
    CK(cudaMemsetAsync(c->status, 0, sizeof(int), st));
    CK(cudaMemsetAsync(c->amax, 0, sizeof(float), st));
    CK(cudaMemsetAsync(c->Linv16, 0, (size_t)c->cap_nb * npad * sizeof(uint16_t), st));
    CK(cudaMemsetAsync(c->Uinv16, 0, (size_t)c->cap_nb * npad * sizeof(uint16_t), st));
    CKI(reset_fused_barriers(c, st));
    c->gemm_launches = 0;
    c->kernel_launches = 0;
    c->trail_count = 0;
    c->trail_flops = c->trail_bytes = 0;
    c->mark_count = 0;
    const Sched S{c, ld, (long long)c->cap_nb};
    const Lane all{st, 0};
    for (int j = 0; j < nt; ++j) {
        const int c0 = j * NB, c1 = (c0 + NB < npad) ? c0 + NB : npad, w = c1 - c0;
        const int real = (n < c1 ? n : c1) - c0;  // columns of A in this block column (the rest is padding)
        if (real > 0)
            CK(cudaMemcpy2DAsync(dA + (size_t)c0 * n, (size_t)n * sizeof(double), hA + (size_t)c0 * lda,
                                 (size_t)lda * sizeof(double), (size_t)n * sizeof(double), real, cudaMemcpyHostToDevice, cp));
        cudaEvent_t& e = c->ev_copy[j];
        if (!e) CK(cudaEventCreate(&e));
        CK(cudaEventRecord(e, cp));
        CK(cudaStreamWaitEvent(st, e, 0));
        CKI(launch_first_touch_cols(dA, n, n, c->W, ld, npad, c0, c1, c->amax, c->rowsum_part, j * per, per, st));
        if (j == 0) CKI(launch_scales(c->amax, c->scales, c->opts.a_exp, c->opts.l_exp, bf16, st));
        CKI(launch_shadow_cast(c->W + (long long)c0 * ld, ld, c->Wh + (long long)c0 * ld, ld, npad, w, c->scales + SC_A,
                               bf16, c->status, st));
        c->kernel_launches += (j == 0) ? 3 : 2;
        for (int k0 = 0; k0 < c0; k0 += NB) {
            const int k1 = k0 + NB;
            CKI(S.trsm_u(all, k0, k0, NB, c0, c1));
            // the last update shadows everything below (GETRF / L-panel solve read it), the others only tile row k+1
            const bool last = k1 >= c0;
            CKI(S.schur(all, k1, npad, c0, c1, k0, k1, last ? npad - k1 : NB, last ? w : 0));
        }
        CKI(S.getrf(all, c0, c0, w));
        if (c1 < npad) CKI(S.trsm_l(all, c0, c0, w, c1, npad));
    }
    c->copy_last = nt - 1;
    CKI(launch_anorm(c->rowsum_part, n, nt * per, c->anorm, st));
    c->kernel_launches++;
    c->factored = true;
    return 0;
}

__global__ void widen_kernel(const float* __restrict__ W, long long ldw, int n, double* __restrict__ out,
                             long long ldo) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    for (int c = blockIdx.y; c < n; c += gridDim.y) out[r + (long long)c * ldo] = (double)W[r + (long long)c * ldw];
}

int refine(const RefineOps& ops, int n, int k, int max_iters, double tol, RefineResult* res) {
    const double eps = 2.220446049250313e-16 / 2.0;  // LAPACK dlamch('E')
    if (max_iters <= 0) max_iters = 30;
    res->col.assign(k, RefineColumn{});
    std::vector<double> h(3 * (size_t)k);
    CKI(ops.first_solve());
    for (bool first = true;; first = false) {
        bool formed_anorm = false;
        CKI(ops.residual(&formed_anorm));
        CK(cudaMemcpyAsync(h.data(), ops.norms, h.size() * sizeof(double), cudaMemcpyDeviceToHost, ops.st));
        if (first || formed_anorm) CK(cudaMemcpyAsync(&res->anorm, ops.anorm, sizeof(double), cudaMemcpyDeviceToHost, ops.st));
        CKI(ops.wait());
        const double an = res->anorm;
        bool all = true, nan = false;
        for (int j = 0; j < k; ++j) {
            RefineColumn& cj = res->col[j];
            cj.rnorm = h[2 * j];
            cj.xnorm = h[2 * j + 1];
            cj.bnorm = h[2 * k + j];
            cj.berr = backward_error(cj.rnorm, an, cj.xnorm, cj.bnorm);
            if (first) cj.first_berr = cj.berr;
            const double thresh = tol > 0 ? tol * an * cj.xnorm : cj.xnorm * an * eps * std::sqrt((double)n);
            if (!(cj.rnorm == cj.rnorm)) nan = true;
            if (!(cj.rnorm <= thresh)) all = false;
        }
        if (nan) break;  // NaN: give up
        if (all) { res->converged = 1; break; }
        if (res->iters >= max_iters) break;
        int steps = 0;
        CKI(ops.correct(&steps));
        res->gmres_iters += steps;
        ++res->iters;
    }
    return 0;
}

void refine_stats(const RefineResult& res, int n, double* berr, mplu_stats* stats) {
    const int k = (int)res.col.size();
    if (berr)
        for (int j = 0; j < k; ++j) berr[j] = res.col[j].berr;
    if (!stats) return;
    int w = 0;  // the worst column (a NaN is worse than anything)
    for (int j = 1; j < k; ++j) {
        const double bj = res.col[j].berr, bw = res.col[w].berr;
        if (bj > bw || (bj != bj && bw == bw)) w = j;
    }
    stats->n = n;
    stats->iters = res.iters;
    stats->converged = res.converged;
    stats->anorm_inf = res.anorm;
    stats->bnorm_inf = res.col[w].bnorm;
    stats->xnorm_inf = res.col[w].xnorm;
    stats->rnorm_inf = res.col[w].rnorm;
    stats->backward_error = res.col[w].berr;
    stats->first_backward_error = std::max_element(res.col.begin(), res.col.end(), [](const RefineColumn& a, const RefineColumn& b) {
        return a.first_berr < b.first_berr;
    })->first_berr;
}

int refine_rc(int converged, int status_bits) {
    if (converged) return 0;
    if (status_bits & 1) return MPLU_E_OVERFLOW;
    if (status_bits & 2) return MPLU_E_ZEROPIVOT;
    return MPLU_E_NOCONV;
}

int dsgesv_iter(int rc, int iters) {
    return rc == 0 ? iters : (rc == MPLU_E_OVERFLOW ? -2 : (rc == MPLU_E_NOCONV ? -(iters + 1) : -3));
}

// The right-hand sides of one call: nrhs column-major columns of B (ldb) and X (ldx); berr: host array of nrhs or null.
struct RhsBlock {
    int nrhs;
    const double* B; long long ldb;
    double* X; long long ldx;
    double* berr;
};

// X = (LU)^-1 B, refined.  One column runs the single-vector kernels on c->r / c->norms.  More columns run the block
// kernels on the rb_* buffers, which stream A and the factors once per kResidualBlock / kSolveBlock columns; GMRES
// refinement runs gmres_correction column by column (not batched).
int solve_impl(mplu_context* c, const double* dA, long long lda, const RhsBlock& b, mplu_stats* stats) {
    if (!c->factored) return MPLU_E_NOTFACTORED;
    const int n = c->n, npad = c->npad, k = b.nrhs;
    const long long ld = npad;
    cudaStream_t st = c->stream;
    if (k > 1) CKI(ensure_rhs_work(c, k));
    double* R = k == 1 ? c->r : c->rb_R;  // the residual columns (ld n)
    double* norms = k == 1 ? c->norms : c->rb_norms;
    // D = (LU)^-1 rhs: D -> d_out, or x_accum += D (both with ld ldo)
    auto solve = [&](const double* rhs, long long ldr, double* d_out, double* x_accum, long long ldo) -> int {
        if (k == 1) {
            c->kernel_launches += 1;
            return launch_lu_solve(c->W, ld, n, npad, c->Linv32, c->Uinv32, rhs, c->y, d_out, x_accum, c->ready, st);
        }
        for (int j0 = 0; j0 < k; j0 += kSolveBlock) {
            const int kc = std::min(kSolveBlock, k - j0);
            CKI(launch_lu_solve_block(c->W, ld, n, npad, c->Linv32, c->Uinv32, rhs + (long long)j0 * ldr, ldr, kc, c->rb_y,
                                      d_out ? d_out + (long long)j0 * ldo : nullptr, ldo,
                                      x_accum ? x_accum + (long long)j0 * ldo : nullptr, ldo, c->ready, st));
            c->kernel_launches += 2;
        }
        return 0;
    };
    // equilibrated factors (of diag(r) A diag(c)): every solve with them is C (LU)^-1 R, through the n x k scratch D
    const bool eq_rows = c->equed & 1, eq_cols = c->equed & 2;
    if (c->equed) CKI(ensure_equil_scratch(c, (size_t)n * k));
    double* D = c->eq_D;
    auto scale = [&](const double* s, const double* in, long long ldi, double* out, long long ldo, int accumulate) -> int {
        c->kernel_launches += 1;
        return launch_diag_scale(s, n, k, in, ldi, out, ldo, accumulate, st);
    };
    RefineOps ops;
    ops.norms = norms;
    ops.anorm = c->anorm;
    ops.st = st;
    ops.first_solve = [&]() -> int {
        CKI(launch_column_absmax(b.B, b.ldb, n, k, norms + 2 * k, st));
        c->kernel_launches += 1;
        if (!eq_rows) CKI(solve(b.B, b.ldb, b.X, nullptr, b.ldx));
        else {
            CKI(scale(c->eq_r, b.B, b.ldb, D, n, 0));
            CKI(solve(D, n, b.X, nullptr, b.ldx));
        }
        return eq_cols ? scale(c->eq_c, b.X, b.ldx, b.X, b.ldx, 0) : 0;
    };
    ops.residual = [&](bool* formed_anorm) -> int {
        // lazy first touch: ||A||_inf rides in the first residual pass (of the first column block): it streams A anyway
        const bool with_anorm = c->anorm_pending;
        if (k == 1) {
            CKI(launch_residual(dA, lda, n, b.X, b.B, R, c->partial, c->nchunk, norms, st, with_anorm ? c->rowsum_part : nullptr,
                                with_anorm ? c->anorm : nullptr));
            c->kernel_launches += 2;
        } else {
            for (int j0 = 0; j0 < k; j0 += kResidualBlock) {
                const int kc = std::min(kResidualBlock, k - j0);
                const bool abs_here = with_anorm && j0 == 0;
                CKI(launch_residual_block(dA, lda, n, b.X + (long long)j0 * b.ldx, b.ldx, b.B + (long long)j0 * b.ldb, b.ldb,
                                          R + (long long)j0 * n, n, kc, c->rb_partial, norms + 2 * j0, st,
                                          abs_here ? c->rowsum_part : nullptr, abs_here ? c->anorm : nullptr));
                c->kernel_launches += 2;
            }
        }
        c->anorm_pending = false;
        *formed_anorm = with_anorm;
        return 0;
    };
    ops.correct = [&](int* krylov_steps) -> int {
        if (c->opts.refinement != MPLU_REFINE_GMRES) {
            // R is recomputed by the next residual pass, so it is scaled in place; without C the correction accumulates
            // straight into X
            if (eq_rows) CKI(scale(c->eq_r, R, n, R, n, 0));
            if (!eq_cols) return solve(R, n, nullptr, b.X, b.ldx);
            CKI(solve(R, n, D, nullptr, n));
            return scale(c->eq_c, D, n, b.X, b.ldx, 1);
        }
        for (int j = 0; j < k; ++j) {
            int inner = 0;
            CKI(gmres_correction(c, dA, lda, R + (long long)j * n, b.X + (long long)j * b.ldx, &inner));
            *krylov_steps += inner;
        }
        return 0;
    };
    ops.wait = [&]() -> int { return (int)cudaStreamSynchronize(st); };
    RefineResult res;
    CKI(refine(ops, n, k, c->opts.max_iters, c->opts.tol, &res));
    int h_status = 0;
    CK(cudaMemcpy(&h_status, c->status, sizeof(int), cudaMemcpyDeviceToHost));
    refine_stats(res, n, b.berr, stats);
    if (stats) {
        stats->status_bits = h_status;
        stats->equed = c->equed;
        stats->gmres_iters = res.gmres_iters;
        stats->gemm_launches = c->gemm_launches;
        stats->kernel_launches = c->kernel_launches;
        stats->trailing_launches = c->trail_count;
        stats->trailing_flops = c->trail_flops;
        stats->trailing_bytes = c->trail_bytes;
        float tms = 0.f;
        for (int i = 0; i < c->trail_count; ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, c->trail_ev[2 * i], c->trail_ev[2 * i + 1]) == cudaSuccess) tms += ms;
        }
        stats->trailing_ms = tms;
    }
    return refine_rc(res.converged, h_status);
}

// factor + solve from device-resident inputs with the cascade of LAPACK dsgesv: early-scale redo, bf16 on fp16 overflow,
// fp64 fallback (mplu_gesv_device / mplu_gesv_device_nrhs; arguments already checked)
int gesv_device_impl(mplu_context* c, int n, const double* dA, long long lda, const RhsBlock& b, const mplu_options* opts,
                     mplu_stats* stats) {
    CK(cudaSetDevice(c->device));
    if (opts) c->opts = *opts;
    const OptionsScope scope(c);
    resolve_options(c, n);
    if (stats) memset(stats, 0, sizeof(*stats));
    c->factored = false;
    CK(cudaEventRecord(c->ev[0], c->stream));
    int rc = factor_impl(c, n, dA, lda);
    if (rc) return rc;
    CK(cudaEventRecord(c->ev[1], c->stream));
    rc = solve_impl(c, dA, lda, b, stats);
    if (rc == MPLU_E_OVERFLOW && c->used_early_scale) {
        // the fp16 scale taken from the first block column did not fit a later one: once more with the global scale
        c->allow_early = false;
        c->factored = false;
        rc = factor_impl(c, n, dA, lda);
        c->allow_early = true;
        if (rc) return rc;
        if (stats) memset(stats, 0, sizeof(*stats));
        rc = solve_impl(c, dA, lda, b, stats);
    }
    if (rc == MPLU_E_OVERFLOW && c->opts.precision == MPLU_FP16 && c->opts.bf16_fallback) {
        // like dsgesv's fall back to full precision: same algorithm, operand type without the range problem
        c->opts.precision = MPLU_BF16;
        c->factored = false;
        rc = factor_impl(c, n, dA, lda);
        if (rc) return rc;
        if (stats) memset(stats, 0, sizeof(*stats));
        rc = solve_impl(c, dA, lda, b, stats);
    }
    if (stats) {
        stats->precision_used = c->opts.precision;
        stats->dsgesv_iter = dsgesv_iter(rc, stats->iters);
    }
    if ((rc == MPLU_E_OVERFLOW || rc == MPLU_E_ZEROPIVOT || rc == MPLU_E_NOCONV) && c->opts.fp64_fallback)
        rc = fp64_fallback_solve(c, n, dA, lda, b.nrhs, b.B, b.ldb, b.X, b.ldx, rc, b.berr, stats);  // dsgesv: full-precision factorization and solve
    CK(cudaEventRecord(c->ev[2], c->stream));
    CK(cudaEventSynchronize(c->ev[2]));
    if (stats) {
        cudaEventElapsedTime(&stats->factor_ms, c->ev[0], c->ev[1]);
        cudaEventElapsedTime(&stats->solve_ms, c->ev[1], c->ev[2]);
        cudaEventElapsedTime(&stats->total_ms, c->ev[0], c->ev[2]);
    }
    return rc;
}

// n x ncols column-major copy between host and device (one contiguous copy for a single column)
cudaError_t copy_columns(double* dst, long long ldd, const double* src, long long lds, int n, int ncols, cudaMemcpyKind kind,
                         cudaStream_t st) {
    if (ncols == 1) return cudaMemcpyAsync(dst, src, n * sizeof(double), kind, st);
    return cudaMemcpy2DAsync(dst, (size_t)ldd * sizeof(double), src, (size_t)lds * sizeof(double), (size_t)n * sizeof(double),
                             ncols, kind, st);
}

// factor + solve from host buffers (mplu_gesv_host / mplu_gesv_host_nrhs; arguments already checked): b holds HOST pointers
int gesv_host_impl(mplu_context* c, int n, const double* hA, long long lda, const RhsBlock& hb, const mplu_options* opts,
                   mplu_stats* stats) {
    CK(cudaSetDevice(c->device));
    const size_t need = (size_t)n * n;
    if (need > c->dA_cap) {
        cudaFree(c->dA_stage);
        c->dA_stage = nullptr; c->dA_cap = 0;
        CK(cudaMalloc(&c->dA_stage, need * sizeof(double)));
        c->dA_cap = need;
    }
    const size_t vneed = (size_t)n * hb.nrhs;
    if (vneed > c->dv_cap) {
        cudaFree(c->db_stage); cudaFree(c->dx_stage);
        c->db_stage = c->dx_stage = nullptr; c->dv_cap = 0;
        CK(cudaMalloc(&c->db_stage, vneed * sizeof(double)));
        CK(cudaMalloc(&c->dx_stage, vneed * sizeof(double)));
        c->dv_cap = vneed;
    }
    const RhsBlock db{hb.nrhs, c->db_stage, n, c->dx_stage, n, hb.berr};  // the staged copies (ld n)
    cudaStream_t st = c->stream;
    if (opts) c->opts = *opts;
    const OptionsScope scope(c);
    const mplu_options used = c->opts;  // the request: the device path below resolves it again for itself
    resolve_options(c, n);
    CK(cudaEventRecord(c->ev[3], st));
    int rc;
    float h2d = 0.f;
    if (c->opts.stream_host && c->opts.equilibrate == 0 && streamed_supported(c, n)) {
        // block columns are factored as they arrive (factor_streamed); the staged copy of A stays for the residuals
        if (stats) memset(stats, 0, sizeof(*stats));
        c->factored = false;
        CK(cudaStreamWaitEvent(c->copy, c->ev[3], 0));
        CK(copy_columns(c->db_stage, n, hb.B, hb.ldb, n, hb.nrhs, cudaMemcpyHostToDevice, st));
        rc = factor_streamed(c, n, hA, lda, c->dA_stage);
        if (rc) return rc;
        CK(cudaEventRecord(c->ev[1], st));
        rc = solve_impl(c, c->dA_stage, n, db, stats);
        if (stats) {
            stats->precision_used = c->opts.precision;
            stats->dsgesv_iter = dsgesv_iter(rc, stats->iters);
        }
        if ((rc == MPLU_E_ZEROPIVOT || rc == MPLU_E_NOCONV) && c->opts.fp64_fallback)
            rc = fp64_fallback_solve(c, n, c->dA_stage, n, db.nrhs, db.B, db.ldb, db.X, db.ldx, rc, db.berr, stats);
        CK(cudaEventRecord(c->ev[2], st));
        CK(cudaEventSynchronize(c->ev[2]));
        cudaEventElapsedTime(&h2d, c->ev[3], c->ev_copy[c->copy_last]);
        if (stats) {
            // total = h2d (start .. last byte on the device) + factor (the tail left after it) + solve
            cudaEventElapsedTime(&stats->factor_ms, c->ev_copy[c->copy_last], c->ev[1]);
            cudaEventElapsedTime(&stats->solve_ms, c->ev[1], c->ev[2]);
            stats->total_ms = stats->factor_ms + stats->solve_ms;
        }
        if (rc == MPLU_E_OVERFLOW) {
            // the scale taken from the first block column did not fit a later one: A is resident now, redo the solve
            // with the global scale (and, if that overflows too, in bf16)
            const float streamed_ms = h2d + (stats ? stats->total_ms : 0.f);
            rc = gesv_device_impl(c, n, c->dA_stage, n, db, &used, stats);
            h2d = streamed_ms;  // everything before the redo counts as transfer time
        }
    } else {
        CK(cudaMemcpy2DAsync(c->dA_stage, (size_t)n * sizeof(double), hA, (size_t)lda * sizeof(double),
                             (size_t)n * sizeof(double), n, cudaMemcpyHostToDevice, st));
        CK(copy_columns(c->db_stage, n, hb.B, hb.ldb, n, hb.nrhs, cudaMemcpyHostToDevice, st));
        rc = gesv_device_impl(c, n, c->dA_stage, n, db, &used, stats);
        cudaEventElapsedTime(&h2d, c->ev[3], c->ev[0]);
    }
    if (rc != 0 && rc != MPLU_E_NOCONV) return rc;
    CK(cudaEventRecord(c->ev[0], st));
    CK(copy_columns(hb.X, hb.ldx, c->dx_stage, n, n, hb.nrhs, cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(c->ev[1], st));
    CK(cudaEventSynchronize(c->ev[1]));
    if (stats) {
        float d2h = 0.f;
        cudaEventElapsedTime(&d2h, c->ev[0], c->ev[1]);
        stats->h2d_ms = h2d;
        stats->d2h_ms = d2h;
        stats->total_ms += h2d + d2h;
    }
    return rc;
}

// option values the entry points check (null: the context's options, already checked)
bool options_valid(const mplu_options* o) { return !o || o->equilibrate == 0 || o->equilibrate == 1; }

// the regions spanned by the columns of B and X (first to last element) share an address: X would overwrite B
bool columns_overlap(const double* B, long long ldb, const double* X, long long ldx, int n, int nrhs) {
    const double* b1 = B + (long long)(nrhs - 1) * ldb + n;
    const double* x1 = X + (long long)(nrhs - 1) * ldx + n;
    return X < b1 && B < x1;
}

}  // namespace mplu_detail

extern "C" {

void mplu_default_options(mplu_options* o) {
    if (!o) return;
    o->precision = MPLU_FP16;
    o->nb = 0;  // auto: 2048 for n >= 12288, 1024 for n >= 4096, else 512
    o->max_iters = 30;
    o->tol = 0.0;
    o->gemm_variant = MPLU_GEMM_AUTO;
    o->max_sms = 0;
    o->a_exp = 11;
    o->l_exp = 11;
    o->lookahead = 1;
    o->side_sms = 40;
    o->use_graph = 1;
    o->pdl = 0;
    o->group = 1;
    o->refinement = MPLU_REFINE_CLASSIC;
    o->gmres_restart = 50;
    o->gmres_tol = 1e-6;
    o->bf16_fallback = 1;
    o->tile_ws = 0;
    o->l2_persist = 0;
    o->cg2_min_elems = 2048 * 2048;
    o->side_sms_early = 16;
    o->early_pct = 55;
    o->late_pct = 35;
    o->tri_skip = 1;
    o->stream_host = 1;
    o->schedule = MPLU_SCHED_LEFT;
    o->side_sms_left = 16;
    o->eager = 1;
    o->stream_c = 1;
    o->early_scale = 0;
    o->fuse_w = 512;
    o->fuse_ctas = 8;
    o->lazy_touch = 1;
    o->flow_w = 2048;
    o->flow_ctas = 16;
    o->flow_merge_ctas = -1;
    o->fp64_fallback = 1;
    o->edge_nb = 0;
    o->pair_ts = 0;
    o->update_pair = 0;
    o->equilibrate = 0;
}

int mplu_create(mplu_context** out, int device) {
    if (!out) return MPLU_E_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return MPLU_E_NODEVICE;
    if (device < 0 || device >= ndev) return MPLU_E_ARG;
    CK(cudaSetDevice(device));
    mplu_context* c = new (std::nothrow) mplu_context();
    if (!c) return MPLU_E_ARG;
    c->device = device;
    mplu_default_options(&c->opts);
    auto init = [&]() -> int {
        CK(cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device));
        if (gemm_tc_init() != 0) return MPLU_E_TMAP;
        CKI(panel_init());
        CKI(getrf_fused_init());
        CKI(getrf_flow_init());
        CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
        for (auto& e : c->ev) CK(cudaEventCreate(&e));
        CK(cudaMalloc(&c->scales, SC_COUNT * sizeof(float)));
        CK(cudaMalloc(&c->amax, sizeof(float)));
        CK(cudaMalloc(&c->anorm, sizeof(double)));
        CK(cudaMalloc(&c->norms, 3 * sizeof(double)));
        CK(cudaMalloc(&c->status, sizeof(int)));
        CK(cudaMalloc(&c->ready, sizeof(unsigned)));
        return 0;
    };
    const int rc = init();
    if (rc) { mplu_destroy(c); return rc; }  // mplu_destroy copes with a partially built context
    *out = c;
    return 0;
}

void mplu_destroy(mplu_context* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    free_work(c);
    cudaFree(c->scales); cudaFree(c->amax); cudaFree(c->anorm); cudaFree(c->norms); cudaFree(c->status); cudaFree(c->ready);
    cudaFree(c->dA_stage); cudaFree(c->db_stage); cudaFree(c->dx_stage);
    cudaFree(c->gm_V); cudaFree(c->gm_w); cudaFree(c->gm_h); cudaFree(c->gm_zero); cudaFree(c->aref);
    cudaFree(c->eq_r); cudaFree(c->eq_c); cudaFree(c->eq_words); cudaFree(c->eq_D);
    if (c->tile) { mplu_destroy(c->tile); c->tile = nullptr; }
    for (auto& e : c->ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->trail_ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_step) if (e) cudaEventDestroy(e);
    for (auto& e : c->mark_ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_copy) if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_pro) if (e) cudaEventDestroy(e);
    if (c->copy) cudaStreamDestroy(c->copy);
    if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

void* mplu_stream(mplu_context* c) { return c ? (void*)c->stream : nullptr; }

int mplu_factor_device(mplu_context* c, int n, const double* dA, long long lda, const mplu_options* opts) {
    if (!c || !dA || n <= 0 || lda < n || !options_valid(opts)) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    if (opts) c->opts = *opts;
    const OptionsScope scope(c);
    resolve_options(c, n);
    c->factored = false;
    c->allow_early = false;  // factor and solve are separate calls here: nothing could redo an early-scale overflow
    const int rc = factor_impl(c, n, dA, lda);
    c->allow_early = true;
    return rc;
}

int mplu_solve_device(mplu_context* c, const double* dA, long long lda, const double* db, double* dx,
                      mplu_stats* stats) {
    if (!c || !dA || !db || !dx) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    if (stats) memset(stats, 0, sizeof(*stats));
    return solve_impl(c, dA, lda, RhsBlock{1, db, c->n, dx, c->n, nullptr}, stats);
}

int mplu_gesv_device(mplu_context* c, int n, const double* dA, long long lda, const double* db, double* dx,
                     const mplu_options* opts, mplu_stats* stats) {
    if (!c || !dA || !db || !dx || n <= 0 || lda < n || !options_valid(opts)) return MPLU_E_ARG;
    return gesv_device_impl(c, n, dA, lda, RhsBlock{1, db, n, dx, n, nullptr}, opts, stats);
}

int mplu_gesv_host(mplu_context* c, int n, const double* hA, long long lda, const double* hb, double* hx,
                   const mplu_options* opts, mplu_stats* stats) {
    if (!c || !hA || !hb || !hx || n <= 0 || lda < n || !options_valid(opts)) return MPLU_E_ARG;
    return gesv_host_impl(c, n, hA, lda, RhsBlock{1, hb, n, hx, n, nullptr}, opts, stats);
}

int mplu_solve_device_nrhs(mplu_context* c, int nrhs, const double* dA, long long lda, const double* dB, long long ldb,
                           double* dX, long long ldx, double* berr, mplu_stats* stats) {
    if (!c || !dA || !dB || !dX || nrhs < 1 || lda < c->n || ldb < c->n || ldx < c->n) return MPLU_E_ARG;
    if (columns_overlap(dB, ldb, dX, ldx, c->n, nrhs)) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    if (stats) memset(stats, 0, sizeof(*stats));
    return solve_impl(c, dA, lda, RhsBlock{nrhs, dB, ldb, dX, ldx, berr}, stats);
}

int mplu_gesv_device_nrhs(mplu_context* c, int n, int nrhs, const double* dA, long long lda, const double* dB, long long ldb,
                          double* dX, long long ldx, const mplu_options* opts, double* berr, mplu_stats* stats) {
    if (!c || !dA || !dB || !dX || n <= 0 || nrhs < 1 || lda < n || ldb < n || ldx < n || !options_valid(opts)) return MPLU_E_ARG;
    if (columns_overlap(dB, ldb, dX, ldx, n, nrhs)) return MPLU_E_ARG;
    return gesv_device_impl(c, n, dA, lda, RhsBlock{nrhs, dB, ldb, dX, ldx, berr}, opts, stats);
}

int mplu_gesv_host_nrhs(mplu_context* c, int n, int nrhs, const double* hA, long long lda, const double* hB, long long ldb,
                        double* hX, long long ldx, const mplu_options* opts, double* berr, mplu_stats* stats) {
    if (!c || !hA || !hB || !hX || n <= 0 || nrhs < 1 || lda < n || ldb < n || ldx < n || !options_valid(opts)) return MPLU_E_ARG;
    if (columns_overlap(hB, ldb, hX, ldx, n, nrhs)) return MPLU_E_ARG;
    return gesv_host_impl(c, n, hA, lda, RhsBlock{nrhs, hB, ldb, hX, ldx, berr}, opts, stats);
}

int mplu_get_factors(mplu_context* c, double* LU, long long ldlu, int on_device) {
    if (!c || !LU || !c->factored || ldlu < c->n) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    const int n = c->n;
    double* dst = LU;
    double* tmp = nullptr;
    if (!on_device) {
        CK(cudaMalloc(&tmp, (size_t)n * n * sizeof(double)));
        dst = tmp;
    }
    dim3 grid((n + 255) / 256, n < 32768 ? n : 32768);  // gridDim.y <= 65535: columns on a grid-stride loop
    widen_kernel<<<grid, 256, 0, c->stream>>>(c->W, c->npad, n, dst, on_device ? ldlu : n);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && !on_device)
        e = cudaMemcpy2DAsync(LU, (size_t)ldlu * sizeof(double), tmp, (size_t)n * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (tmp) cudaFree(tmp);
    return (int)e;
}

int mplu_get_equilibration(mplu_context* c, int* equed, double* r, double* cs, int on_device) {
    if (!c) return MPLU_E_ARG;
    if (!c->factored) return MPLU_E_NOTFACTORED;
    CK(cudaSetDevice(c->device));
    const int n = c->n;
    if (equed) *equed = c->equed;
    const std::vector<double> ones(c->equed ? 0 : (size_t)n, 1.0);  // no scale applied: r = c = 1
    const cudaMemcpyKind kind = on_device ? (c->equed ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice)
                                          : (c->equed ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost);
    const double* src[2] = {c->equed ? c->eq_r : ones.data(), c->equed ? c->eq_c : ones.data()};
    double* dst[2] = {r, cs};
    for (int i = 0; i < 2; ++i)
        if (dst[i]) CK(cudaMemcpyAsync(dst[i], src[i], (size_t)n * sizeof(double), kind, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------ kernel hooks
int mplu_gemm16(int variant, int bf16, int M, int N, int K, float alpha, const void* dA, long long lda,
                const void* dB, long long ldb, float beta, float* dC, long long ldc, void* dH, long long ldh,
                float hscale, int max_sms, void* stream) {
    if (M <= 0 || N <= 0 || K <= 0 || K % 64 != 0 || !dA || !dB) return MPLU_E_ARG;
    if (beta != 0.f && beta != 1.f) return MPLU_E_ARG;
    if (gemm_tc_init() != 0) return MPLU_E_TMAP;
    uint32_t abr, abc, bbr, bbc;
    gemm_box_shapes(variant, &abr, &abc, &bbr, &bbc);
    const bool amn = (variant == GEMM_CG1_AMN || variant == GEMM_CG2_AMN);
    CUtensorMap tA, tB;
    if (amn) { if (make_tmap_16bit(&tA, dA, M, K, lda, abr, abc)) return MPLU_E_TMAP; }
    else     { if (make_tmap_16bit(&tA, dA, K, M, lda, abr, abc)) return MPLU_E_TMAP; }
    if (make_tmap_16bit(&tB, dB, K, N, ldb, bbr, bbc)) return MPLU_E_TMAP;
    GemmParams p{};
    p.M = M; p.N = N; p.K = K;
    p.C = dC; p.ldc = ldc;
    p.Cin = (beta == 1.f) ? dC : nullptr; p.ldcin = ldc;
    p.H = dH; p.ldh = ldh; p.h_rows = M; p.h_cols = N;
    p.alpha = alpha; p.hscale = hscale; p.bf16 = bf16;
    return launch_gemm_tc(variant, &tA, &tB, p, max_sms, (cudaStream_t)stream);
}

int mplu_diag_lu128(float* dW, long long ldw, float* dLinv, float* dUinv, void* stream) {
    if (!dW || !dLinv || !dUinv) return MPLU_E_ARG;
    CKI(panel_init());
    uint16_t* tmp16 = nullptr;
    float* sc = nullptr;
    int rc = (int)cudaMalloc(&tmp16, 2 * 128 * 128 * sizeof(uint16_t));
    if (!rc) rc = (int)cudaMalloc(&sc, 4 * sizeof(float));
    // the kernel stores triangles only
    if (!rc) rc = (int)cudaMemsetAsync(dLinv, 0, 128 * 128 * sizeof(float), (cudaStream_t)stream);
    if (!rc) rc = (int)cudaMemsetAsync(dUinv, 0, 128 * 128 * sizeof(float), (cudaStream_t)stream);
    if (!rc) rc = launch_diag_lu(dW, ldw, 0, tmp16, tmp16 + 128 * 128, 128, dLinv, dUinv, sc, 1, 0, 0, nullptr,
                                 (cudaStream_t)stream);
    cudaStreamSynchronize((cudaStream_t)stream);
    cudaFree(tmp16);
    cudaFree(sc);
    return rc;
}

// development aid: same as mplu_diag_lu128 with clock64() stamps of the kernel's phases written to d_clocks[0..31]
int mplu_diag_lu128_timed(float* dW, long long ldw, float* dLinv, float* dUinv, long long* d_clocks, void* stream) {
    if (!dW || !dLinv || !dUinv) return MPLU_E_ARG;
    CKI(panel_init());
    uint16_t* tmp16 = nullptr;
    float* sc = nullptr;
    int rc = (int)cudaMalloc(&tmp16, 2 * 128 * 128 * sizeof(uint16_t));
    if (!rc) rc = (int)cudaMalloc(&sc, 4 * sizeof(float));
    if (!rc) rc = launch_diag_lu(dW, ldw, 0, tmp16, tmp16 + 128 * 128, 128, dLinv, dUinv, sc, 1, 0, 0, nullptr,
                                 (cudaStream_t)stream, d_clocks);
    cudaStreamSynchronize((cudaStream_t)stream);
    cudaFree(tmp16);
    cudaFree(sc);
    return rc;
}

// development aid: `reps` dependent launches of one GEMM shape (C += alpha*A*B, optional shadow) captured into a CUDA
// graph and replayed; returns the average device time per launch in microseconds through *us_per_launch.
int mplu_bench_gemm_chain(int variant, int M, int N, int K, int reps, int pdl, int shadow, int accumulate,
                          int max_sms, float* us_per_launch) {
    if (M <= 0 || N <= 0 || K <= 0 || K % 64 || reps <= 0 || !us_per_launch) return MPLU_E_ARG;
    if (gemm_tc_init() != 0) return MPLU_E_TMAP;
    uint16_t *A = nullptr, *B = nullptr, *H = nullptr;
    float* Cm = nullptr;
    cudaStream_t st = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto body = [&]() -> int {  // every exit path goes through the clean-up below
        CK(cudaMalloc(&A, (size_t)M * K * 2)); CK(cudaMalloc(&B, (size_t)K * N * 2));
        CK(cudaMalloc(&H, (size_t)M * N * 2)); CK(cudaMalloc(&Cm, (size_t)M * N * 4));
        CK(cudaMemset(A, 0, (size_t)M * K * 2)); CK(cudaMemset(B, 0, (size_t)K * N * 2));
        CK(cudaMemset(Cm, 0, (size_t)M * N * 4));
        uint32_t abr, abc, bbr, bbc;
        gemm_box_shapes(variant, &abr, &abc, &bbr, &bbc);
        CUtensorMap tA, tB;
        if (make_tmap_16bit(&tA, A, M, K, M, abr, abc)) return MPLU_E_TMAP;
        if (make_tmap_16bit(&tB, B, K, N, K, bbr, bbc)) return MPLU_E_TMAP;
        GemmParams p{};
        p.M = M; p.N = N; p.K = K; p.C = Cm; p.ldc = M; p.Cin = accumulate ? Cm : nullptr; p.ldcin = M;
        p.H = shadow ? H : nullptr; p.ldh = M; p.h_rows = M; p.h_cols = N; p.alpha = -1.f; p.hscale = 1.f; p.pdl = pdl;
        CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
        int rc = 0;
        for (int i = 0; i < reps && !rc; ++i) rc = launch_gemm_tc(variant, &tA, &tB, p, max_sms, st);
        CK(cudaStreamEndCapture(st, &graph));
        if (rc) return rc;
        CK(cudaGraphInstantiate(&exec, graph, 0));
        CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
        CK(cudaGraphLaunch(exec, st));
        CK(cudaEventRecord(e0, st));
        CK(cudaGraphLaunch(exec, st));
        CK(cudaEventRecord(e1, st));
        CK(cudaStreamSynchronize(st));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        *us_per_launch = 1e3f * ms / reps;
        return 0;
    };
    const int rc = body();
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (st) cudaStreamDestroy(st);
    cudaFree(A); cudaFree(B); cudaFree(H); cudaFree(Cm);
    return rc;
}

// Dry run of the device factorization schedule for an n x n matrix (host logic only, no device needed): what would be
// launched on which lane, which array regions each launch reads / writes, and every cross-lane event record / wait.
// Serialised as ints: per op  kind, stream, event, group, nregions, then nregions x (array, r0, r1, c0, c1, write).
// Returns the number of ints the full trace needs (at most `max` are written).
int mplu_debug_trace(int n, int nb, const mplu_options* opts, int* out, int max) {
    if (n <= 0) return MPLU_E_ARG;
    mplu_context* c = new (std::nothrow) mplu_context();
    if (!c) return MPLU_E_ARG;
    if (opts) c->opts = *opts; else mplu_default_options(&c->opts);
    c->opts.nb = nb;
    c->opts.tile_ws = 0;
    resolve_options(c, n);
    c->n = n;
    c->npad = ((n + kDiagBlock - 1) / kDiagBlock) * kDiagBlock;
    c->cap_npad = c->npad;
    c->cap_nb = effective_nb(c, c->npad);
    c->num_sms = 148;
    // fake, never dereferenced: distinct address ranges so that a pointer identifies its array
    c->W = reinterpret_cast<float*>(1ull << 44);
    c->Wh = reinterpret_cast<uint16_t*>(2ull << 44);
    c->Fh = reinterpret_cast<uint16_t*>(3ull << 44);
    c->Linv16 = reinterpret_cast<uint16_t*>(4ull << 44);
    c->Uinv16 = reinterpret_cast<uint16_t*>(5ull << 44);
    c->Tb1 = reinterpret_cast<uint16_t*>(6ull << 44);
    c->Tb2 = reinterpret_cast<uint16_t*>(7ull << 44);
    c->scales = reinterpret_cast<float*>(8ull << 44);
    c->inv_scales = reinterpret_cast<float*>(9ull << 44);
    c->stream = reinterpret_cast<cudaStream_t>(1);
    c->side = reinterpret_cast<cudaStream_t>(2);
    c->ev_fork = reinterpret_cast<cudaEvent_t>(900000);
    c->ev_join = reinterpret_cast<cudaEvent_t>(900001);
    std::vector<TraceOp> tr;
    c->trace = &tr;
    const int rc = c->opts.schedule == MPLU_SCHED_LEFT ? enqueue_factorization_left(c) : enqueue_factorization(c);
    delete c;
    if (rc) return rc < 0 ? rc : -rc;
    long long pos = 0;
    auto put = [&](int v) { if (out && pos < max) out[pos] = v; ++pos; };
    for (const TraceOp& op : tr) {
        put(op.kind); put(op.stream); put(op.ev); put(op.group); put((int)op.regs.size());
        for (const TraceRegion& r : op.regs) { put(r.arr); put(r.r0); put(r.r1); put(r.c0); put(r.c1); put(r.write); }
    }
    return (int)pos;
}

int mplu_device_alloc(void** ptr, unsigned long long bytes) {
    if (!ptr) return MPLU_E_ARG;
    CK(cudaMalloc(ptr, (size_t)bytes));
    return 0;
}
int mplu_device_free(void* ptr) {
    CK(cudaFree(ptr));
    return 0;
}
int mplu_device_to_host(void* dst, const void* src, unsigned long long bytes) {
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost));
    return 0;
}

// sizes of the interface structs, so that a binding (ctypes, cgo, JNI) can check its mirror of include/mplu.h
int mplu_sizeof_options(void) { return (int)sizeof(mplu_options); }
int mplu_sizeof_stats(void) { return (int)sizeof(mplu_stats); }

// The left-looking schedule's bulk-lane plan for an n x n matrix tiled by nb (host logic only, no device needed):
// (step, k, m0, m1, mandatory) quintuples into out[0 .. 5*max); returns the number of ops.
// boundaries of the left-looking schedule's block columns for (n, nb, edge_nb); returns their count (tiles + 1)
int mplu_debug_tile_bounds(int n, int nb, int edge, int* out, int max) {
    if (n <= 0 || nb < kDiagBlock) return MPLU_E_ARG;
    const int npad = ((n + kDiagBlock - 1) / kDiagBlock) * kDiagBlock;
    nb = (nb / kDiagBlock) * kDiagBlock;
    const std::vector<int> tb = tile_bounds(npad, nb > npad ? npad : nb, edge);
    if (out && (int)tb.size() <= max) for (size_t i = 0; i < tb.size(); ++i) out[i] = tb[i];
    return (int)tb.size();
}
// the plan for those boundaries (5 ints per op: step, k, m0, m1, mandatory)
// eager: bit 0 = eager updates, bit 1 = paired updates (an op with kn = 2 is reported as its two updates k and k+1)
int mplu_debug_plan_left_edge(int n, int nb, int edge, int eager, int* out, int max) {
    if (n <= 0 || nb < kDiagBlock) return MPLU_E_ARG;
    const int npad = ((n + kDiagBlock - 1) / kDiagBlock) * kDiagBlock;
    nb = (nb / kDiagBlock) * kDiagBlock;
    std::vector<LeftOp> ops;
    for (const LeftOp& o : plan_left(tile_bounds(npad, nb > npad ? npad : nb, edge), (eager & 1) != 0, (eager & 2) != 0))
        for (int i = 0; i < o.kn; ++i) ops.push_back({o.step, o.k + i, o.m0, o.m1, o.mandatory, 1});
    if (out && (int)ops.size() <= max)
        for (size_t i = 0; i < ops.size(); ++i) {
            out[5 * i] = ops[i].step; out[5 * i + 1] = ops[i].k; out[5 * i + 2] = ops[i].m0; out[5 * i + 3] = ops[i].m1; out[5 * i + 4] = ops[i].mandatory;
        }
    return (int)ops.size();
}

int mplu_debug_plan_left(int n, int nb, int eager, int* out, int max) {
    if (n <= 0 || nb < kDiagBlock || nb % kDiagBlock) return MPLU_E_ARG;
    const int npad = ((n + kDiagBlock - 1) / kDiagBlock) * kDiagBlock;
    const std::vector<LeftOp> ops = plan_left(tile_bounds(npad, nb > npad ? npad : nb, 0), eager != 0);
    for (size_t i = 0; i < ops.size() && (int)i < max && out; ++i) {
        out[5 * i] = ops[i].step; out[5 * i + 1] = ops[i].k; out[5 * i + 2] = ops[i].m0; out[5 * i + 3] = ops[i].m1;
        out[5 * i + 4] = ops[i].mandatory;
    }
    return (int)ops.size();
}

// development aid: switch timeline marks on (takes effect at the next schedule capture) / read them back as
// (tag, milliseconds since the first mark) pairs after a synchronised factorization.  Returns the number of marks.
void mplu_debug_marks_enable(mplu_context* c, int on) {
    if (!c) return;
    c->marks_on = on != 0;
    if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
}
int mplu_debug_timeline(mplu_context* c, int* tags, float* ms, int max) {
    if (!c || !tags || !ms) return 0;
    cudaStreamSynchronize(c->stream);
    int n = c->mark_count < max ? c->mark_count : max;
    for (int i = 0; i < n; ++i) {
        tags[i] = c->mark_tag[i];
        ms[i] = 0.f;
        cudaEventElapsedTime(&ms[i], c->mark_ev[0], c->mark_ev[i]);
    }
    return n;
}

// test hook: the fp32 inverses of the unit-lower / upper factor of diagonal 128-block `blk` (column-major 128 x 128 each,
// device or host destination) as the triangular solves use them
int mplu_debug_block_inverses(mplu_context* c, int blk, float* Linv, float* Uinv) {
    if (!c || !c->factored || blk < 0 || blk >= c->npad / kDiagBlock || !Linv || !Uinv) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    const size_t bytes = (size_t)kDiagBlock * kDiagBlock * sizeof(float);
    CK(cudaMemcpy(Linv, c->Linv32 + (size_t)blk * kDiagBlock * kDiagBlock, bytes, cudaMemcpyDefault));
    CK(cudaMemcpy(Uinv, c->Uinv32 + (size_t)blk * kDiagBlock * kDiagBlock, bytes, cudaMemcpyDefault));
    return 0;
}

// development aid: per-step time stamps of the fused GETRF launches.  enable: takes effect at the next schedule capture.
// mplu_debug_fused_profile: for fused launch `launch` of the last factorization writes, per step, (kind, tiles, K of the
// first product | leaf origin, clock64 at the step's head) as 4 long longs, then one record (-1, 0, ns of the whole
// launch by %globaltimer, clock64 at the end).  Returns the number of records, 0 if that launch was not profiled.
int mplu_debug_fused_profile_enable(mplu_context* c, int on) {
    if (!c) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    c->fprof_on = on != 0;
    c->fprof_sub = on > 1;
    if (c->fprof_on && !c->fprof && c->fbar_cap > 0)
        CK(cudaMalloc(&c->fprof, (size_t)c->fbar_cap * mplu_context::kFusedProfSlots * sizeof(long long)));
    if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
    return 0;
}
int mplu_debug_fused_profile(mplu_context* c, int launch, long long* out, int max_records) {
    if (!c || !out || !c->fprof || launch < 0 || launch >= (int)c->fprof_prog.size() || c->fprof_prog[launch] < 0) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    const mplu_context::FusedProg& fp = c->fprogs[c->fprof_prog[launch]];
    std::vector<long long> clk(mplu_context::kFusedProfSlots);
    if (cudaMemcpy(clk.data(), c->fprof + (size_t)launch * mplu_context::kFusedProfSlots, clk.size() * sizeof(long long),
                   cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    const FusedStep* steps = reinterpret_cast<const FusedStep*>(c->fprog_host.data() + fp.offset);
    const FusedProblem* probs = reinterpret_cast<const FusedProblem*>(c->fprog_host.data() + fp.offset + fp.num_steps * sizeof(FusedStep));
    int nrec = 0;
    for (int s = 0; s < fp.num_steps && nrec < max_records; ++s, ++nrec) {
        const FusedStep& st = steps[s];
        out[4 * nrec] = st.kind;
        out[4 * nrec + 1] = st.kind == FS_GEMM ? st.tile_end[st.num_problems - 1] : 1;
        out[4 * nrec + 2] = st.kind == FS_GEMM ? probs[st.first_problem].K : st.k0;
        out[4 * nrec + 3] = clk[s];
        if (s < 61 && st.kind == FS_GEMM && c->fprof_sub) {  // sub-stamps relative to the step's head, packed into field 1
            const long long t0 = clk[s];
            auto rel = [&](int i) { long long d = clk[64 + 3 * s + i] - t0; return d < 0 ? 0 : (d > 0xFFFFF ? 0xFFFFF : d); };
            out[4 * nrec + 1] |= (rel(0) << 20) | (rel(1) << 40);
            out[4 * nrec + 2] |= rel(2) << 20;
        }
    }
    for (int i = 0; i < 48 && nrec < max_records; ++i, ++nrec) {  // phase stamps of one leaf of the launch (CTA 0's clock)
        out[4 * nrec] = -2; out[4 * nrec + 1] = i; out[4 * nrec + 2] = 0; out[4 * nrec + 3] = clk[300 + i];
    }
    if (nrec < max_records) {
        out[4 * nrec] = -1; out[4 * nrec + 1] = 0;
        out[4 * nrec + 2] = clk[fp.num_steps + 2] - clk[fp.num_steps + 1];
        out[4 * nrec + 3] = clk[fp.num_steps];
        ++nrec;
    }
    return nrec;
}

// the raw time-stamp slots of fused launch `launch` (layout: see getrf_fused.cu / tools/fused_profile.py)
// Development aid: %globaltimer stamps of the `launch`-th dataflow GETRF launch of the following factorizations
// (launch < 0: off).  Takes effect at the next schedule capture.
int mplu_debug_flow_profile_enable(mplu_context* c, int launch) {
    if (!c) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    if (launch >= 0 && !c->flow_prof) {
        c->flow_prof_cap = (size_t)8 << 20;
        CK(cudaMalloc(&c->flow_prof, c->flow_prof_cap));
    }
    if (c->flow_prof) CK(cudaMemset(c->flow_prof, 0, c->flow_prof_cap));
    c->flow_prof_launch = launch;
    return 0;
}
// After a synchronised factorization: stamps[0 .. 2 L) = (start, end) of the L leaves, then per task (taken from the list,
// dependencies met, result signalled, CTA); tasks_out receives the 32-byte task records.  Returns the task count (< 0: error).
int mplu_debug_flow_profile(mplu_context* c, long long* stamps, int max_stamps, unsigned char* tasks_out, int max_task_bytes,
                            int* num_leaves) {
    if (!c || !c->flow_prof || c->flow_prof_prog < 0 || c->flow_prof_prog >= (int)c->flow_progs.size()) return MPLU_E_ARG;
    CK(cudaSetDevice(c->device));
    const mplu_context::FlowProg& fp = c->flow_progs[c->flow_prof_prog];
    const int ns = 2 * fp.num_leaves + 4 * fp.num_tasks;
    if (ns > max_stamps || fp.num_tasks * (int)sizeof(FlowTask) > max_task_bytes) return MPLU_E_ARG;
    CK(cudaMemcpy(stamps, c->flow_prof, (size_t)ns * sizeof(long long), cudaMemcpyDeviceToHost));
    memcpy(tasks_out, c->flow_host.data() + fp.off_tasks, (size_t)fp.num_tasks * sizeof(FlowTask));
    *num_leaves = fp.num_leaves;
    return fp.num_tasks;
}

int mplu_debug_fused_raw(mplu_context* c, int launch, long long* out, int max_slots) {
    if (!c || !out || !c->fprof || launch < 0 || launch >= c->fbar_cap) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    const int k = max_slots < mplu_context::kFusedProfSlots ? max_slots : mplu_context::kFusedProfSlots;
    if (cudaMemcpy(out, c->fprof + (size_t)launch * mplu_context::kFusedProfSlots, (size_t)k * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess)
        return 0;
    return k;
}

int mplu_residual(int n, const double* dA, long long lda, const double* dx, const double* db, double* dr,
                  double* dnorms, void* stream) {
    if (n <= 0 || !dA || !dx || !db || !dr || !dnorms) return MPLU_E_ARG;
    double* partial = nullptr;
    const int nchunk = 64;
    CK(cudaMalloc(&partial, (size_t)nchunk * n * sizeof(double)));
    int rc = launch_residual(dA, lda, n, dx, db, dr, partial, nchunk, dnorms, (cudaStream_t)stream);
    cudaStreamSynchronize((cudaStream_t)stream);
    cudaFree(partial);
    return rc;
}

}  // extern "C"
