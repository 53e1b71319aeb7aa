// GMRES-based iterative refinement (SURVEY.md section 8f item 3; Carson & Higham's GMRES-IR): the correction equation
// A d = r of each refinement step is solved by GMRES in fp64, left-preconditioned with the low-precision factors,
//     M^-1 A d = M^-1 r,   M^-1 = (LU)^-1, or C (LU)^-1 R with equilibrated factors of diag(r) A diag(c),
// instead of the single solve d = (LU)^-1 r of classic refinement.  The preconditioned operator is applied with the
// kernels the classic path already has (fp64 A*v: residual kernels; (LU)^-1: lu_solve_kernel on the fp32 factors), so
// this file only adds the Krylov bookkeeping: classical Gram-Schmidt with re-orthogonalisation on the device (two
// tall-skinny products per pass), Givens rotations of the small Hessenberg matrix on the host.
// The reference has no solve path at all; this is what makes BASELINE.json's condition-number sweep reach 1e7..1e8,
// where classic refinement with 16-bit factors stagnates (tools/kappa_sweep.py).
#include "lu_internal.h"

#include <cmath>
#include <vector>

using namespace mplu;
using namespace mplu_detail;

namespace {

// h[i] += sum_r V[r + i*n] * w[r]   i < k     grid (k, chunks), block 256
__global__ void vt_w_kernel(const double* __restrict__ V, const double* __restrict__ w, int n, double* h) {
    const int i = blockIdx.x;
    const double* v = V + (size_t)i * n;
    double s = 0.0;
    for (int r = blockIdx.y * blockDim.x + threadIdx.x; r < n; r += gridDim.y * blockDim.x) s = fma(v[r], w[r], s);
    __shared__ double sm[8];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int q = 0; q < (int)(blockDim.x >> 5); ++q) t += sm[q];
        atomicAdd(h + i, t);
    }
}
// out[r] = beta*w[r] + alpha * sum_i V[r + i*n] * h[i]    (out may alias w)
__global__ void v_h_kernel(const double* __restrict__ V, const double* __restrict__ h, int k, int n, double alpha,
                           double beta, const double* w, double* out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    double s = 0.0;
    for (int i = 0; i < k; ++i) s = fma(V[r + (size_t)i * n], h[i], s);
    out[r] = (beta != 0.0 ? beta * w[r] : 0.0) + alpha * s;
}
__global__ void scale_to_kernel(const double* __restrict__ w, double a, double* out, int n) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) out[r] = a * w[r];
}

}  // namespace

namespace mplu_detail {

// out = M^-1 in for the preconditioner M^-1 = C (LU)^-1 R of the stored factors (R, C: the equilibration's scales where
// applied, identity otherwise; eq_D is the scratch of the scaled right-hand side)
int apply_preconditioner(mplu_context* c, const double* in, double* out) {
    const int n = c->n;
    cudaStream_t st = c->stream;
    const double* rhs = in;
    if (c->equed & 1) {
        CKI(launch_diag_scale(c->eq_r, n, 1, in, n, c->eq_D, n, 0, st));
        rhs = c->eq_D;
        c->kernel_launches += 1;
    }
    CKI(launch_lu_solve(c->W, c->npad, n, c->npad, c->Linv32, c->Uinv32, rhs, c->y, out, nullptr, c->ready, st));
    if (c->equed & 2) {
        CKI(launch_diag_scale(c->eq_c, n, 1, out, n, out, n, 0, st));
        c->kernel_launches += 1;
    }
    return 0;
}

// One GMRES solve of A d = r (r: n doubles on the device), x += d.  Returns 0 or an error code; *inner = Krylov steps taken.
int gmres_correction(mplu_context* c, const double* dA, long long lda, const double* r, double* dx, int* inner) {
    const int n = c->n;
    cudaStream_t st = c->stream;
    const int m = c->opts.gmres_restart > 0 ? c->opts.gmres_restart : 50;
    const double tol = c->opts.gmres_tol > 0 ? c->opts.gmres_tol : 1e-6;
    if (c->gm_cap_n < n || c->gm_cap_m < m) {
        cudaFree(c->gm_V); cudaFree(c->gm_w); cudaFree(c->gm_h); cudaFree(c->gm_zero);
        c->gm_V = c->gm_w = c->gm_h = c->gm_zero = nullptr;
        CK(cudaMalloc(&c->gm_V, (size_t)n * (m + 1) * sizeof(double)));
        CK(cudaMalloc(&c->gm_w, 2 * (size_t)n * sizeof(double)));
        CK(cudaMalloc(&c->gm_h, 2 * (size_t)(m + 2) * sizeof(double)));
        CK(cudaMalloc(&c->gm_zero, (size_t)n * sizeof(double)));
        CK(cudaMemset(c->gm_zero, 0, (size_t)n * sizeof(double)));
        c->gm_cap_n = n;
        c->gm_cap_m = m;
    }
    double* V = c->gm_V;
    double* w = c->gm_w;
    double* tmp = c->gm_w + n;
    double* dh = c->gm_h;
    const int nb256 = (n + 255) / 256;
    const int chunks = n >= 1 << 16 ? 16 : (n >= 1 << 13 ? 8 : 2);
    std::vector<double> H((size_t)(m + 1) * m, 0.0), cs(m, 0.0), sn(m, 0.0), g(m + 1, 0.0), hh(m + 2), h2(m + 2);

    auto dots = [&](const double* vec, int k, double* host) {  // host[0..k) = V[:, :k]^T vec, host[k] = vec^T vec
        if (cudaMemsetAsync(dh, 0, (k + 1) * sizeof(double), st) != cudaSuccess) return (int)cudaGetLastError();
        if (k > 0) vt_w_kernel<<<dim3(k, chunks), 256, 0, st>>>(V, vec, n, dh);
        vt_w_kernel<<<dim3(1, chunks), 256, 0, st>>>(vec, vec, n, dh + k);
        c->kernel_launches += 2;
        if (cudaMemcpyAsync(host, dh, (k + 1) * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess) return (int)cudaGetLastError();
        return (int)cudaStreamSynchronize(st);
    };

    // z0 = M^-1 r -> V[:,0]
    CKI(apply_preconditioner(c, r, w));
    CKI(dots(w, 0, hh.data()));
    const double beta = std::sqrt(hh[0]);
    *inner = 0;
    if (!(beta > 0.0) || !std::isfinite(beta)) return 0;
    scale_to_kernel<<<nb256, 256, 0, st>>>(w, 1.0 / beta, V, n);
    g[0] = beta;
    int k = 0;
    for (int j = 0; j < m; ++j) {
        // w = M^-1 (A v_j):  tmp = 0 - A v_j, w = -M^-1 tmp
        CKI(launch_residual(dA, lda, n, V + (size_t)j * n, c->gm_zero, tmp, c->partial, c->nchunk, c->norms, st));
        CKI(apply_preconditioner(c, tmp, w));
        scale_to_kernel<<<nb256, 256, 0, st>>>(w, -1.0, w, n);
        c->kernel_launches += 4;
        // classical Gram-Schmidt, twice
        CKI(dots(w, j + 1, hh.data()));
        CK(cudaMemcpyAsync(dh + m + 2, hh.data(), (j + 1) * sizeof(double), cudaMemcpyHostToDevice, st));
        v_h_kernel<<<nb256, 256, 0, st>>>(V, dh + m + 2, j + 1, n, -1.0, 1.0, w, w);
        CKI(dots(w, j + 1, h2.data()));
        CK(cudaMemcpyAsync(dh + m + 2, h2.data(), (j + 1) * sizeof(double), cudaMemcpyHostToDevice, st));
        v_h_kernel<<<nb256, 256, 0, st>>>(V, dh + m + 2, j + 1, n, -1.0, 1.0, w, w);
        double corr = 0.0;
        for (int i = 0; i <= j; ++i) { hh[i] += h2[i]; corr += h2[i] * h2[i]; }
        double hn2 = h2[j + 1] - corr;  // ||w||^2 after the second pass
        if (!(hn2 > 0.0)) hn2 = 0.0;
        const double hn = std::sqrt(hn2);
        c->kernel_launches += 2;
        // Hessenberg column j, previous rotations, new rotation
        for (int i = 0; i <= j; ++i) H[(size_t)j * (m + 1) + i] = hh[i];
        H[(size_t)j * (m + 1) + j + 1] = hn;
        double* col = &H[(size_t)j * (m + 1)];
        for (int i = 0; i < j; ++i) {
            const double t = cs[i] * col[i] + sn[i] * col[i + 1];
            col[i + 1] = -sn[i] * col[i] + cs[i] * col[i + 1];
            col[i] = t;
        }
        const double den = std::hypot(col[j], col[j + 1]);
        if (den == 0.0) { k = j; break; }
        cs[j] = col[j] / den;
        sn[j] = col[j + 1] / den;
        col[j] = den;
        col[j + 1] = 0.0;
        g[j + 1] = -sn[j] * g[j];
        g[j] = cs[j] * g[j];
        k = j + 1;
        if (hn > 0.0 && j + 1 < m + 1) scale_to_kernel<<<nb256, 256, 0, st>>>(w, 1.0 / hn, V + (size_t)(j + 1) * n, n);
        if (std::fabs(g[j + 1]) <= tol * beta || hn == 0.0) break;
    }
    *inner = k;
    if (k == 0) return 0;
    // back substitution H y = g, x += V y
    std::vector<double> y(k);
    for (int i = k - 1; i >= 0; --i) {
        double s = g[i];
        for (int q = i + 1; q < k; ++q) s -= H[(size_t)q * (m + 1) + i] * y[q];
        y[i] = s / H[(size_t)i * (m + 1) + i];
    }
    CK(cudaMemcpyAsync(dh + m + 2, y.data(), k * sizeof(double), cudaMemcpyHostToDevice, st));
    v_h_kernel<<<nb256, 256, 0, st>>>(V, dh + m + 2, k, n, 1.0, 1.0, dx, dx);
    c->kernel_launches += 1;
    return (int)cudaGetLastError();
}

}  // namespace mplu_detail
