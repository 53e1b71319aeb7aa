"""CPU oracle for the mixed-precision LU hot path -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module.
The product (libmplu.so) never calls it and has no CPU fallback.

What is restated here, with the reference lines each piece follows:

* glibc ``rand()`` stream + ``matrix_generator`` text format          matrix_generator.cpp:53-85
* ``double_to_fp16`` (via float, clamp +-65504, flush |x|<6.10352e-5)    fp16_utils.h:15-23
* ``HGETF2_kernel``: fp16 partial-pivot panel LU, first-max pivot       hgetf2_kernel.cu:22-119
* ``LASWP_kernel``: sequential row swaps on the whole fp64 matrix       MPF.cu:42-59
* ``dgetf2_native_npv``: fp64 no-pivot panel LU                         dgetf2_native_npv.cu:18-35
* ``MPF``: the panel loop incl. Dtrsm / Dgemm and the IPIV quirks       MPF.cu:100-241
* ``check_correctitude``: P*L*U == A to 1e-10                           benchmark.cpp:59-144

Pinning status.  The reference ships NO golden vectors (SURVEY.md section 4).  The oracle is pinned by
 (a) libc's real rand() (ctypes) for the generator, first 2x2 = 8.3 8.6 / 7.7 1.5           (tests/test_oracle.py)
 (b) host LAPACK dgetrf on column-dominant inputs: identity pivots, factors equal to 1e-12    (tests/test_oracle.py)
 (c) outputs of the UNMODIFIED reference built from /root/reference by oracle/Makefile and run on a B200 through
     oracle/make_golden.py; fixtures under tests/golden/ (tests/test_oracle.py, tests/test_gpu_mpf.py), and LIVE in the
     GPU tests through oracle/run_ref_mpf.py at n = 1024 / 4096 (tests/test_gpu_configs.py)
The iterative-refinement part has no reference counterpart at all: for it "parity unpinned" applies and the
comparator is host LAPACK dgetrs / dsgesv (SURVEY.md section 8c).
"""
from __future__ import annotations

import math

import numpy as np

U64 = np.uint64
FP16_MAX = np.float32(65504.0)
FP16_MIN_POS = np.float32(6.10352e-05)


# --------------------------------------------------------------------------------------------------------------
# generators
# --------------------------------------------------------------------------------------------------------------
class GlibcRand:
    """glibc TYPE_3 additive-feedback rand() with the default seed 1 (matrix_generator.cpp never calls srand)."""

    def __init__(self, seed: int = 1):
        r = [0] * 34
        r[0] = seed
        for i in range(1, 31):
            hi, lo = divmod(r[i - 1], 127773)
            word = 16807 * lo - 2836 * hi
            if word < 0:
                word += 2147483647
            r[i] = word
        for i in range(31, 34):
            r[i] = r[i - 31]
        self._r = r
        for _ in range(34, 344):
            self._step()

    def _step(self) -> int:
        r = self._r
        v = (r[-31] + r[-3]) & 0xFFFFFFFF
        r.append(v)
        if len(r) > 64:
            del r[:-34]
        return v

    def rand(self) -> int:
        return self._step() >> 1

    def fill(self, count: int) -> np.ndarray:
        """`count` successive rand() values (vectorised in blocks through the lag-31/lag-3 recurrence)."""
        out = np.empty(count, dtype=np.int64)
        for k in range(count):
            out[k] = self._step() >> 1
        return out


def matrix_generator_sizes(max_size: int, step: int = 2, func: str = "exp"):
    size, sizes = 2, []
    while size <= max_size:
        sizes.append(size)
        size = size * step if func == "exp" else size + step
    return sizes


def matrix_generator_stream(max_size: int, step: int = 2, func: str = "exp"):
    """Yield (n, M) for every matrix `matrix_generator file max_size step func` writes (dense, sparsity 0):
    M[i, j] is the j-th value on printed row i, value = (rand() % 100) / 10.0 (matrix_generator.cpp:60-67)."""
    g = GlibcRand()
    for n in matrix_generator_sizes(max_size, step, func):
        v = g.fill(n * n)
        yield n, ((v % 100) / 10.0).reshape(n, n)


def as_benchmark_reads(M_printed: np.ndarray) -> np.ndarray:
    """benchmark.cpp:192-194 reads the n*n values sequentially into a buffer it then treats as column-major
    (benchmark.cpp:19), so the matrix actually factored is the transpose of the printed one."""
    return np.ascontiguousarray(M_printed.T)


def splitmix64(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        x = (x + U64(0x9E3779B97F4A7C15)).astype(U64)
        z = x
        z = ((z ^ (z >> U64(30))) * U64(0xBF58476D1CE4E5B9)).astype(U64)
        z = ((z ^ (z >> U64(27))) * U64(0x94D049BB133111EB)).astype(U64)
        return z ^ (z >> U64(31))


def counter_matrix(n: int, seed: int = 1, dominant: bool = True, rows=None) -> np.ndarray:
    """Counter-based stand-in for the reference value distribution (values k/10, k = 0..99), usable at any size
    and on the device: a(i,j) = (splitmix64(seed<<40 | i<<20 | j) % 100) / 10.  With dominant=True the diagonal is
    replaced by the column's off-diagonal absolute sum + 1 (strict column diagonal dominance => partial pivoting
    selects the diagonal, SURVEY.md section 0).  Same formula as mplu_generate (csrc/generate.cu)."""
    i = np.arange(n, dtype=U64)[:, None]
    j = np.arange(n, dtype=U64)[None, :]
    key = (U64(seed) << U64(40)) | (i << U64(20)) | j
    K = (splitmix64(key) % U64(100)).astype(np.int64)
    A = K.astype(np.float64) / 10.0
    if dominant:
        off = K.sum(axis=0) - np.diag(K)  # exact integer tenths, so host and device agree bit for bit
        A[np.arange(n), np.arange(n)] = off.astype(np.float64) / 10.0 + 1.0
    return A


def spd_kappa_matrix(n: int, kappa: float, seed: int = 1) -> np.ndarray:
    """SPD test matrix H diag(sigma) H with one Householder reflector H = I - 2uu^T and geometric singular values
    in [1/kappa, 1] (config 5 of BASELINE.json; SURVEY.md section 8d)."""
    rng = np.random.default_rng(seed)
    u = rng.standard_normal(n)
    u /= np.linalg.norm(u)
    sigma = kappa ** (-np.arange(n) / max(n - 1, 1))
    H = np.eye(n) - 2.0 * np.outer(u, u)
    return (H * sigma) @ H


def counter_matrix_into(out: np.ndarray, seed: int = 1, dominant: bool = True, block: int = 512) -> np.ndarray:
    """counter_matrix(n, seed, dominant) written into the preallocated column-major n x n array `out` by column blocks
    (bounded temporaries: the full-size n = 32768 input of bench.py's reference arm is 8 GiB).  Uses torch's threaded
    CPU integer ops when torch is importable (same values bit for bit: tests/test_oracle.py), numpy otherwise."""
    n = out.shape[0]
    assert out.shape == (n, n) and out.dtype == np.float64 and out.flags.f_contiguous
    try:
        import torch
    except ImportError:
        torch = None
    if torch is None:
        i = np.arange(n, dtype=U64)[:, None]
        for c0 in range(0, n, block):
            c1 = min(n, c0 + block)
            j = np.arange(c0, c1, dtype=U64)[None, :]
            K = (splitmix64((U64(seed) << U64(40)) | (i << U64(20)) | j) % U64(100)).astype(np.int64)
            blk = K.astype(np.float64) / 10.0
            if dominant:
                d = np.arange(c0, c1)
                blk[d, d - c0] = (K.sum(axis=0) - K[d, d - c0]).astype(np.float64) / 10.0 + 1.0
            out[:, c0:c1] = blk
        return out

    def lsr(v, k):  # logical shift right on int64 bit patterns
        return (v >> k) & ((1 << (64 - k)) - 1)

    outT = torch.from_numpy(out.T)  # C-contiguous: outT[c, r] = A[r, c]
    i = torch.arange(n, dtype=torch.int64)[None, :]
    for c0 in range(0, n, block):
        c1 = min(n, c0 + block)
        j = torch.arange(c0, c1, dtype=torch.int64)[:, None]
        z = ((seed << 40) | (i << 20) | j) + (-7046029254386353131)   # + 0x9E3779B97F4A7C15 (mod 2^64)
        z = (z ^ lsr(z, 30)) * (-4658895280553007687)                 # * 0xBF58476D1CE4E5B9
        z = (z ^ lsr(z, 27)) * (-7723592293110705685)                 # * 0x94D049BB133111EB
        z = z ^ lsr(z, 31)
        K = ((lsr(z, 32) % 100) * (2 ** 32 % 100) + (z & 0xFFFFFFFF) % 100) % 100  # unsigned 64-bit value mod 100
        blk = K.to(torch.float64) / 10.0
        if dominant:
            d = torch.arange(c0, c1)
            blk[d - c0, d] = (K.sum(dim=1) - K[d - c0, d]).to(torch.float64) / 10.0 + 1.0
        outT[c0:c1] = blk
    return out


# --------------------------------------------------------------------------------------------------------------
# fp16 helpers
# --------------------------------------------------------------------------------------------------------------
def double_to_fp16(x: np.ndarray) -> np.ndarray:
    """fp16_utils.h:15-23: double -> float (RN) -> clamp to +-65504 -> flush |x| < 6.10352e-5 to 0 -> half (RN)."""
    xf = np.asarray(x, dtype=np.float64).astype(np.float32)
    xf = np.minimum(np.maximum(xf, -FP16_MAX), FP16_MAX)
    xf = np.where((xf > -FP16_MIN_POS) & (xf < FP16_MIN_POS), np.float32(0), xf)
    return xf.astype(np.float16)


def _h(x64):
    """round an exactly computed (float64) value to fp16 once"""
    with np.errstate(over="ignore"):
        return np.asarray(x64, dtype=np.float64).astype(np.float16)


def _hgetf2_tie_order(nmax: int = 1 << 20) -> np.ndarray:
    """rank of row offset rel = row - j in the reference's tie-break: (rel // 256, bitreverse8(rel % 256))"""
    rel = np.arange(nmax, dtype=np.int64)
    t = rel & 255
    rev = np.zeros_like(t)
    for b in range(8):
        rev |= ((t >> b) & 1) << (7 - b)
    return ((rel >> 8) << 8) | rev


_HGETF2_TIE_ORDER = _hgetf2_tie_order()


def hgetf2(panel: np.ndarray, fused: bool = True):
    """fp16 partial-pivot LU of a rows x cols panel (hgetf2_kernel.cu:22-119).  Returns (panel_out, ipiv) with
    ipiv 1-based panel-local.  Pivot = a row attaining max |a| over rows j..; among EQUAL maxima the reference's
    reductions (strict '>' in the 256-slot shared-memory tree, :48-56, then a linear scan over the blocks, :72-79) keep
    the lower slot at every merge, i.e. the winner is the tied row with the smallest (block, bit-reversed thread index)
    -- not the first row (found by the live-reference parity test on a tie-rich input).  NaN never wins.  Multiplier = fp16 division; update a -= m*b either fused (one rounding: what -O3
    emits, SURVEY.md section 3.3) or as two rounded fp16 operations (the reference's own -O0 build)."""
    P = np.array(panel, dtype=np.float16, copy=True)
    rows, cols = P.shape
    ipiv = np.zeros(cols, dtype=np.int32)
    for j in range(cols):
        if j >= rows:
            ipiv[j] = j + 1
            continue
        col = np.abs(P[j:, j].astype(np.float32))
        col = np.where(np.isnan(col), np.float32(-1), col)
        p = j
        if col.size and col.max() > 0:
            tied = np.flatnonzero(col == col.max())
            p = int(tied[np.argmin(_HGETF2_TIE_ORDER[tied])]) + j
        ipiv[j] = p + 1
        if p != j:
            P[[j, p], :] = P[[p, j], :]
        if j + 1 < rows:
            piv = np.float64(P[j, j])
            with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
                m = _h(P[j + 1:, j].astype(np.float64) / piv)
                P[j + 1:, j] = m
                if j + 1 < cols:
                    m64 = m.astype(np.float64)[:, None]
                    b64 = P[j, j + 1:].astype(np.float64)[None, :]
                    if fused:
                        P[j + 1:, j + 1:] = _h(P[j + 1:, j + 1:].astype(np.float64) - m64 * b64)
                    else:
                        prod = _h(m64 * b64)
                        P[j + 1:, j + 1:] = _h(P[j + 1:, j + 1:].astype(np.float64) - prod.astype(np.float64))
    return P, ipiv


def dgetf2_npv(panel: np.ndarray) -> np.ndarray:
    """fp64 no-pivot LU of an m x n panel, in the reference's operation order (dgetf2_native_npv.cu:18-35):
    multiplier = a[r,j] / a[j,j]; a[r,k] -= multiplier * a[j,k] (contracted to an FMA by nvcc, SURVEY.md 2.1)."""
    P = np.array(panel, dtype=np.float64, copy=True)
    m, n = P.shape
    for j in range(min(n, m)):
        if j + 1 < m:
            P[j + 1:, j] = P[j + 1:, j] / P[j, j]
            if j + 1 < n:
                P[j + 1:, j + 1:] -= np.outer(P[j + 1:, j], P[j, j + 1:])
    return P


def mpf_reference(A: np.ndarray, r: int = 32, fused: bool = True):
    """The reference MPF(A, N, r, IPIV) restated (MPF.cu:100-241).  A is the column-major matrix as a 2-D array
    A[row, col].  Returns (LU, IPIV) with IPIV pre-filled with i+1 as benchmark.cpp:215-217 does, so the entry MPF
    never writes when the last panel is a single row (MPF.cu:104) keeps its identity value."""
    A = np.array(A, dtype=np.float64, copy=True)
    N = A.shape[0]
    ipiv = np.arange(1, N + 1, dtype=np.int32)
    for k in range(0, N, r):
        pc = min(r, N - k)
        pr = N - k
        if pr <= 1:
            continue
        _, ip = hgetf2(double_to_fp16(A[k:, k:k + pc]), fused=fused)
        gp = ip + k
        ipiv[k:k + pc] = gp
        for j in range(pc):  # LASWP over all N columns (MPF.cu:42-59)
            cur, piv = k + j, gp[j] - 1
            if piv != cur:
                A[[cur, piv], :] = A[[piv, cur], :]
        A[k:, k:k + pc] = dgetf2_npv(A[k:, k:k + pc])
        if k + pc < N:
            L11 = np.tril(A[k:k + pc, k:k + pc], -1) + np.eye(pc)
            A[k:k + pc, k + pc:] = np.linalg.solve(L11, A[k:k + pc, k + pc:])  # Dtrsm unit-lower (MPF.cu:215)
            A[k + pc:, k + pc:] -= A[k + pc:, k:k + pc] @ A[k:k + pc, k + pc:]  # Dgemm (MPF.cu:230)
    return A, ipiv


def check_correctitude(A: np.ndarray, LU: np.ndarray, ipiv: np.ndarray, tol: float = 1e-10) -> bool:
    """benchmark.cpp:59-144: P*(L*U) == A element-wise to `tol`, swaps applied for i = n-1 .. 0."""
    n = A.shape[0]
    L = np.tril(LU, -1) + np.eye(n)
    U = np.triu(LU)
    PLU = L @ U
    for i in range(n - 1, -1, -1):
        p = int(ipiv[i]) - 1
        if p != i:
            PLU[[i, p], :] = PLU[[p, i], :]
    return bool(np.all(np.abs(A - PLU) <= tol))


# --------------------------------------------------------------------------------------------------------------
# the north_star algorithm: no-pivot blocked LU in 16-bit with fp32 accumulation + fp64 refinement
# --------------------------------------------------------------------------------------------------------------
def lu_nopivot_fp64(A: np.ndarray, nb: int = 128) -> np.ndarray:
    """Exact-arithmetic target of the low-precision factorization: blocked no-pivot LU in fp64."""
    A = np.array(A, dtype=np.float64, copy=True)
    n = A.shape[0]
    for k in range(0, n, nb):
        e = min(n, k + nb)
        A[k:, k:e] = dgetf2_npv(A[k:, k:e])
        if e < n:
            L11 = np.tril(A[k:e, k:e], -1) + np.eye(e - k)
            A[k:e, e:] = np.linalg.solve(L11, A[k:e, e:])
            A[e:, e:] -= A[e:, k:e] @ A[k:e, e:]
    return A


def round16(x: np.ndarray, bf16: bool = False) -> np.ndarray:
    x = np.asarray(x, dtype=np.float32)
    if not bf16:
        with np.errstate(over="ignore"):
            return x.astype(np.float16).astype(np.float32)
    u = x.view(np.uint32).astype(np.uint64)
    u = (u + U64(0x7FFF) + ((u >> U64(16)) & U64(1))) & U64(0xFFFF0000)
    return u.astype(np.uint32).view(np.float32)


def lu_mixed_emulated(A: np.ndarray, nb: int = 128, bf16: bool = False, a_exp: int = 11, l_exp: int = 11):
    """Emulation of the device algorithm's rounding model: panels in fp32, every GEMM operand rounded to the 16-bit
    type after power-of-two scaling, products accumulated in fp32 (numpy float32 matmul), factors stored in fp32.
    Not bit-identical to tensor-core accumulation order; used for tolerance calibration and iteration counts."""
    W = np.array(A, dtype=np.float64).astype(np.float32)
    n = W.shape[0]
    amax = float(np.abs(W).max())
    sA = np.float32(1.0) if bf16 or amax == 0 else np.float32(2.0 ** (a_exp - math.frexp(amax)[1]))
    sL = np.float32(1.0) if bf16 else np.float32(2.0 ** l_exp)
    for k in range(0, n, nb):
        e = min(n, k + nb)
        D = dgetf2_npv(W[k:e, k:e].astype(np.float64)).astype(np.float32)
        W[k:e, k:e] = D
        if e < n:
            L11 = (np.tril(D, -1) + np.eye(e - k)).astype(np.float64)
            U11 = np.triu(D).astype(np.float64)
            Linv = np.linalg.inv(L11).astype(np.float32)
            Uinv = np.linalg.inv(U11).astype(np.float32)
            sLi = np.float32(1.0) if bf16 else np.float32(2.0 ** (11 - math.frexp(float(np.abs(Linv).max()))[1]))
            sUi = np.float32(1.0) if bf16 else np.float32(2.0 ** (11 - math.frexp(float(np.abs(Uinv).max()))[1]))
            A21h = round16(W[e:, k:e] * sA, bf16)
            A12h = round16(W[k:e, e:] * sA, bf16)
            L21 = (A21h @ round16(Uinv * sUi, bf16)) / (sA * sUi)
            U12 = (round16(Linv * sLi, bf16) @ A12h) / (sA * sLi)
            W[e:, k:e] = L21
            W[k:e, e:] = U12
            W[e:, e:] -= (round16(L21 * sL, bf16) @ round16(U12 * sA, bf16)) / (sL * sA)
    return W


def lu_solve(LU: np.ndarray, b: np.ndarray, dtype=np.float32) -> np.ndarray:
    from scipy.linalg import solve_triangular
    LU = np.asarray(LU, dtype=dtype)
    y = solve_triangular(LU, np.asarray(b, dtype=dtype), lower=True, unit_diagonal=True, check_finite=False)
    return solve_triangular(LU, y, lower=False, check_finite=False)


def factor_tile_ratio(A, LU, tile: int = 128):
    """Componentwise backward error of a no-pivot factorization, tile by tile: with L = tril(LU,-1) + I, U = triu(LU),
    E = |L U - A| and M = |L| |U| (fp64), returns rho[I, J] = max E_IJ / max M_IJ over the tile x tile tiles (the last
    row / column of tiles is ragged when n is not a multiple of `tile`).  A tile whose M is all zero must have E = 0:
    its rho is 0 then, inf otherwise.  Unlike a bound relative to max|LU| (the diagonal, on dominant inputs) it does not
    let a wrong off-diagonal tile hide behind a large diagonal.  numpy arrays or torch tensors; CUDA tensors stay on the
    device and the result is a numpy array either way."""
    try:
        import torch
    except ImportError:
        torch = None
    if torch is not None and (isinstance(A, torch.Tensor) or isinstance(LU, torch.Tensor)):
        dev = LU.device if isinstance(LU, torch.Tensor) else A.device
        A = torch.as_tensor(A, dtype=torch.float64, device=dev)
        LU = torch.as_tensor(LU, dtype=torch.float64, device=dev)
        n = LU.shape[0]
        L = torch.tril(LU, -1) + torch.eye(n, dtype=torch.float64, device=dev)
        U = torch.triu(LU)
        E = (L @ U - A).abs()
        M = L.abs() @ U.abs()
        del L, U
        npad = -(-n // tile) * tile
        E = torch.nn.functional.pad(E, (0, npad - n, 0, npad - n))
        M = torch.nn.functional.pad(M, (0, npad - n, 0, npad - n))
        nt = npad // tile
        Emax = E.reshape(nt, tile, nt, tile).amax(dim=(1, 3)).cpu().numpy()
        Mmax = M.reshape(nt, tile, nt, tile).amax(dim=(1, 3)).cpu().numpy()
    else:
        A = np.asarray(A, dtype=np.float64)
        LU = np.asarray(LU, dtype=np.float64)
        n = LU.shape[0]
        L = np.tril(LU, -1) + np.eye(n)
        U = np.triu(LU)
        npad = -(-n // tile) * tile
        E = np.zeros((npad, npad))
        M = np.zeros((npad, npad))
        E[:n, :n] = np.abs(L @ U - A)
        M[:n, :n] = np.abs(L) @ np.abs(U)
        nt = npad // tile
        Emax = E.reshape(nt, tile, nt, tile).max(axis=(1, 3))
        Mmax = M.reshape(nt, tile, nt, tile).max(axis=(1, 3))
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(Mmax > 0, Emax / np.where(Mmax > 0, Mmax, 1.0), np.where(Emax == 0, 0.0, np.inf))


def factor_tile_distance(LU, LU_ref, tile: int = 128):
    """How far two factorizations of the same matrix are apart, in the units of factor_tile_ratio: per tile
    max|L U - L_ref U_ref| / max(|L| |U|).  Two schedules documented to form the same products up to fp32 rounding
    must stay far below the factors' own backward error here; a wrong tile in one of them shows at its own size even
    where it stays under the backward-error bound.  numpy arrays or torch tensors (CUDA tensors stay on the device)."""
    try:
        import torch
    except ImportError:
        torch = None
    if torch is not None and isinstance(LU_ref, torch.Tensor):
        n = LU_ref.shape[0]
        R = LU_ref.to(torch.float64)
        P = (torch.tril(R, -1) + torch.eye(n, dtype=torch.float64, device=R.device)) @ torch.triu(R)
    else:
        R = np.asarray(LU_ref, dtype=np.float64)
        P = (np.tril(R, -1) + np.eye(R.shape[0])) @ np.triu(R)
    return factor_tile_ratio(P, LU, tile)


def blocked_sweeps(LU, Linv, Uinv, B, dtype=np.float64, store=np.float32, blk: int = 128):
    """Host restatement of the device triangular solve L U X = B (lu_solve_kernel, lu_solve_block_kernel in csrc/ir.cu).
    LU: n x n factors (the fp32 working matrix, widened); Linv / Uinv: the device's fp32 inverses of the unit-lower /
    upper diagonal blk-blocks, shape (npad/blk, blk, blk); B: n or n x k.  The order is padded to npad = ceil(n/blk)*blk
    with identity factors and a zero right-hand side, the right-hand side is cast to fp32 (static_cast<float>(rhs[row]))
    and the two sweeps are left-looking over block rows:
        forward   y_i = Linv_i (b_i - sum_{j<i} L_ij y_j)
        backward  x_i = Uinv_i (y_i - sum_{j>i} U_ij x_j)
    Each solved block is rounded to `store` (the kernels keep ysol / xsol in fp32); everything else is evaluated in `dtype`:
    fp64 gives the reference, fp32 a same-order evaluation whose distance from it sizes the kernels' own rounding.
    Returns X in fp64 with B's shape."""
    LU = np.asarray(LU, dtype=np.float64)
    B = np.asarray(B, dtype=np.float64)
    vec = B.ndim == 1
    B = B.reshape(B.shape[0], -1)
    n, k = B.shape
    npad = -(-n // blk) * blk
    nblk = npad // blk
    F = np.eye(npad, dtype=dtype)
    F[:n, :n] = LU
    Li = np.asarray(Linv, dtype=dtype).reshape(nblk, blk, blk)
    Ui = np.asarray(Uinv, dtype=dtype).reshape(nblk, blk, blk)
    rhs = np.zeros((npad, k), dtype=dtype)
    rhs[:n] = B.astype(np.float32)
    y = np.zeros((npad, k), dtype=dtype)
    x = np.zeros((npad, k), dtype=dtype)
    for i in range(nblk):
        r = slice(i * blk, (i + 1) * blk)
        acc = rhs[r] - F[r, :i * blk] @ y[:i * blk]
        y[r] = (Li[i] @ acc).astype(store)
    for i in reversed(range(nblk)):
        r = slice(i * blk, (i + 1) * blk)
        acc = y[r] - F[r, (i + 1) * blk:] @ x[(i + 1) * blk:]
        x[r] = (Ui[i] @ acc).astype(store)
    X = x[:n].astype(np.float64)
    return X[:, 0] if vec else X


def refine(A: np.ndarray, b: np.ndarray, LU: np.ndarray, max_iters: int = 30, tol: float = 0.0):
    """fp64 iterative refinement with low-precision factors and LAPACK dsgesv's stopping rule
    ||r||_inf <= ||x||_inf ||A||_inf eps sqrt(n).  Returns dict(x, iters, converged, backward_error, first)."""
    n = A.shape[0]
    anorm = np.abs(A).sum(axis=1).max()
    bnorm = np.abs(b).max()
    eps = np.finfo(np.float64).eps / 2
    x = lu_solve(LU, b).astype(np.float64)
    iters, conv, first = 0, False, None
    while True:
        r = b - A @ x
        rn, xn = np.abs(r).max(), np.abs(x).max()
        be = rn / (anorm * xn + bnorm)
        if first is None:
            first = be
        thr = tol * anorm * xn if tol > 0 else xn * anorm * eps * math.sqrt(n)
        if not np.isfinite(rn):
            break
        if rn <= thr:
            conv = True
            break
        if iters >= max_iters:
            break
        x = x + lu_solve(LU, r).astype(np.float64)
        iters += 1
    return dict(x=x, iters=iters, converged=conv, backward_error=be, first_backward_error=first,
                rnorm=rn, xnorm=xn, anorm=anorm, bnorm=bnorm)


def lapack_gesv(A: np.ndarray, b: np.ndarray):
    """Host LAPACK dgetrf + dgetrs (the CPU arm of benchmark.cpp:240 plus the solve the north_star adds)."""
    from scipy.linalg import lu_factor, lu_solve as _ls
    lu, piv = lu_factor(A, check_finite=False)
    return _ls((lu, piv), b, check_finite=False), lu, piv
