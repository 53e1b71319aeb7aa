"""ctypes binding of libmplu.so -- the B200-native mixed-precision LU + iterative refinement solver.

Python is plumbing only (device memory via torch, tests, bench); every numerical step runs in the CUDA kernels of
csrc/.  The library must be present: there is no CPU or PyTorch fallback, loading fails loudly instead.

Mirrors the reference's interface for this path: ``MPF(A, N, r, IPIV)`` (/root/reference/MPF.h:3) plus the
``mplu_*`` C ABI of include/mplu.h.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libmplu.so"

MPLU_FP16, MPLU_BF16 = 0, 1
GEMM_AUTO, GEMM_CG1, GEMM_CG2 = -1, 0, 1
REFINE_CLASSIC, REFINE_GMRES = 0, 1

ERRORS = {
    0: "ok", -1: "bad argument", -2: "no CUDA device", -3: "not factored", -4: "TMA descriptor encoding failed",
    -5: "fp16 overflow in a panel", -6: "zero pivot", -7: "refinement did not converge", -8: "NCCL error / unavailable",
}


class Options(C.Structure):
    _fields_ = [("precision", C.c_int), ("nb", C.c_int), ("max_iters", C.c_int), ("tol", C.c_double),
                ("gemm_variant", C.c_int), ("max_sms", C.c_int), ("a_exp", C.c_int), ("l_exp", C.c_int),
                ("lookahead", C.c_int), ("side_sms", C.c_int), ("use_graph", C.c_int), ("pdl", C.c_int), ("group", C.c_int),
                ("refinement", C.c_int), ("gmres_restart", C.c_int), ("gmres_tol", C.c_double), ("bf16_fallback", C.c_int), ("tile_ws", C.c_int), ("cg2_min_elems", C.c_int), ("side_sms_early", C.c_int), ("early_pct", C.c_int), ("tri_skip", C.c_int), ("late_pct", C.c_int), ("l2_persist", C.c_int), ("stream_host", C.c_int), ("schedule", C.c_int), ("eager", C.c_int), ("side_sms_left", C.c_int), ("stream_c", C.c_int), ("early_scale", C.c_int), ("fuse_w", C.c_int), ("fuse_ctas", C.c_int), ("lazy_touch", C.c_int), ("flow_w", C.c_int), ("flow_ctas", C.c_int), ("fp64_fallback", C.c_int), ("edge_nb", C.c_int), ("pair_ts", C.c_int), ("update_pair", C.c_int), ("flow_merge_ctas", C.c_int), ("equilibrate", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("n", C.c_int), ("iters", C.c_int), ("converged", C.c_int), ("status_bits", C.c_int),
                ("anorm_inf", C.c_double), ("bnorm_inf", C.c_double), ("xnorm_inf", C.c_double),
                ("rnorm_inf", C.c_double), ("backward_error", C.c_double), ("first_backward_error", C.c_double),
                ("factor_ms", C.c_float), ("solve_ms", C.c_float), ("total_ms", C.c_float),
                ("h2d_ms", C.c_float), ("d2h_ms", C.c_float), ("gemm_launches", C.c_int),
                ("kernel_launches", C.c_int), ("trailing_launches", C.c_int), ("trailing_ms", C.c_float),
                ("trailing_flops", C.c_double), ("trailing_bytes", C.c_double), ("gmres_iters", C.c_int), ("precision_used", C.c_int), ("fp64_fallback", C.c_int), ("dsgesv_iter", C.c_int), ("equed", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class MpluError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        msg = ERRORS.get(code, f"cudaError {code}" if code > 0 else f"error {code}")
        super().__init__(f"{where}: {msg} ({code})")


_lib = None


def load_library(path: os.PathLike | None = None) -> C.CDLL:
    """Load libmplu.so (built by build.py / __graft_entry__.build()).  Raises if it is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise FileNotFoundError(f"{p} not found: run `python __graft_entry__.py build` (no CPU fallback exists)")
    lib = C.CDLL(str(p), mode=C.RTLD_GLOBAL)
    vp, ll, i, f, d = C.c_void_p, C.c_longlong, C.c_int, C.c_float, C.c_double
    lib.mplu_default_options.argtypes = [C.POINTER(Options)]
    lib.mplu_default_options.restype = None
    lib.mplu_create.argtypes = [C.POINTER(vp), i]
    lib.mplu_destroy.argtypes = [vp]
    lib.mplu_destroy.restype = None
    lib.mplu_stream.argtypes = [vp]
    lib.mplu_stream.restype = vp
    lib.mplu_factor_device.argtypes = [vp, i, vp, ll, C.POINTER(Options)]
    lib.mplu_solve_device.argtypes = [vp, vp, ll, vp, vp, C.POINTER(Stats)]
    lib.mplu_gesv_device.argtypes = [vp, i, vp, ll, vp, vp, C.POINTER(Options), C.POINTER(Stats)]
    lib.mplu_gesv_host.argtypes = [vp, i, vp, ll, vp, vp, C.POINTER(Options), C.POINTER(Stats)]
    lib.mplu_get_factors.argtypes = [vp, vp, ll, i]
    lib.mplu_get_equilibration.argtypes = [vp, C.POINTER(i), vp, vp, i]
    dp = C.POINTER(C.c_double)
    lib.mplu_solve_device_nrhs.argtypes = [vp, i, vp, ll, vp, ll, vp, ll, dp, C.POINTER(Stats)]
    lib.mplu_gesv_device_nrhs.argtypes = [vp, i, i, vp, ll, vp, ll, vp, ll, C.POINTER(Options), dp, C.POINTER(Stats)]
    lib.mplu_gesv_host_nrhs.argtypes = lib.mplu_gesv_device_nrhs.argtypes
    lib.mplu_gemm16.argtypes = [i, i, i, i, i, f, vp, ll, vp, ll, f, vp, ll, vp, ll, f, i, vp]
    lib.mplu_diag_lu128.argtypes = [vp, ll, vp, vp, vp]
    lib.mplu_residual.argtypes = [i, vp, ll, vp, vp, vp, vp, vp]
    lib.mplu_generate.argtypes = [i, C.c_ulonglong, i, vp, ll, vp, vp]
    lib.mplu_generate.restype = i
    for name in ("mplu_create", "mplu_factor_device", "mplu_solve_device", "mplu_gesv_device", "mplu_gesv_host",
                 "mplu_get_factors", "mplu_gemm16", "mplu_diag_lu128", "mplu_residual", "mplu_solve_device_nrhs",
                 "mplu_gesv_device_nrhs", "mplu_gesv_host_nrhs", "mplu_get_equilibration"):
        getattr(lib, name).restype = i
    lib.mplu_MPF.argtypes = [vp, i, i, vp]
    lib.mplu_MPF.restype = i
    lib.mplu_hgetf2.argtypes = [vp, i, i, i, vp, vp]
    lib.mplu_hgetf2.restype = i
    lib.mplu_dgetf2_npv.argtypes = [i, i, vp, i, vp]
    lib.mplu_dgetf2_npv.restype = i
    lib.mplu_dist_unique_id.argtypes = [vp]
    lib.mplu_dist_create.argtypes = [C.POINTER(vp), i, i, i, i, i, vp]
    lib.mplu_dist_create_local.argtypes = [C.POINTER(vp), i, i, i]
    lib.mplu_dist_destroy.argtypes = [vp]
    lib.mplu_dist_destroy.restype = None
    lib.mplu_dist_num_local.argtypes = [vp]
    lib.mplu_dist_local_shape.argtypes = [vp, i, i, i, C.POINTER(i), C.POINTER(i), C.POINTER(ll), C.POINTER(ll)]
    lib.mplu_dist_gesv.argtypes = [vp, i, i, C.POINTER(vp), C.POINTER(ll), C.POINTER(vp), C.POINTER(vp),
                                   C.POINTER(Options), C.POINTER(Stats)]
    lib.mplu_dist_gesv_host.argtypes = lib.mplu_dist_gesv.argtypes
    lib.mplu_dist_gesv_host.restype = i
    lib.mplu_dist_release_staging.argtypes = [vp]
    lib.mplu_dist_release_staging.restype = None
    lib.mplu_dist_get_local_factors.argtypes = [vp, i, vp, ll]
    lib.mplu_generate_local.argtypes = [i, C.c_ulonglong, i, i, i, i, i, vp, ll, vp, vp]
    for name in ("mplu_dist_unique_id", "mplu_dist_create", "mplu_dist_create_local", "mplu_dist_num_local",
                 "mplu_dist_local_shape", "mplu_dist_gesv", "mplu_dist_get_local_factors", "mplu_generate_local"):
        getattr(lib, name).restype = i
    if path is None:
        _lib = lib
    return lib


def default_options(**kw) -> Options:
    o = Options()
    load_library().mplu_default_options(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise TypeError(f"unknown option {k}")
        setattr(o, k, v)
    return o


def _dptr(a):
    """numpy float64 array -> double* for ctypes"""
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _check(code: int, where: str, allow=()):
    if code != 0 and code not in allow:
        raise MpluError(code, where)
    return code


class Solver:
    """One solver context (one CUDA device, one stream, reusable workspaces)."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        self._ctx = C.c_void_p()
        _check(self._lib.mplu_create(C.byref(self._ctx), device), "mplu_create")

    def close(self):
        if self._ctx:
            self._lib.mplu_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self) -> int:
        return self._lib.mplu_stream(self._ctx) or 0

    # raw device pointers -------------------------------------------------------------------------------------
    def factor_ptr(self, n, dA, lda, opts=None):
        _check(self._lib.mplu_factor_device(self._ctx, n, dA, lda, C.byref(opts) if opts else None), "mplu_factor_device")

    def solve_ptr(self, dA, lda, db, dx, allow_noconv=False) -> Stats:
        st = Stats()
        _check(self._lib.mplu_solve_device(self._ctx, dA, lda, db, dx, C.byref(st)), "mplu_solve_device",
               allow=(-7,) if allow_noconv else ())
        return st

    def gesv_ptr(self, n, dA, lda, db, dx, opts=None, allow_noconv=False) -> Stats:
        st = Stats()
        _check(self._lib.mplu_gesv_device(self._ctx, n, dA, lda, db, dx, C.byref(opts) if opts else None, C.byref(st)),
               "mplu_gesv_device", allow=(-7,) if allow_noconv else ())
        return st

    def gesv_host_ptr(self, n, hA, lda, hb, hx, opts=None, allow_noconv=False) -> Stats:
        st = Stats()
        _check(self._lib.mplu_gesv_host(self._ctx, n, hA, lda, hb, hx, C.byref(opts) if opts else None, C.byref(st)),
               "mplu_gesv_host", allow=(-7,) if allow_noconv else ())
        return st

    # several right-hand sides: B / X column-major n x nrhs (leading dimensions ldb / ldx); returns (Stats, berr), berr a
    # numpy array of the nrhs per-column backward errors
    def solve_nrhs_ptr(self, nrhs, dA, lda, dB, ldb, dX, ldx, allow_noconv=False):
        import numpy as np
        st, berr = Stats(), np.zeros(max(nrhs, 1))
        _check(self._lib.mplu_solve_device_nrhs(self._ctx, nrhs, dA, lda, dB, ldb, dX, ldx, _dptr(berr), C.byref(st)),
               "mplu_solve_device_nrhs", allow=(-7,) if allow_noconv else ())
        return st, berr[:nrhs]

    def gesv_nrhs_ptr(self, n, nrhs, dA, lda, dB, ldb, dX, ldx, opts=None, allow_noconv=False):
        import numpy as np
        st, berr = Stats(), np.zeros(max(nrhs, 1))
        _check(self._lib.mplu_gesv_device_nrhs(self._ctx, n, nrhs, dA, lda, dB, ldb, dX, ldx, C.byref(opts) if opts else None,
                                                _dptr(berr), C.byref(st)), "mplu_gesv_device_nrhs",
               allow=(-7,) if allow_noconv else ())
        return st, berr[:nrhs]

    def gesv_host_nrhs_ptr(self, n, nrhs, hA, lda, hB, ldb, hX, ldx, opts=None, allow_noconv=False):
        import numpy as np
        st, berr = Stats(), np.zeros(max(nrhs, 1))
        _check(self._lib.mplu_gesv_host_nrhs(self._ctx, n, nrhs, hA, lda, hB, ldb, hX, ldx, C.byref(opts) if opts else None,
                                              _dptr(berr), C.byref(st)), "mplu_gesv_host_nrhs",
               allow=(-7,) if allow_noconv else ())
        return st, berr[:nrhs]

    # torch conveniences (column-major convention: pass A.t().contiguous() storage, i.e. a tensor whose memory is
    # column-major; helpers below take "colmajor" tensors of shape (n, n) created with torch.empty(n, n).t()) -----
    def gesv(self, A_cm, b, opts=None, allow_noconv=False):
        """A_cm: torch fp64 CUDA tensor whose storage is column-major n x n (e.g. M.t() of a contiguous M^T)."""
        import torch
        n = A_cm.shape[0]
        assert A_cm.dtype == torch.float64 and A_cm.is_cuda and A_cm.stride(0) == 1
        lda = A_cm.stride(1)
        x = torch.empty(n, dtype=torch.float64, device=A_cm.device)
        torch.cuda.synchronize(A_cm.device)
        st = self.gesv_ptr(n, A_cm.data_ptr(), lda, b.data_ptr(), x.data_ptr(), opts, allow_noconv)
        return x, st

    def gesv_nrhs(self, A_cm, B_cm, opts=None, allow_noconv=False):
        """A X = B.  A_cm (n x n) and B_cm (n x nrhs): torch fp64 CUDA tensors with column-major storage.  Returns
        (X, stats, berr): X column-major n x nrhs, berr a numpy array of the per-column backward errors."""
        import torch
        n, nrhs = B_cm.shape
        assert A_cm.dtype == torch.float64 and A_cm.is_cuda and A_cm.stride(0) == 1 and A_cm.shape == (n, n)
        assert B_cm.dtype == torch.float64 and B_cm.is_cuda and B_cm.stride(0) == 1
        X = torch.empty(nrhs, n, dtype=torch.float64, device=A_cm.device).t()  # column-major storage
        torch.cuda.synchronize(A_cm.device)
        st, berr = self.gesv_nrhs_ptr(n, nrhs, A_cm.data_ptr(), A_cm.stride(1), B_cm.data_ptr(), max(B_cm.stride(1), n),
                                      X.data_ptr(), n, opts, allow_noconv)
        return X, st, berr

    def factors(self, n):
        import torch
        LU = torch.empty(n, n, dtype=torch.float64, device="cuda").t()  # column-major storage
        _check(self._lib.mplu_get_factors(self._ctx, LU.data_ptr(), n, 1), "mplu_get_factors")
        return LU

    def equilibration(self, n):
        """(equed, r, c) of the last factorization (opts.equilibrate): EQUED 0 N / 1 R / 2 C / 3 B and the row / column
        scales as fp64 CUDA tensors of length n (ones on a side that was not applied); the stored factors are those of
        diag(r) A diag(c)."""
        import torch
        r = torch.empty(n, dtype=torch.float64, device="cuda")
        c = torch.empty(n, dtype=torch.float64, device="cuda")
        equed = C.c_int()
        torch.cuda.synchronize()
        _check(self._lib.mplu_get_equilibration(self._ctx, C.byref(equed), r.data_ptr(), c.data_ptr(), 1),
               "mplu_get_equilibration")
        return equed.value, r, c


# ---- 2D block-cyclic layout (host-side helpers; the same index maps as csrc/dist.cu) ------------------------------
def grid_shape(nranks: int):
    """P x Q process grid for `nranks` GPUs: the most square factorization with P <= Q (8 -> 2 x 4)."""
    p = int(nranks ** 0.5)
    while nranks % p:
        p -= 1
    return p, nranks // p


def tiles_local(T: int, P: int, p: int) -> int:
    """Number of the T tiles of one dimension that process p of P owns (tiles dealt round-robin)."""
    return (T - p + P - 1) // P if p < T else 0


def local_to_global(l: int, nb: int, P: int, p: int) -> int:
    """Global row/column index of local index l on process p (ScaLAPACK local order)."""
    return ((l // nb) * P + p) * nb + l % nb


def global_to_local(g: int, nb: int, P: int):
    """(owning process, local index) of global row/column g."""
    t = g // nb
    return t % P, (t // P) * nb + g % nb


def scatter_block_cyclic(A, nb: int, P: int, Q: int):
    """Split a global n x n array (numpy or torch) into the P*Q local arrays, row-major over (p, q)."""
    n = A.shape[0]
    T = n // nb
    out = []
    for p in range(P):
        rows = [i for t in range(p, T, P) for i in range(t * nb, (t + 1) * nb)]
        for q in range(Q):
            cols = [j for t in range(q, T, Q) for j in range(t * nb, (t + 1) * nb)]
            out.append(A[rows][:, cols])
    return out


def gather_block_cyclic(parts, n: int, nb: int, P: int, Q: int):
    """Inverse of scatter_block_cyclic (numpy arrays)."""
    import numpy as np
    T = n // nb
    A = np.zeros((n, n), dtype=parts[0].dtype)
    for p in range(P):
        rows = [i for t in range(p, T, P) for i in range(t * nb, (t + 1) * nb)]
        for q in range(Q):
            cols = [j for t in range(q, T, Q) for j in range(t * nb, (t + 1) * nb)]
            if rows and cols:
                A[np.ix_(rows, cols)] = parts[p * Q + q]
    return A


class DistSolver:
    """Block-cyclic LU + IR over a P x Q process grid (csrc/dist.cu).

    unique_id=None: "local" mode, all P*Q logical ranks live in this process on `device` (collectives are device
    copies) -- used by the single-GPU tests.  Otherwise one rank of an NCCL communicator (one process per GPU)."""

    def __init__(self, device: int, P: int, Q: int, rank: int | None = None, unique_id: bytes | None = None):
        self._lib = load_library()
        self._d = C.c_void_p()
        self.P, self.Q = P, Q
        if unique_id is None:
            _check(self._lib.mplu_dist_create_local(C.byref(self._d), device, P, Q), "mplu_dist_create_local")
        else:
            buf = C.create_string_buffer(bytes(unique_id), 128)
            _check(self._lib.mplu_dist_create(C.byref(self._d), device, rank, P * Q, P, Q, buf), "mplu_dist_create")
        self.num_local = self._lib.mplu_dist_num_local(self._d)

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _check(load_library().mplu_dist_unique_id(buf), "mplu_dist_unique_id")
        return buf.raw

    def close(self):
        if self._d:
            self._lib.mplu_dist_destroy(self._d)
            self._d = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def local_shape(self, i, n, nb):
        p, q, m, nn = C.c_int(), C.c_int(), C.c_longlong(), C.c_longlong()
        _check(self._lib.mplu_dist_local_shape(self._d, i, n, nb, C.byref(p), C.byref(q), C.byref(m), C.byref(nn)),
               "mplu_dist_local_shape")
        return p.value, q.value, m.value, nn.value

    def generate(self, n, nb, seed=1):
        """Local tiles of the synthetic dominant system for every logical rank of this process + the full b."""
        import torch
        As, bs = [], []
        for i in range(self.num_local):
            p, q, m, nn = self.local_shape(i, n, nb)
            A = torch.zeros(max(nn, 1), max(m, 1), dtype=torch.float64, device="cuda").t()  # column-major m x nn
            b = torch.empty(n, dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            _check(self._lib.mplu_generate_local(n, seed, nb, self.P, self.Q, p, q, A.data_ptr(), A.stride(1),
                                                 b.data_ptr(), None), "mplu_generate_local")
            As.append(A)
            bs.append(b)
        torch.cuda.synchronize()
        return As, bs

    def gesv(self, n, nb, As, bs, opts=None, allow_noconv=False):
        import torch
        L = self.num_local
        xs = [torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(L)]
        pa = (C.c_void_p * L)(*[a.data_ptr() for a in As])
        ld = (C.c_longlong * L)(*[a.stride(1) for a in As])
        pb = (C.c_void_p * L)(*[b.data_ptr() for b in bs])
        px = (C.c_void_p * L)(*[x.data_ptr() for x in xs])
        st = Stats()
        torch.cuda.synchronize()
        _check(self._lib.mplu_dist_gesv(self._d, n, nb, pa, ld, pb, px, C.byref(opts) if opts else None, C.byref(st)),
               "mplu_dist_gesv", allow=(-7,) if allow_noconv else ())
        return xs, st

    def gesv_host(self, n, nb, hAs, hbs, hxs, opts=None, allow_noconv=False):
        """hAs: host (ideally pinned) torch tensors with column-major local tiles; hbs / hxs: full host vectors."""
        L = self.num_local
        pa = (C.c_void_p * L)(*[a.data_ptr() for a in hAs])
        ld = (C.c_longlong * L)(*[a.stride(1) for a in hAs])
        pb = (C.c_void_p * L)(*[b.data_ptr() for b in hbs])
        px = (C.c_void_p * L)(*[x.data_ptr() for x in hxs])
        st = Stats()
        _check(self._lib.mplu_dist_gesv_host(self._d, n, nb, pa, ld, pb, px, C.byref(opts) if opts else None,
                                             C.byref(st)), "mplu_dist_gesv_host", allow=(-7,) if allow_noconv else ())
        return st

    def release_staging(self):
        self._lib.mplu_dist_release_staging(self._d)

    def local_factors(self, i, n, nb):
        import torch
        _, _, m, nn = self.local_shape(i, n, nb)
        LU = torch.empty(max(nn, 1), max(m, 1), dtype=torch.float64, device="cuda").t()
        _check(self._lib.mplu_dist_get_local_factors(self._d, i, LU.data_ptr(), LU.stride(1)), "mplu_dist_get_local_factors")
        return LU


def gemm16(variant, A, B, C_io=None, alpha=1.0, beta=0.0, want_shadow=False, hscale=1.0, max_sms=0, a_transposed=None):
    """Kernel-level hook used by the parity tests.  A (M x K) and B (K x N) are 16-bit CUDA tensors with
    column-major storage (stride(0) == 1); for variants 2/3 pass `a_transposed` = K x M column-major instead."""
    import torch
    lib = load_library()
    if variant in (2, 3):
        At = a_transposed
        K, M = At.shape
        a_ptr, lda = At.data_ptr(), At.stride(1)
        dt = At.dtype
    else:
        M, K = A.shape
        assert A.stride(0) == 1
        a_ptr, lda = A.data_ptr(), A.stride(1)
        dt = A.dtype
    K2, N = B.shape
    assert K2 == K and B.stride(0) == 1
    bf16 = 1 if dt == torch.bfloat16 else 0
    if C_io is None:
        C_io = torch.zeros(N, M, dtype=torch.float32, device=B.device).t()
    assert C_io.stride(0) == 1
    H = torch.zeros(N, M, dtype=dt, device=B.device).t() if want_shadow else None
    torch.cuda.synchronize()
    rc = lib.mplu_gemm16(variant, bf16, M, N, K, alpha, a_ptr, lda, B.data_ptr(), B.stride(1), beta,
                         C_io.data_ptr(), C_io.stride(1), H.data_ptr() if H is not None else None,
                         H.stride(1) if H is not None else 0, hscale, max_sms, None)
    _check(rc, "mplu_gemm16")
    torch.cuda.synchronize()
    return (C_io, H) if want_shadow else C_io


def generate(n, seed=1, dominant=True, with_rhs=True):
    """Device-resident synthetic system (column-major fp64 A, b = A*1) -- same formula as the oracle's counter_matrix."""
    import torch
    A = torch.empty(n, n, dtype=torch.float64, device="cuda").t()
    b = torch.empty(n, dtype=torch.float64, device="cuda") if with_rhs else None
    torch.cuda.synchronize()
    _check(load_library().mplu_generate(n, seed, 1 if dominant else 0, A.data_ptr(), n,
                                        b.data_ptr() if with_rhs else None, None), "mplu_generate")
    torch.cuda.synchronize()
    return A, b


def generate_spd(n, kappa, seed=1):
    """Device-resident SPD test matrix A = H diag(sigma) H, H = I - 2uu^T, sigma geometric in [1/kappa, 1] (the
    condition-number sweep of BASELINE.json configs[4]; same construction as the oracle's spd_kappa_matrix, built in
    O(n^2) on the device).  Symmetric, so its row-major storage is also its column-major storage."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    u /= u.norm()
    sig = kappa ** (-torch.arange(n, dtype=torch.float64, device="cuda") / max(n - 1, 1))
    du = sig * u
    A = torch.diag(sig)
    A -= 2.0 * torch.outer(u, du)
    A -= 2.0 * torch.outer(du, u)
    A += 4.0 * torch.dot(u, du) * torch.outer(u, u)
    return A


def MPF(A, r=32, ipiv=None):
    """Reference-compatible entry point (/root/reference/MPF.h:3): factor the column-major fp64 HOST matrix `A`
    (numpy, Fortran order, modified in place) with panel width r; returns the 1-based pivot vector."""
    import numpy as np
    assert A.dtype == np.float64 and A.flags.f_contiguous and A.shape[0] == A.shape[1]
    n = A.shape[0]
    if ipiv is None:
        ipiv = np.arange(1, n + 1, dtype=np.int32)  # benchmark.cpp:215-217
    _check(load_library().mplu_MPF(A.ctypes.data, n, r, ipiv.ctypes.data), "MPF")
    return ipiv
