"""GPU tests against plain fp64 references of the same operations, on inputs where a wrong off-diagonal tile matters.

* The 16-bit factors of every GETRF path, tile by tile: the componentwise backward error of each 128 x 128 tile
  (oracle.factor_tile_ratio) must stay within 3 unit roundoffs of the 16-bit type.  A bound relative to max|LU| does not
  see a wrong off-diagonal tile next to a large diagonal, and refinement converges on such factors all the same.
* The unrefined first solve and one correction (both outputs of lu_solve_kernel and lu_solve_block_kernel) against a
  host restatement of the blocked sweeps with the device's own factors and block inverses (oracle.blocked_sweeps).
* The norms of the stopping rule (||A||_inf, ||b||_inf, ||x||_inf, the backward errors) against host values.

The matrix is randn + 2 sqrt(n) I: stable without pivoting, and its off-diagonal blocks carry O(1) weight."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
RHO = 3  # bound on the tile-wise componentwise backward error of the factors, in unit roundoffs of the 16-bit type
# bound on the tile-wise distance (oracle.factor_tile_distance) between the factors of paired updates (opts.update_pair)
# and of one update per pass, in unit roundoffs of the 16-bit type.  The two form the same 16-bit products; their sums
# differ by fp32 rounding, and where that rounds a 16-bit multiplier the other way the tile moves by about 1.6 u
# (measured on a B200: 0.3-0.4 u on randn + 2 sqrt(n) I, 1.61 u on the counter matrices).  One tile of a paired product
# scaled by 1.01 moves it to 2.3 u and 3.2 u, while its backward error stays under RHO on randn + 2 sqrt(n) I.
AGREE = 2


def u16(precision):
    return 2.0 ** -11 if precision == 0 else 2.0 ** -8


def cm(t):
    return t.t().contiguous().t()


def randn_dominant(n, seed=0):
    return np.random.default_rng(seed).standard_normal((n, n)) + 2.0 * np.sqrt(n) * np.eye(n)


_SYSTEMS = {}


def system(n):
    """(A, b, device A) for order n, built once per session"""
    import torch
    if n not in _SYSTEMS:
        A = randn_dominant(n, seed=n)
        b = A @ np.random.default_rng(n + 1).standard_normal(n)
        _SYSTEMS[n] = (A, b, cm(torch.tensor(A, device="cuda")))
    return _SYSTEMS[n]


_EMULATED = {}


def emulated_first_berr(oracle, n, precision):
    """first backward error of refinement with the host emulation of the 16-bit factorization"""
    if (n, precision) not in _EMULATED:
        A, b, _ = system(n)
        W = oracle.lu_mixed_emulated(A, 128, bf16=bool(precision))
        _EMULATED[n, precision] = oracle.refine(A, b, W)["first_backward_error"]
    return _EMULATED[n, precision]


def check_factors(oracle, record_property, A, LU, precision, label="rho"):
    rho = oracle.factor_tile_ratio(A, LU)
    worst = np.unravel_index(np.argmax(rho), rho.shape)
    record_property(label, f"{rho.max() / u16(precision):.3f} u")
    assert rho.max() <= RHO * u16(precision), (label, rho.max() / u16(precision), "tile", worst)


def check_agreement(oracle, record_property, LU, LU_ref, precision, label="dist"):
    """LU (paired updates) and LU_ref (one update per pass) factor the same matrix with the same 16-bit products: tile by
    tile their products L U stay within AGREE, below the RHO bound, so a wrong tile that RHO lets pass still shows"""
    d = oracle.factor_tile_distance(LU, LU_ref)
    worst = np.unravel_index(np.argmax(d), d.shape)
    record_property(label, f"{d.max() / u16(precision):.4f} u")
    assert d.max() <= AGREE * u16(precision), (label, d.max() / u16(precision), "tile", worst)


# ---- section 1: the factors of every GETRF path ---------------------------------------------------------------------
_LEFT = {}


def left_factors(mplu, n, precision):
    """factors of the default schedule at nb = 512 (one update per pass), the reference of the paired updates"""
    import torch
    if (n, precision) not in _LEFT:
        A, b, dA = system(n)
        s = mplu.Solver(0)
        try:
            x, st = s.gesv(dA, torch.tensor(b, device="cuda"), mplu.default_options(nb=512, precision=precision))
            assert st.converged == 1 and st.status_bits == 0
            _LEFT[n, precision] = s.factors(n).clone()
        finally:
            s.close()
    return _LEFT[n, precision]


PATHS = {
    "left": dict(),
    "right": dict(schedule=0),
    "fused": dict(flow_w=0),
    "unfused": dict(flow_w=0, fuse_w=0),
    "flow256": dict(flow_w=256),
    "update_pair": dict(update_pair=1),
    "edge_nb": dict(edge_nb=256),
    "pair_ts": dict(pair_ts=1),
    "eager0": dict(eager=0),
    "lazy_touch0": dict(lazy_touch=0),
    "cg1": dict(gemm_variant=0),
    "cg2": dict(gemm_variant=1),
}


@pytest.mark.parametrize("n", [1000, 2304, 4096])
@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("path", list(PATHS))
def test_factors_of_every_path(mplu, oracle, solver, record_property, path, precision, n):
    A, b, dA = system(n)
    import torch
    db = torch.tensor(b, device="cuda")
    x, st = solver.gesv(dA, db, mplu.default_options(nb=512, precision=precision, **PATHS[path]))
    assert st.converged == 1 and st.status_bits == 0 and st.precision_used == precision
    LU = solver.factors(n)
    check_factors(oracle, record_property, dA, LU, precision)
    if path == "update_pair":
        check_agreement(oracle, record_property, LU, left_factors(mplu, n, precision), precision)
    record_property("first_berr", st.first_backward_error)
    if n <= 2304:
        emu = emulated_first_berr(oracle, n, precision)
        record_property("first_berr_over_emulated", st.first_backward_error / emu)
        assert st.first_backward_error <= 4 * emu, (st.first_backward_error, emu)


@pytest.mark.parametrize("n", [1000, 2304, 4096])
@pytest.mark.parametrize("precision", [0, 1])
def test_factors_of_the_streamed_host_path(mplu, oracle, record_property, n, precision):
    A, b, dA = system(n)
    A = np.asfortranarray(A)
    x = np.empty(n)
    s = mplu.Solver(0)
    try:
        st = s.gesv_host_ptr(n, A.ctypes.data, n, b.ctypes.data, x.ctypes.data,
                             mplu.default_options(nb=512, precision=precision, stream_host=1))
        assert st.converged == 1 and st.status_bits == 0 and st.precision_used == precision
        check_factors(oracle, record_property, dA, s.factors(n), precision)
        if n <= 2304:
            assert st.first_backward_error <= 4 * emulated_first_berr(oracle, n, precision)
    finally:
        s.close()


@pytest.mark.parametrize("precision", [0, 1])
def test_factors_n8192(mplu, oracle, solver, record_property, precision):
    import torch
    n = 8192
    A = cm(torch.tensor(randn_dominant(n, seed=3), device="cuda"))
    b = A @ torch.ones(n, dtype=torch.float64, device="cuda")
    x, st = solver.gesv(A, b, mplu.default_options(precision=precision))
    assert st.converged == 1 and st.status_bits == 0
    check_factors(oracle, record_property, A, solver.factors(n), precision)


# ---- section 2: the unrefined first solve and one correction against the host sweeps -------------------------------
def sweep_reference(mplu, oracle, s, n, B):
    """(x_ref, x_ref32): the blocked sweeps of B with the context's factors and fp32 block inverses, evaluated in fp64
    and in fp32"""
    lib = mplu.load_library()
    lib.mplu_debug_block_inverses.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    nblk = (n + 127) // 128
    Li = np.zeros((nblk, 128, 128), dtype=np.float32)
    Ui = np.zeros((nblk, 128, 128), dtype=np.float32)
    for k in range(nblk):
        Lk = np.zeros((128, 128), dtype=np.float32, order="F")
        Uk = np.zeros((128, 128), dtype=np.float32, order="F")
        assert lib.mplu_debug_block_inverses(s._ctx, k, Lk.ctypes.data, Uk.ctypes.data) == 0
        Li[k], Ui[k] = Lk, Uk
    LU = s.factors(n).cpu().numpy()
    # the inverses enter the kernels and the reference alike: each must invert its diagonal block (the last one with its
    # identity padding), or a wrong one would cancel out of the comparison
    F = np.eye(nblk * 128)
    F[:n, :n] = LU
    for k in range(nblk):
        D = F[128 * k:128 * (k + 1), 128 * k:128 * (k + 1)]
        assert np.abs(Li[k].astype(np.float64) @ (np.tril(D, -1) + np.eye(128)) - np.eye(128)).max() <= 1e-4, k
        assert np.abs(np.triu(D) @ Ui[k].astype(np.float64) - np.eye(128)).max() <= 1e-4, k
    return oracle.blocked_sweeps(LU, Li, Ui, B), oracle.blocked_sweeps(LU, Li, Ui, B, dtype=np.float32)


def check_sweeps(got, ref, ref32, record_property=None):
    """per column: ||got - ref|| <= 16 ||ref32 - ref|| + 4 u32 ||ref||"""
    got, ref, ref32 = (np.asarray(v).reshape(len(v), -1) for v in (got, ref, ref32))
    worst = 0.0
    for j in range(ref.shape[1]):
        err = np.abs(got[:, j] - ref[:, j]).max()
        tol = 16 * np.abs(ref32[:, j] - ref[:, j]).max() + 4 * U32 * np.abs(ref[:, j]).max()
        assert err <= tol, (j, err, tol)
        worst = max(worst, err / tol)
    if record_property:
        record_property("err_over_tol", worst)


@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 1000, 2304, 4097])
def test_first_solve_single_vector(mplu, oracle, solver, record_property, n):
    """opts.tol = 1: the first residual meets the stopping rule, x is the first solve (lu_solve_kernel)"""
    A, b, dA = system(n)
    import torch
    x, st = solver.gesv(dA, torch.tensor(b, device="cuda"), mplu.default_options(tol=1.0))
    assert st.converged == 1 and st.iters == 0
    ref, ref32 = sweep_reference(mplu, oracle, solver, n, b)
    check_sweeps(x.cpu().numpy(), ref, ref32, record_property)
    # the norms of the stopping rule against the host
    x0 = x.cpu().numpy()
    r = b - A @ x0
    anorm = np.abs(A).sum(axis=1).max()
    assert st.anorm_inf == pytest.approx(anorm, rel=1e-13, abs=0)
    assert st.bnorm_inf == np.abs(b).max() and st.xnorm_inf == np.abs(x0).max()
    berr = np.abs(r).max() / (anorm * np.abs(x0).max() + np.abs(b).max())
    assert st.backward_error == pytest.approx(berr, rel=1e-6, abs=0)
    assert st.first_backward_error == st.backward_error


def block_buffers(B, ldb, ldx):
    """B in a column-major buffer with leading dimension ldb, an X buffer with ldx (rows n.. hold markers)"""
    import torch
    n, k = B.shape
    Bbuf = torch.full((k, ldb), 7.0, dtype=torch.float64, device="cuda")
    Bbuf[:, :n] = torch.tensor(B.T, device="cuda")
    Xbuf = torch.full((k, ldx), -12345.0, dtype=torch.float64, device="cuda")
    return Bbuf, Xbuf


@pytest.mark.parametrize("nrhs", [2, 3, 8, 9, 17])
def test_first_solve_block(mplu, oracle, record_property, nrhs):
    """lu_solve_block_kernel's first solve (8 columns per launch: kc < 8, kc = 8 and a second column block occur) against
    the host sweeps, column by column; each column bit-identical to the single-vector first solve of that column"""
    import torch
    n, ldb, ldx = 1000, 1003, 1010
    A, _, dA = system(n)
    B = A @ np.random.default_rng(nrhs).standard_normal((n, nrhs))
    B[:, 0] *= 1e-8
    B[:, -1] *= 1e8
    Bbuf, Xbuf = block_buffers(B, ldb, ldx)
    s = mplu.Solver(0)
    try:
        torch.cuda.synchronize()
        st, berr = s.gesv_nrhs_ptr(n, nrhs, dA.data_ptr(), n, Bbuf.data_ptr(), ldb, Xbuf.data_ptr(), ldx,
                                   mplu.default_options(tol=1.0))
        assert st.converged == 1 and st.iters == 0
        Xh = Xbuf.cpu().numpy()
        assert (Xh[:, n:] == -12345.0).all()
        X0 = Xh[:, :n].T.copy()
        ref, ref32 = sweep_reference(mplu, oracle, s, n, B)
        check_sweeps(X0, ref, ref32, record_property)
        # the same first solve through the stored factors, and column by column through the single-vector kernel
        X2 = torch.empty(nrhs, n, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        st2, berr2 = s.solve_nrhs_ptr(nrhs, dA.data_ptr(), n, Bbuf.data_ptr(), ldb, X2.data_ptr(), n)
        assert st2.iters == 0
        np.testing.assert_array_equal(X2.cpu().numpy().T, X0)
        for j in range(nrhs):
            bj = Bbuf[j, :n].contiguous()
            xj = torch.empty(n, dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            sj = s.solve_ptr(dA.data_ptr(), n, bj.data_ptr(), xj.data_ptr())
            assert sj.iters == 0
            np.testing.assert_array_equal(xj.cpu().numpy(), X0[:, j], err_msg=f"column {j}")
        # the norms: per-column backward errors, ||b|| and ||x|| of the worst column, ||A||_inf
        anorm = np.abs(A).sum(axis=1).max()
        R = B - A @ X0
        ref_berr = np.abs(R).max(axis=0) / (anorm * np.abs(X0).max(axis=0) + np.abs(B).max(axis=0))
        np.testing.assert_allclose(berr, ref_berr, rtol=1e-6, atol=0)
        w = int(np.argmax(berr))
        assert st.bnorm_inf == np.abs(B[:, w]).max() and st.xnorm_inf == np.abs(X0[:, w]).max()
        assert st.anorm_inf == pytest.approx(anorm, rel=1e-13, abs=0)
    finally:
        s.close()


@pytest.mark.parametrize("nrhs", [1, 9])
def test_correction(mplu, oracle, solver, record_property, nrhs):
    """the other output of both sweep kernels, x_accum += D: one correction x1 = x0 + (LU)^-1 (b - A x0)
    against the host sweeps of the host residual of x0 (this also checks the entries of the block residual)"""
    import torch
    n = 2304
    A, _, dA = system(n)
    B = A @ np.random.default_rng(5).standard_normal((n, nrhs))
    dB = cm(torch.tensor(B, device="cuda"))

    def run(**kw):
        if nrhs == 1:
            x, st = solver.gesv(dA, dB[:, 0].contiguous(), mplu.default_options(**kw), allow_noconv=True)
            return x.cpu().numpy().reshape(n, 1), st
        X, st, _ = solver.gesv_nrhs(dA, dB, mplu.default_options(**kw), allow_noconv=True)
        return X.cpu().numpy(), st

    X0, st0 = run(tol=1.0)
    assert st0.iters == 0
    X1, st1 = run(max_iters=1, tol=1e-300, fp64_fallback=0)
    assert st1.iters == 1 and st1.converged == 0
    R0 = B - A @ X0
    ref, ref32 = sweep_reference(mplu, oracle, solver, n, R0)
    check_sweeps(X1 - X0, ref.reshape(n, -1), ref32.reshape(n, -1), record_property)


# ---- section 3: ||A||_inf against the host on every path that forms it ---------------------------------------------
@pytest.mark.parametrize("lazy", [1, 0])
def test_anorm_single_vector(mplu, solver, lazy):
    import torch
    n = 2304  # a multiple of 128
    A, b, dA = system(n)
    x, st = solver.gesv(dA, torch.tensor(b, device="cuda"), mplu.default_options(lazy_touch=lazy))
    assert st.converged == 1
    assert st.anorm_inf == pytest.approx(np.abs(A).sum(axis=1).max(), rel=1e-13, abs=0)


def test_anorm_block_lazy(mplu, solver):
    """nrhs = 20: two residual column blocks, only the first forms the row sums of |A|"""
    import torch
    n, nrhs = 2304, 20
    A, _, dA = system(n)
    B = A @ np.random.default_rng(20).standard_normal((n, nrhs))
    X, st, berr = solver.gesv_nrhs(dA, cm(torch.tensor(B, device="cuda")), mplu.default_options(lazy_touch=1))
    assert st.converged == 1
    assert st.anorm_inf == pytest.approx(np.abs(A).sum(axis=1).max(), rel=1e-13, abs=0)


def test_anorm_streamed_host(mplu):
    n = 2304
    A, b, _ = system(n)
    A = np.asfortranarray(A)
    x = np.empty(n)
    s = mplu.Solver(0)
    try:
        st = s.gesv_host_ptr(n, A.ctypes.data, n, b.ctypes.data, x.ctypes.data, mplu.default_options(nb=512, stream_host=1))
        assert st.converged == 1
        assert st.anorm_inf == pytest.approx(np.abs(A).sum(axis=1).max(), rel=1e-13, abs=0)
    finally:
        s.close()


def test_anorm_block_cyclic(mplu, oracle):
    n, nb = 1024, 256
    ds = mplu.DistSolver(0, 2, 2)
    try:
        As, bs = ds.generate(n, nb, seed=1)
        xs, st = ds.gesv(n, nb, As, bs, mplu.default_options())
        assert st.converged == 1
        A = oracle.counter_matrix(n, seed=1)
        assert st.anorm_inf == pytest.approx(np.abs(A).sum(axis=1).max(), rel=1e-13, abs=0)
        assert st.bnorm_inf == np.abs(bs[0].cpu().numpy()).max()
    finally:
        ds.close()
