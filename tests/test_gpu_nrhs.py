"""GPU tests of the multi-column solve (mplu_solve_device_nrhs / mplu_gesv_device_nrhs / mplu_gesv_host_nrhs): batched
fp64 residual and fp32 triangular-solve kernels, dsgesv refinement over a block of right-hand sides."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps / 2  # unit roundoff
TIMING = {"factor_ms", "solve_ms", "total_ms", "h2d_ms", "d2h_ms", "trailing_ms"}


def cm(t):
    return t.t().contiguous().t()


def dev(a):
    import torch
    return cm(torch.tensor(np.asarray(a, dtype=np.float64).reshape(a.shape[0], -1), device="cuda"))


def system(oracle, n, nrhs, seed=0):
    A = oracle.counter_matrix(n, seed=2)
    Xt = np.random.default_rng(seed).standard_normal((n, nrhs))
    return A, Xt, A @ Xt


def gesv_nrhs(mplu, solver, A, B, allow_noconv=False, **kw):
    import torch
    dA, dB = dev(A), dev(B)
    B0 = dB.clone()
    X, st, berr = solver.gesv_nrhs(dA, dB, mplu.default_options(**kw), allow_noconv)
    assert torch.equal(dB.view(torch.int64), B0.view(torch.int64))  # B is not modified (bit for bit: B may hold a NaN)
    return X.cpu().numpy(), st, berr


@pytest.mark.parametrize("n", [1000, 2304, 4096])
@pytest.mark.parametrize("nrhs", [2, 3, 16, 17, 40])
def test_shapes(mplu, oracle, solver, n, nrhs):
    """ragged and block-aligned n; nrhs below, at and across the column blocks of both kernels"""
    A, Xt, B = system(oracle, n, nrhs)
    X, st, berr = gesv_nrhs(mplu, solver, A, B)
    assert st.converged == 1 and st.status_bits == 0 and st.fp64_fallback == 0
    assert berr.shape == (nrhs,) and (berr <= 2 * n * EPS).all(), berr
    assert st.backward_error == berr.max()
    np.testing.assert_allclose(X, Xt, rtol=0, atol=1e-11)


def test_one_column_is_the_single_vector_path(mplu, oracle, solver):
    import torch
    n = 1000
    A, Xt, B = system(oracle, n, 1)
    dA, db = dev(A), torch.tensor(B[:, 0], device="cuda")
    x1, s1 = solver.gesv(dA, db, mplu.default_options())
    X2, s2, berr = solver.gesv_nrhs(dA, cm(db.reshape(n, 1)), mplu.default_options())
    assert torch.equal(x1, X2[:, 0])
    d1, d2 = s1.as_dict(), s2.as_dict()
    assert {k: v for k, v in d1.items() if k not in TIMING} == {k: v for k, v in d2.items() if k not in TIMING}
    assert berr[0] == s1.backward_error
    # solve with stored factors
    x3 = torch.empty(n, dtype=torch.float64, device="cuda")
    X4 = torch.empty(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    s3 = solver.solve_ptr(dA.data_ptr(), n, db.data_ptr(), x3.data_ptr())
    s4, _ = solver.solve_nrhs_ptr(1, dA.data_ptr(), n, db.data_ptr(), n, X4.data_ptr(), n)
    assert torch.equal(x3, X4)
    skip = TIMING | {"kernel_launches"}  # the launch counter runs on across solves with the same factors
    assert {k: v for k, v in s3.as_dict().items() if k not in skip} == {k: v for k, v in s4.as_dict().items() if k not in skip}
    # b = 0: x = 0 solves it exactly, so the backward error is 0, as for a zero column of a block
    z = torch.zeros(n, dtype=torch.float64, device="cuda")
    x5, s5 = solver.gesv(dA, z, mplu.default_options())
    X6, s6, berr6 = solver.gesv_nrhs(dA, cm(z.reshape(n, 1)), mplu.default_options())
    torch.cuda.synchronize()
    s7 = solver.solve_ptr(dA.data_ptr(), n, z.data_ptr(), x3.data_ptr())
    for s in (s5, s6, s7):
        assert s.converged == 1 and s.backward_error == 0.0 and s.first_backward_error == 0.0
    assert (x5 == 0).all() and (X6 == 0).all() and (x3 == 0).all() and berr6[0] == 0.0
    # ||b||_inf keeps a NaN of b, like the column norms of a block
    z[n // 2] = float("nan")
    torch.cuda.synchronize()
    s8 = solver.solve_ptr(dA.data_ptr(), n, z.data_ptr(), x3.data_ptr(), allow_noconv=True)
    assert np.isnan(s8.bnorm_inf)


def test_column_independence(mplu, oracle, solver):
    n, nrhs = 2304, 21
    A, Xt, B = system(oracle, n, nrhs, seed=1)
    B[:, 12] = B[:, 5]   # duplicated column
    B[:, 3] = 0.0        # zero column
    X, st, berr = gesv_nrhs(mplu, solver, A, B)
    assert st.converged == 1
    np.testing.assert_array_equal(X[:, 12], X[:, 5])
    assert (X[:, 3] == 0).all() and berr[3] == 0.0
    others = [j for j in range(nrhs) if j != 3]
    assert (berr[others] <= 2 * n * EPS).all()
    perm = np.random.default_rng(7).permutation(nrhs)
    Xp, stp, berrp = gesv_nrhs(mplu, solver, A, B[:, perm])
    np.testing.assert_array_equal(Xp, X[:, perm])
    np.testing.assert_array_equal(berrp, berr[perm])
    assert stp.iters == st.iters


def test_agrees_with_single_vector_solves(mplu, oracle, solver):
    import torch
    n, nrhs = 2304, 10
    A, Xt, B = system(oracle, n, nrhs, seed=2)
    Xt[:, 1] *= 1e-8
    Xt[:, 6] *= 1e8
    B = A @ Xt
    dA, dB = dev(A), dev(B)
    solver.factor_ptr(n, dA.data_ptr(), n, mplu.default_options())
    X = torch.empty(nrhs, n, dtype=torch.float64, device="cuda").t()
    torch.cuda.synchronize()
    st, berr = solver.solve_nrhs_ptr(nrhs, dA.data_ptr(), n, dB.data_ptr(), n, X.data_ptr(), n)
    assert st.converged == 1 and (berr <= 2 * n * EPS).all()
    for j in range(nrhs):
        b = dB[:, j].contiguous()
        x = torch.empty(n, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        sj = solver.solve_ptr(dA.data_ptr(), n, b.data_ptr(), x.data_ptr())
        scale = x.abs().max().item()
        assert (X[:, j] - x).abs().max().item() <= 1e-11 * scale, j
        assert abs(sj.iters - st.iters) <= 1
        np.testing.assert_allclose(X[:, j].cpu().numpy(), Xt[:, j], rtol=0, atol=1e-11 * np.abs(Xt[:, j]).max())


def test_leading_dimensions(mplu, oracle, solver):
    import torch
    n, nrhs, ldb, ldx = 1000, 11, 1003, 1010
    A, Xt, B = system(oracle, n, nrhs, seed=3)
    dA = dev(A)
    Bbuf = torch.full((nrhs, ldb), 7.0, dtype=torch.float64, device="cuda")
    Bbuf[:, :n] = torch.tensor(B.T, device="cuda")
    Xbuf = torch.full((nrhs, ldx), -12345.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    st, berr = solver.gesv_nrhs_ptr(n, nrhs, dA.data_ptr(), n, Bbuf.data_ptr(), ldb, Xbuf.data_ptr(), ldx,
                                    mplu.default_options())
    assert st.converged == 1
    Xh = Xbuf.cpu().numpy()
    assert (Xh[:, n:] == -12345.0).all()  # rows n .. ldx-1 are not written
    np.testing.assert_allclose(Xh[:, :n].T, Xt, rtol=0, atol=1e-11)
    assert (Bbuf[:, n:] == 7.0).all()


def test_lazy_first_touch_is_bit_identical(mplu, oracle, solver):
    n, nrhs = 2304, 5
    A, Xt, B = system(oracle, n, nrhs, seed=4)
    X0, s0, b0 = gesv_nrhs(mplu, solver, A, B, nb=512, lazy_touch=0)
    X1, s1, b1 = gesv_nrhs(mplu, solver, A, B, nb=512, lazy_touch=1)
    assert s0.converged == 1 and s1.converged == 1 and s0.iters == s1.iters
    np.testing.assert_array_equal(X0, X1)


def _spd(oracle, n, kappa):
    return oracle.spd_kappa_matrix(n, kappa, seed=1)


@pytest.mark.parametrize("host", [False, True])
def test_full_precision_fallback(mplu, oracle, solver, host):
    """the three cases of test_full_precision_fallback_like_dsgesv with four right-hand sides"""
    n, nrhs = 512, 4
    rng = np.random.default_rng(3)

    def solve(A, B, allow_noconv=False, **kw):
        if host:
            hA, hB, hX = np.asfortranarray(A), np.asfortranarray(B), np.empty((n, nrhs), order="F")
            st, berr = solver.gesv_host_nrhs_ptr(n, nrhs, hA.ctypes.data, n, hB.ctypes.data, n, hX.ctypes.data, n,
                                                 mplu.default_options(**kw), allow_noconv)
            return hX, st, berr
        return gesv_nrhs(mplu, solver, A, B, allow_noconv, **kw)

    A = rng.standard_normal((n, n)) + 30.0 * np.eye(n)
    A[0, 0] = 0.0
    A[0, 1] = A[1, 0] = 25.0
    Xt = rng.standard_normal((n, nrhs))
    X, st, berr = solve(A, A @ Xt)
    assert st.fp64_fallback == 1 and st.dsgesv_iter == -3 and st.converged == 1
    assert (berr <= 2 * n * EPS).all()
    assert np.abs(X - Xt).max() <= 1e-10 * np.abs(Xt).max()
    A2 = _spd(oracle, n, 1e10)
    X2, st2, berr2 = solve(A2, A2 @ np.ones((n, nrhs)) * np.array([1.0, -2.0, 0.5, 3.0]), max_iters=8, bf16_fallback=1)
    assert st2.fp64_fallback == 1 and st2.dsgesv_iter in (-9, -2, -3) and st2.converged == 1
    assert (berr2 <= 2 * n * EPS).all()
    A3 = oracle.counter_matrix(n, seed=2)
    X3, st3, berr3 = solve(A3, A3 @ Xt)
    assert st3.fp64_fallback == 0 and st3.dsgesv_iter == st3.iters >= 1 and st3.converged == 1
    assert (berr3 <= 2 * n * EPS).all()
    # two columns end in NaN (an Inf and a NaN in b): the stats describe the first of them
    B4 = A @ Xt
    B4[5, 1] = np.inf
    B4[9, 2] = np.nan
    X4, st4, berr4 = solve(A, B4, allow_noconv=True)
    assert st4.fp64_fallback == 1 and st4.dsgesv_iter == -3 and st4.converged == 0
    assert np.isnan(berr4[1]) and np.isnan(berr4[2]) and (berr4[[0, 3]] <= 2 * n * EPS).all()
    assert np.isnan(st4.backward_error) and st4.bnorm_inf == np.inf


def test_fp16_overflow_falls_back_to_bf16(mplu, oracle, solver):
    import torch
    n = 512
    A = _spd(oracle, n, 1e12)
    b = A.sum(axis=1)
    overflowed = False
    try:
        solver.gesv(dev(A), torch.tensor(b, device="cuda"),
                    mplu.default_options(refinement=mplu.REFINE_GMRES, bf16_fallback=0, fp64_fallback=0), allow_noconv=True)
    except mplu.MpluError as e:
        assert e.code == -5
        overflowed = True
    B = np.stack([b, 2.0 * b, -b, 0.5 * b], axis=1)
    X, st, berr = solver.gesv_nrhs(dev(A), dev(B), mplu.default_options(refinement=mplu.REFINE_GMRES), allow_noconv=True)
    assert st.precision_used == (mplu.MPLU_BF16 if overflowed else mplu.MPLU_FP16)
    assert np.isfinite(X.cpu().numpy()).all()


def test_gmres_refinement(mplu, oracle, solver):
    n, nrhs = 1024, 3
    A = _spd(oracle, n, 1e7)
    Xt = np.random.default_rng(5).standard_normal((n, nrhs))
    X, st, berr = gesv_nrhs(mplu, solver, A, A @ Xt, refinement=mplu.REFINE_GMRES, fp64_fallback=0)
    assert st.converged == 1 and st.gmres_iters >= st.iters >= 1
    assert (berr <= np.sqrt(n) * EPS).all(), berr  # each column met the stopping rule


@pytest.mark.parametrize("pinned", [False, True])
def test_host_variant_matches_device(mplu, oracle, pinned):
    import torch
    n, nb, nrhs = 2304, 512, 5
    A, Xt, B = system(oracle, n, nrhs, seed=6)
    A = np.asfortranarray(A)
    s = mplu.Solver(0)
    try:
        Xd, sd, bd = s.gesv_nrhs(dev(A), dev(B), mplu.default_options(nb=nb, update_pair=0))
        Xd = Xd.cpu().numpy()
        if pinned:
            hA = torch.empty(n, n, dtype=torch.float64, pin_memory=True)
            hA.copy_(torch.from_numpy(np.ascontiguousarray(A.T)))
            hB = torch.empty(nrhs, n, dtype=torch.float64, pin_memory=True)
            hB.copy_(torch.from_numpy(np.ascontiguousarray(B.T)))
            hX = torch.empty(nrhs, n, dtype=torch.float64, pin_memory=True)
            pA, pB, pX = hA.data_ptr(), hB.data_ptr(), hX.data_ptr()
            read = lambda: hX.numpy().T.copy()  # noqa: E731
        else:
            Bf, Xf = np.asfortranarray(B), np.empty((n, nrhs), order="F")
            pA, pB, pX = A.ctypes.data, Bf.ctypes.data, Xf.ctypes.data
            read = lambda: Xf.copy()  # noqa: E731
        for stream_host in (1, 0):
            st, berr = s.gesv_host_nrhs_ptr(n, nrhs, pA, n, pB, n, pX, n,
                                            mplu.default_options(nb=nb, stream_host=stream_host, update_pair=0))
            assert st.converged == 1 and st.h2d_ms > 0 and st.iters == sd.iters
            np.testing.assert_array_equal(read(), Xd)
            np.testing.assert_allclose(berr, bd, rtol=1e-12)  # ||A|| is summed in another order by the streamed path
    finally:
        s.close()


def test_argument_errors_leave_x_untouched(mplu, oracle, solver):
    import torch
    lib = mplu.load_library()
    n, nrhs = 256, 3
    A, Xt, B = system(oracle, n, nrhs)
    dA, dB = dev(A), dev(B)
    X = torch.full((nrhs, n), 5.0, dtype=torch.float64, device="cuda")
    solver.factor_ptr(n, dA.data_ptr(), n, mplu.default_options())
    torch.cuda.synchronize()
    o = mplu.default_options()
    a, b, x = dA.data_ptr(), dB.data_ptr(), X.data_ptr()
    ctx = solver._ctx
    calls = [
        lambda: lib.mplu_gesv_device_nrhs(ctx, n, 0, a, n, b, n, x, n, C.byref(o), None, None),      # nrhs < 1
        lambda: lib.mplu_gesv_device_nrhs(ctx, n, nrhs, a, n, b, n - 1, x, n, C.byref(o), None, None),  # ldb < n
        lambda: lib.mplu_gesv_device_nrhs(ctx, n, nrhs, a, n, b, n, x, n - 1, C.byref(o), None, None),  # ldx < n
        lambda: lib.mplu_gesv_device_nrhs(ctx, n, nrhs, None, n, b, n, x, n, C.byref(o), None, None),
        lambda: lib.mplu_gesv_device_nrhs(ctx, n, nrhs, a, n, None, n, x, n, C.byref(o), None, None),
        lambda: lib.mplu_gesv_device_nrhs(ctx, n, nrhs, a, n, b, n, None, n, C.byref(o), None, None),
        lambda: lib.mplu_gesv_device_nrhs(None, n, nrhs, a, n, b, n, x, n, C.byref(o), None, None),
        lambda: lib.mplu_gesv_device_nrhs(ctx, n, nrhs, a, n, x, n, x + 8 * 5, n, C.byref(o), None, None),  # X overlaps B
        lambda: lib.mplu_solve_device_nrhs(ctx, 0, a, n, b, n, x, n, None, None),
        lambda: lib.mplu_solve_device_nrhs(ctx, nrhs, a, n, b, n - 1, x, n, None, None),
        lambda: lib.mplu_solve_device_nrhs(ctx, nrhs, a, n, b, n, x, n - 1, None, None),
        lambda: lib.mplu_solve_device_nrhs(ctx, nrhs, a, n, b, n, None, n, None, None),
        lambda: lib.mplu_solve_device_nrhs(ctx, nrhs, a, n, b, n, b + 8, n, None, None),
    ]
    hA, hB, hX = np.asfortranarray(A), np.asfortranarray(B), np.full((n, nrhs), 5.0, order="F")
    calls += [
        lambda: lib.mplu_gesv_host_nrhs(ctx, n, 0, hA.ctypes.data, n, hB.ctypes.data, n, hX.ctypes.data, n, C.byref(o), None, None),
        lambda: lib.mplu_gesv_host_nrhs(ctx, n, nrhs, hA.ctypes.data, n, hB.ctypes.data, n - 1, hX.ctypes.data, n, C.byref(o), None, None),
        lambda: lib.mplu_gesv_host_nrhs(ctx, n, nrhs, hA.ctypes.data, n, hB.ctypes.data, n, None, n, C.byref(o), None, None),
        lambda: lib.mplu_gesv_host_nrhs(ctx, n, nrhs, hA.ctypes.data, n, hB.ctypes.data, n, hB.ctypes.data + 8, n, C.byref(o), None, None),
    ]
    for i, call in enumerate(calls):
        assert call() == -1, i
    torch.cuda.synchronize()
    assert (X == 5.0).all() and (hX == 5.0).all()
    assert torch.equal(dB, dev(B))
