"""GPU tests of the equilibration (mplu_options::equilibrate, csrc/equil.cu): the device's dgeequb scales and dlaqge
decision against the host reference, bit-identity with equilibrate = 0 where no scale is applied, the factors of
diag(r) A diag(c) where scales are, and badly scaled systems that stay on the fp16 path."""
import math

import numpy as np
import pytest

import equilibrate_ref as eq

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps / 2
U16 = 2.0 ** -11
TIMING = {"factor_ms", "solve_ms", "total_ms", "h2d_ms", "d2h_ms", "trailing_ms"}
EQUIL_LAUNCHES = 4  # row pass, row scales, column pass, decision


def cm(t):
    return t.t().contiguous().t()


def with_lda(A, lda, fill=1e300):
    """column-major copy of A with leading dimension lda; the rows n .. lda-1 hold `fill` (never read)"""
    import torch
    n, m = A.shape
    buf = torch.full((m, lda), fill, dtype=torch.float64, device="cuda")
    view = buf.t()[:n]
    view.copy_(A)
    return view


def pow2(n, spread, g):
    import torch
    return 2.0 ** torch.randint(-spread, spread + 1, (n,), generator=g, device="cuda").double()


def scaled(A0, row_spread, col_spread, seed):
    """diag(d1) A0 diag(d2), d1 / d2 seeded powers of two in 2^+-spread (exact), column-major"""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = A0.shape[0]
    d1 = pow2(n, row_spread, g) if row_spread else torch.ones(n, dtype=torch.float64, device="cuda")
    d2 = pow2(n, col_spread, g) if col_spread else torch.ones(n, dtype=torch.float64, device="cuda")
    return cm(d1[:, None] * A0 * d2[None, :])


def randn_dominant(n, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g) + 2 * math.sqrt(n) * torch.eye(
        n, dtype=torch.float64, device="cuda")


def rhs(A, seed, k=None):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed + 1000)
    x = torch.randn(A.shape[0], *(() if k is None else (k,)), dtype=torch.float64, device="cuda", generator=g)
    return (A @ x).contiguous() if k is None else cm(A @ x)


def plain(d):
    return {k: v for k, v in d.items() if k not in TIMING}


@pytest.mark.parametrize("n", [1000, 2304, 4096])
def test_scales_equal_the_reference(mplu, solver, n):
    import torch
    cases = {}
    counter, _b = mplu.generate(n)
    cases["counter"] = (counter, 0)
    A0 = randn_dominant(n, seed=n)
    cases["rows"] = (scaled(A0, 10, 0, seed=1), None)
    # columns only: a small diagonal, so that every row's maximum comes from the widest columns (ROWCND >= 1/2)
    cases["cols"] = (scaled(A0 - (2 * math.sqrt(n) - 4) * torch.eye(n, dtype=torch.float64, device="cuda"), 0, 10, seed=2), 2)
    cases["both"] = (scaled(A0, 10, 10, seed=3), 3)
    z = A0.clone()
    z[n // 3, :] = 0.0
    cases["zero_row"] = (cm(z), 0)
    nan = A0.clone()
    nan[n // 2, n // 5] = float("nan")
    cases["nan"] = (cm(nan), 0)
    for name, (A, expect) in cases.items():
        dA = with_lda(A, n + 3)
        torch.cuda.synchronize()
        solver.factor_ptr(n, dA.data_ptr(), n + 3, mplu.default_options(equilibrate=1))
        equed, r, c = solver.equilibration(n)
        e_ref, r_ref, c_ref = eq.equilibrate(A.cpu().numpy())
        if expect is not None:
            assert e_ref == expect, name
        else:
            assert e_ref in (1, 3), name
        assert equed == e_ref, name
        np.testing.assert_array_equal(r.cpu().numpy(), r_ref, err_msg=name)
        np.testing.assert_array_equal(c.cpu().numpy(), c_ref, err_msg=name)


def test_no_scale_applied_changes_nothing(mplu, solver):
    """EQUED = N: factors, X and every non-timing statistic of equilibrate = 0, bit for bit (lazy first touch, nrhs 1 and
    17, host path); the launch count grows by the four equilibration launches"""
    import torch
    n = 2304  # a multiple of 128: the default lazy first touch runs
    A, b = mplu.generate(n)
    out = {}
    for e in (0, 1):
        x, st = solver.gesv(A, b, mplu.default_options(equilibrate=e))
        out[e] = (x, st.as_dict(), solver.factors(n))
    assert out[1][1]["equed"] == 0 and out[1][1]["converged"] == 1
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][2], out[1][2])
    s0, s1 = plain(out[0][1]), plain(out[1][1])
    assert s1.pop("kernel_launches") == s0.pop("kernel_launches") + EQUIL_LAUNCHES
    assert s0 == s1
    B = rhs(A, seed=5, k=17)
    X0, t0, b0 = solver.gesv_nrhs(A, B, mplu.default_options(equilibrate=0))
    X1, t1, b1 = solver.gesv_nrhs(A, B, mplu.default_options(equilibrate=1))
    assert torch.equal(X0, X1) and np.array_equal(b0, b1)
    d0, d1 = plain(t0.as_dict()), plain(t1.as_dict())
    assert d1.pop("kernel_launches") == d0.pop("kernel_launches") + EQUIL_LAUNCHES and d0 == d1
    hA, hb = np.asfortranarray(A.cpu().numpy()), b.cpu().numpy()
    hx = {e: np.empty(n) for e in (0, 1)}
    hs = {e: solver.gesv_host_ptr(n, hA.ctypes.data, n, hb.ctypes.data, hx[e].ctypes.data,
                                  mplu.default_options(equilibrate=e, stream_host=0)).as_dict() for e in (0, 1)}
    np.testing.assert_array_equal(hx[0], hx[1])
    h0, h1 = plain(hs[0]), plain(hs[1])
    assert h1.pop("kernel_launches") == h0.pop("kernel_launches") + EQUIL_LAUNCHES and h0 == h1


def test_scaled_factors_are_those_of_the_scaled_matrix(mplu, oracle, solver):
    import torch
    n = 2304
    A = scaled(randn_dominant(n, seed=11), 10, 10, seed=12)
    b = rhs(A, seed=13)
    x, st = solver.gesv(A, b, mplu.default_options(equilibrate=1))
    assert st.equed == 3 and st.converged == 1 and st.fp64_fallback == 0
    LU = solver.factors(n)
    equed, r, c = solver.equilibration(n)
    assert equed == 3
    As = cm(r[:, None] * A * c[None, :])  # exact: powers of two
    ref = mplu.Solver(0)
    try:
        ref.factor_ptr(n, As.data_ptr(), n, mplu.default_options(lazy_touch=0, tol=1.0))
        assert torch.equal(ref.factors(n), LU)
        rho = oracle.factor_tile_ratio(As, LU)
        assert rho.max() <= 3 * U16, rho.max() / U16
        # the unrefined first solve (tol = 1 stops after it) is c o (the plain first solve of A' y = r o b)
        x1, s1 = solver.gesv(A, b, mplu.default_options(equilibrate=1, tol=1.0))
        assert s1.iters == 0
        y = torch.empty(n, dtype=torch.float64, device="cuda")
        rb = (r * b).contiguous()
        torch.cuda.synchronize()
        ref.solve_ptr(As.data_ptr(), n, rb.data_ptr(), y.data_ptr(), allow_noconv=True)
        assert torch.equal(x1, c * y)
    finally:
        ref.close()
    # ||A||_inf of the caller's matrix, not of the scaled one (summed in another order than torch's)
    assert abs(st.anorm_inf - A.abs().sum(dim=1).max().item()) <= 1e-14 * st.anorm_inf


def _fp16_fast_path_case(mplu, solver, record_property, label, A, b, opts_eq, opts_plain):
    import time
    import torch
    torch.cuda.synchronize()
    t = time.perf_counter()
    x0, s0 = solver.gesv(A, b, opts_plain, allow_noconv=True)
    record_property(f"{label}_equilibrate0", dict(status_bits=s0.status_bits, precision_used=s0.precision_used,
                                                   dsgesv_iter=s0.dsgesv_iter, fp64_fallback=s0.fp64_fallback,
                                                   total_ms=round(s0.total_ms, 2),
                                                   wall_ms=round(1e3 * (time.perf_counter() - t), 2)))
    x1, s1 = solver.gesv(A, b, opts_eq)
    record_property(f"{label}_equilibrate1", dict(equed=s1.equed, iters=s1.iters, total_ms=round(s1.total_ms, 2)))
    return s0, s1


def test_badly_scaled_system_stays_on_the_fp16_path(mplu, solver, record_property):
    n = 4096
    A0 = randn_dominant(n, seed=21)
    _, base = solver.gesv(cm(A0), rhs(A0, seed=22), mplu.default_options())
    A = scaled(A0, 10, 10, seed=23)
    s0, s = _fp16_fast_path_case(mplu, solver, record_property, "randn_2pm10", A, rhs(A, seed=24),
                                 mplu.default_options(equilibrate=1), mplu.default_options())
    assert s0.precision_used == mplu.MPLU_BF16  # without equilibration: fp16 overflow, the factorization redone in bf16
    assert s.converged == 1 and s.precision_used == mplu.MPLU_FP16 and s.status_bits == 0 and s.fp64_fallback == 0
    assert s.equed != 0 and s.iters <= base.iters + 1, (s.iters, base.iters)


def test_scaled_kappa_1e6_converges_in_fp16(mplu, solver, record_property):
    n = 16384
    A = scaled(mplu.generate_spd(n, 1e6, seed=1), 6, 6, seed=31)
    s0, s = _fp16_fast_path_case(mplu, solver, record_property, "spd1e6_2pm6", A, rhs(A, seed=32),
                                 mplu.default_options(equilibrate=1), mplu.default_options())
    # without equilibration: fp16 overflow -> bf16 -> no convergence -> the fp64 fallback
    assert s0.precision_used == mplu.MPLU_BF16 and s0.fp64_fallback == 1
    assert s.converged == 1 and s.precision_used == mplu.MPLU_FP16 and s.fp64_fallback == 0 and s.equed != 0


def test_several_right_hand_sides(mplu, solver):
    import torch
    n, k, ldb, ldx = 2304, 17, 2311, 2320
    A = scaled(randn_dominant(n, seed=41), 8, 8, seed=42)
    B = rhs(A, seed=43, k=k)
    opts = mplu.default_options(equilibrate=1)

    def solve_block(Bm):
        Bbuf = with_lda(Bm, ldb, fill=7.0)
        Xbuf = with_lda(torch.zeros_like(Bm), ldx, fill=-12345.0)
        torch.cuda.synchronize()
        st, berr = solver.gesv_nrhs_ptr(n, k, A.data_ptr(), A.stride(1), Bbuf.data_ptr(), ldb, Xbuf.data_ptr(), ldx, opts)
        return Xbuf.clone(), st, berr

    X, st, berr = solve_block(B)
    assert st.converged == 1 and st.equed != 0 and (berr <= 2 * n * EPS).all(), berr
    for j in (0, 5, 16):
        x, sj = solver.gesv(A, B[:, j].contiguous(), opts)
        assert sj.equed == st.equed
        assert (X[:, j] - x).abs().max().item() <= 1e-11 * x.abs().max().item(), j
        assert abs(sj.backward_error - berr[j]) <= 0.5 * max(berr[j], sj.backward_error) + n * EPS
    perm = torch.tensor(np.random.default_rng(7).permutation(k), device="cuda")
    Xp, stp, berrp = solve_block(cm(B[:, perm]))
    assert torch.equal(Xp, X[:, perm]) and np.array_equal(berrp, berr[perm.cpu().numpy()])


def test_gmres_refinement_with_equilibration(mplu, solver, record_property):
    n = 16384
    A = scaled(mplu.generate_spd(n, 1e7, seed=2), 6, 6, seed=51)
    x, s = solver.gesv(A, rhs(A, seed=52), mplu.default_options(equilibrate=1, refinement=mplu.REFINE_GMRES))
    record_property("gmres", dict(equed=s.equed, iters=s.iters, gmres_iters=s.gmres_iters, total_ms=round(s.total_ms, 2)))
    assert s.converged == 1 and s.fp64_fallback == 0 and s.equed != 0


def test_factor_reuse_keeps_the_scales(mplu, solver):
    import torch
    n = 2304
    A = scaled(randn_dominant(n, seed=61), 10, 10, seed=62)
    b1, b2 = rhs(A, seed=63), rhs(A, seed=64)
    opts = mplu.default_options(equilibrate=1)
    xg, sg = solver.gesv(A, b1, opts)
    solver.factor_ptr(n, A.data_ptr(), n, opts)
    xs = []
    for b in (b1, b2):
        x = torch.empty(n, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        st = solver.solve_ptr(A.data_ptr(), n, b.data_ptr(), x.data_ptr())
        assert st.converged == 1 and st.equed == sg.equed != 0
        xs.append(x)
    assert torch.equal(xs[0], xg)
    # a well-scaled matrix next: EQUED back to N, and its solve is a fresh context's
    C, bc = mplu.generate(n)
    solver.factor_ptr(n, C.data_ptr(), n, opts)
    assert solver.equilibration(n)[0] == 0
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    st = solver.solve_ptr(C.data_ptr(), n, bc.data_ptr(), x.data_ptr())
    fresh = mplu.Solver(0)
    try:
        fresh.factor_ptr(n, C.data_ptr(), n, opts)
        y = torch.empty(n, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        sf = fresh.solve_ptr(C.data_ptr(), n, bc.data_ptr(), y.data_ptr())
    finally:
        fresh.close()
    assert st.equed == 0 and torch.equal(x, y) and st.iters == sf.iters


def test_host_path_matches_the_device_path(mplu, solver):
    n = 2304
    A = scaled(randn_dominant(n, seed=71), 10, 10, seed=72)
    b = rhs(A, seed=73)
    opts = mplu.default_options(equilibrate=1, stream_host=1)
    xd, sd = solver.gesv(A, b, opts)
    hA, hb, hx = np.asfortranarray(A.cpu().numpy()), b.cpu().numpy(), np.empty(n)
    sh = solver.gesv_host_ptr(n, hA.ctypes.data, n, hb.ctypes.data, hx.ctypes.data, opts)
    np.testing.assert_array_equal(hx, xd.cpu().numpy())
    assert sd.equed == sh.equed != 0
    assert plain(sd.as_dict()) == plain(sh.as_dict())


def test_bf16_with_equilibration(mplu, solver):
    n = 4096
    A = scaled(randn_dominant(n, seed=21), 10, 10, seed=23)
    x, s = solver.gesv(A, rhs(A, seed=24), mplu.default_options(equilibrate=1, precision=mplu.MPLU_BF16))
    assert s.converged == 1 and s.precision_used == mplu.MPLU_BF16 and s.fp64_fallback == 0 and s.equed != 0


def test_argument_errors(mplu, solver):
    import torch
    n = 1000
    A, b = mplu.generate(n)
    x = torch.zeros(n, dtype=torch.float64, device="cuda")
    for bad in (2, -1):
        opts = mplu.default_options(equilibrate=bad)
        with pytest.raises(mplu.MpluError) as e:
            solver.factor_ptr(n, A.data_ptr(), n, opts)
        assert e.value.code == -1
        with pytest.raises(mplu.MpluError) as e:
            solver.gesv(A, b, opts)
        assert e.value.code == -1
        with pytest.raises(mplu.MpluError) as e:
            solver.gesv_nrhs(A, cm(b.reshape(n, 1)), opts)
        assert e.value.code == -1
        hA, hb, hx = np.asfortranarray(A.cpu().numpy()), b.cpu().numpy(), np.empty(n)
        with pytest.raises(mplu.MpluError) as e:
            solver.gesv_host_ptr(n, hA.ctypes.data, n, hb.ctypes.data, hx.ctypes.data, opts)
        assert e.value.code == -1
    assert (x == 0).all()
    d = mplu.DistSolver(0, 1, 1)
    try:
        As, bs = d.generate(512, 128)
        with pytest.raises(mplu.MpluError) as e:
            d.gesv(512, 128, As, bs, mplu.default_options(equilibrate=1))
        assert e.value.code == -1
    finally:
        d.close()
    fresh = mplu.Solver(0)
    try:
        with pytest.raises(mplu.MpluError) as e:
            fresh.equilibration(n)
        assert e.value.code == -3
    finally:
        fresh.close()
