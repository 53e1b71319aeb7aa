"""GPU parity tests of the hot path through the C ABI: no-pivot mixed-precision LU + fp64 iterative refinement vs
the oracle, host LAPACK and the golden outputs of the unmodified reference."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from test_gpu_reference import check_agreement, check_factors

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps / 2  # unit roundoff


def cm(t):
    return t.t().contiguous().t()


def run(mplu, solver, A, b, **kw):
    import torch
    dA = cm(torch.tensor(A, dtype=torch.float64, device="cuda"))
    db = torch.tensor(b, dtype=torch.float64, device="cuda")
    x, st = solver.gesv(dA, db, mplu.default_options(**kw))
    return x.cpu().numpy(), st.as_dict()


@pytest.mark.parametrize("n", [1024])
@pytest.mark.parametrize("precision", [0, 1])
def test_config1_n1024_vs_lapack_and_oracle(mplu, oracle, solver, record_property, n, precision):
    """BASELINE.json configs[0]: n=1024 diagonally dominant, no-pivot LU + IR single RHS vs host dgetrf/dgetrs."""
    A = oracle.counter_matrix(n, seed=1)
    b = A.sum(axis=1)
    x, st = run(mplu, solver, A, b, precision=precision)
    x_ref, lu_ref, piv = oracle.lapack_gesv(A, b)
    assert np.array_equal(piv, np.arange(n))
    emu = oracle.refine(A, b, oracle.lu_mixed_emulated(A, 128, bf16=bool(precision)))
    assert st["converged"] == 1 and st["status_bits"] == 0
    assert st["iters"] <= emu["iters"]  # same or fewer refinement iterations than the emulated algorithm
    assert st["backward_error"] <= 2 * n * EPS  # north_star: about 1e-15 * n
    assert st["backward_error"] <= 4 * max(emu["backward_error"], EPS)
    np.testing.assert_allclose(x, x_ref, rtol=0, atol=1e-12)
    # LU factors vs the fp64 no-pivot LU (= what the reference returns on this input), stated fp16/bf16 tolerance:
    # relative to max|U| a few unit roundoffs of the 16-bit type per 128-wide block step
    LU = solver.factors(n).cpu().numpy()
    u16 = 2.0 ** -11 if precision == 0 else 2.0 ** -8
    assert np.abs(np.triu(LU) - np.triu(lu_ref)).max() <= 0.02 * u16 * np.abs(lu_ref).max()
    assert np.abs(np.tril(LU, -1) - np.tril(lu_ref, -1)).max() <= 2 * u16 * np.abs(np.tril(lu_ref, -1)).max()
    check_factors(oracle, record_property, A, LU, precision)


@pytest.mark.parametrize("n", [128, 256])
def test_factors_vs_golden_reference_output(mplu, oracle, solver, n):
    """Same generated input as the golden run of the unmodified reference MPF(): identity pivots there, so its output
    is the fp64 no-pivot LU our low-precision factors approximate."""
    g = np.load(os.path.join(GOLDEN, f"ref_mpf_dd_n{n}.npz"))
    assert np.array_equal(g["ipiv"], np.arange(1, n + 1))
    A = oracle.counter_matrix(n, seed=int(g["seed"]))
    x, st = run(mplu, solver, A, A.sum(axis=1))
    LU = solver.factors(n).cpu().numpy()
    ref = g["LU"]
    assert np.abs(np.triu(LU - ref)).max() <= 0.02 * 2.0 ** -11 * np.abs(ref).max()
    assert np.abs(np.tril(LU - ref, -1)).max() <= 2 * 2.0 ** -11 * np.abs(np.tril(ref, -1)).max()
    assert st["converged"] == 1 and np.abs(x - 1).max() < 1e-12


@pytest.mark.parametrize("n", [1, 2, 3, 127, 128, 129, 1000, 1537])
def test_ragged_sizes(mplu, oracle, solver, n):
    A = oracle.counter_matrix(n, seed=2)
    b = A @ np.linspace(-1, 1, n)
    x, st = run(mplu, solver, A, b, nb=512)
    assert st["converged"] == 1 and st["status_bits"] == 0  # the identity padding must not raise the overflow bit
    np.testing.assert_allclose(x, np.linspace(-1, 1, n), rtol=0, atol=1e-11)


@pytest.mark.parametrize("nb", [128, 256, 1024, 2048])
@pytest.mark.parametrize("variant", [0, 1])
def test_block_sizes_and_gemm_variants_agree(mplu, oracle, solver, record_property, nb, variant):
    n = 2304
    A = oracle.counter_matrix(n, seed=4)
    b = A.sum(axis=1)
    x, st = run(mplu, solver, A, b, nb=nb, gemm_variant=variant)
    assert st["converged"] == 1 and st["iters"] <= 3
    assert st["backward_error"] <= 2 * n * EPS
    assert np.abs(x - 1).max() < 1e-11
    check_factors(oracle, record_property, A, solver.factors(n), 0)


def test_solve_reuses_factors_for_new_rhs(mplu, oracle, solver):
    import torch
    n = 1024
    A = oracle.counter_matrix(n, seed=9)
    dA = cm(torch.tensor(A, device="cuda"))
    torch.cuda.synchronize()
    solver.factor_ptr(n, dA.data_ptr(), dA.stride(1), mplu.default_options())
    rng = np.random.default_rng(0)
    for _ in range(2):
        xt = rng.standard_normal(n)
        db = torch.tensor(A @ xt, device="cuda")
        dx = torch.empty(n, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        st = solver.solve_ptr(dA.data_ptr(), dA.stride(1), db.data_ptr(), dx.data_ptr())
        assert st.converged == 1
        np.testing.assert_allclose(dx.cpu().numpy(), xt, rtol=0, atol=1e-11)


def test_host_buffer_entry_point(mplu, oracle, solver):
    n = 640
    A = np.asfortranarray(oracle.counter_matrix(n, seed=11))
    b = A.sum(axis=1)
    x = np.empty(n)
    st = solver.gesv_host_ptr(n, A.ctypes.data, n, b.ctypes.data, x.ctypes.data, mplu.default_options())
    assert st.converged == 1 and st.h2d_ms > 0
    np.testing.assert_allclose(x, 1.0, rtol=0, atol=1e-12)


@pytest.mark.parametrize("n,nb", [(2304, 512), (1000, 256), (4096, 1024)])
@pytest.mark.parametrize("pinned", [False, True])
def test_streamed_host_path_gives_bit_identical_factors(mplu, oracle, record_property, n, nb, pinned):
    """mplu_gesv_host factors left-looking, block column by block column, while A is still arriving over PCIe: the same
    products in the same order as the device schedule, hence the same factors bit for bit and the same solution;
    stream_host=0 (copy first, then the device schedule) is the comparison."""
    import torch
    A = np.asfortranarray(oracle.counter_matrix(n, seed=21))
    b = A.sum(axis=1)
    if pinned:
        hA = torch.empty(n, n, dtype=torch.float64, pin_memory=True)
        hA.copy_(torch.from_numpy(np.ascontiguousarray(A.T)))  # contiguous storage of A^T = column-major A
        hb = torch.from_numpy(b.copy()).pin_memory()
        hx = torch.empty(n, dtype=torch.float64, pin_memory=True)
        pA, pb, px = hA.data_ptr(), hb.data_ptr(), hx.data_ptr()
    else:
        x = np.empty(n)
        pA, pb, px = A.ctypes.data, b.ctypes.data, x.ctypes.data
    s = mplu.Solver(0)
    try:
        outs = []
        for stream_host in (1, 0, 1):
            st = s.gesv_host_ptr(n, pA, n, pb, px, mplu.default_options(nb=nb, stream_host=stream_host, update_pair=0))
            assert st.converged == 1 and st.status_bits == 0 and st.h2d_ms > 0
            xs = hx.numpy().copy() if pinned else x.copy()
            outs.append((s.factors(n).clone(), xs, st.iters))
        for LU, xs, it in outs[1:]:
            assert torch.equal(LU, outs[0][0])
            assert it == outs[0][2]
            np.testing.assert_array_equal(xs, outs[0][1])
        np.testing.assert_allclose(outs[0][1], 1.0, rtol=0, atol=1e-11)
        check_factors(oracle, record_property, A, outs[0][0], 0)
    finally:
        s.close()


def test_streamed_host_path_scale_overflow_is_redone(mplu, oracle, record_property):
    """The fp16 scale of the streamed path comes from the first block column; a later block column far outside that
    range must end in a correct solve (redo with the global scale), not in a silent overflow."""
    n, nb = 1536, 512
    A = np.asfortranarray(oracle.counter_matrix(n, seed=5))
    A[:, nb:] *= 64.0  # later block columns 2^6 larger: (2^10, 2^11] * 2^6 leaves the fp16 range
    b = A.sum(axis=1)
    x = np.empty(n)
    s = mplu.Solver(0)
    try:
        st = s.gesv_host_ptr(n, A.ctypes.data, n, b.ctypes.data, x.ctypes.data, mplu.default_options(nb=nb))
        assert st.converged == 1
        np.testing.assert_allclose(x, 1.0, rtol=0, atol=1e-10)
        if st.status_bits == 0:  # an overflow that did not spoil the solve keeps its factors on purpose
            check_factors(oracle, record_property, A, s.factors(n), 0)
    finally:
        s.close()


def test_early_scale_option(mplu, oracle, solver, record_property):
    """early_scale=1 (left-looking schedule): the first touch overlaps the first diagonal tile, so the fp16 scale comes
    from the first block column.  Later block columns 2^6 larger leave the fp16 range under it: the overflow is
    reported (status bit 0) and, had it spoiled the solve, redone with the global scale; the answer must be right
    either way and agree with the global-scale run."""
    n, nb = 1536, 512
    A = oracle.counter_matrix(n, seed=5)
    A[:, nb:] *= 64.0
    b = A.sum(axis=1)
    x1, st1 = run(mplu, solver, A, b, nb=nb, early_scale=1, lazy_touch=0)  # (the lazy first touch has its own test)
    if st1["status_bits"] == 0:  # an overflow that did not spoil the solve keeps its factors on purpose
        check_factors(oracle, record_property, A, solver.factors(n), 0, "rho_early")
    x0, st0 = run(mplu, solver, A, b, nb=nb, early_scale=0, lazy_touch=0)
    assert st0["converged"] == 1 and st0["status_bits"] == 0 and st0["precision_used"] == mplu.MPLU_FP16
    check_factors(oracle, record_property, A, solver.factors(n), 0, "rho_global")
    assert st1["converged"] == 1
    np.testing.assert_allclose(x1, x0, rtol=0, atol=1e-11)
    np.testing.assert_allclose(x1, 1.0, rtol=0, atol=1e-10)
    # same matrix without the jump in magnitude: both scale choices are the same power of two, same factors
    A2 = oracle.counter_matrix(n, seed=5)
    xa, sa = run(mplu, solver, A2, A2.sum(axis=1), nb=nb, early_scale=1, lazy_touch=0)
    xb, sb = run(mplu, solver, A2, A2.sum(axis=1), nb=nb, early_scale=0, lazy_touch=0)
    assert sa["status_bits"] == 0 and sb["status_bits"] == 0
    np.testing.assert_array_equal(xa, xb)


def test_spd_kappa_small(mplu, oracle, solver):
    """config 5 at test size: SPD, kappa = 1e2, classic IR converges (oracle emulation: <= 4 iterations)."""
    n = 1024
    A = oracle.spd_kappa_matrix(n, 1e2, seed=3)
    xt = np.ones(n)
    b = A @ xt
    emu = oracle.refine(A, b, oracle.lu_mixed_emulated(A, 128))
    x, st = run(mplu, solver, A, b)
    assert st["converged"] == 1 and st["iters"] <= emu["iters"] + 1
    assert st["backward_error"] <= 2 * n * EPS


def test_zero_pivot_and_nonconvergence_are_reported(mplu, solver):
    n = 256
    A = np.eye(n)
    A[0, 0] = 0.0
    A[0, 1] = A[1, 0] = 1.0  # needs pivoting: no-pivot LU hits an exact zero pivot
    with pytest.raises(mplu.MpluError) as e:
        run(mplu, solver, A, np.ones(n), fp64_fallback=0)
    assert e.value.code in (-6, -7, -5)


@pytest.mark.parametrize("host", [False, True])
def test_full_precision_fallback_like_dsgesv(mplu, oracle, solver, host):
    """LAPACK dsgesv semantics (opts.fp64_fallback = 1, the default): a solve the low-precision factors cannot deliver is
    redone with an fp64 LU with row pivoting -- the reference's MPF algorithm (/root/reference/MPF.cu:100-241: fp16 pivot
    discovery, fp64 elimination) on the device copy -- and fp64 solves; ITER < 0 says why (dsgesv.f).  Three causes: an
    exact zero pivot without pivoting (-3), classic refinement stalling on an ill-conditioned matrix (-(max_iters + 1)),
    and the healthy case for comparison (ITER = iterations >= 0, no fallback)."""
    import torch
    n = 512
    rng = np.random.default_rng(3)
    # 1. needs pivoting: zero leading pivot, otherwise well conditioned
    A = rng.standard_normal((n, n)) + 30.0 * np.eye(n)
    A[0, 0] = 0.0
    A[0, 1] = A[1, 0] = 25.0
    x_true = rng.standard_normal(n)
    b = A @ x_true
    def solve(A, b, **kw):
        if host:  # pageable host buffers through mplu_gesv_host
            hA, hb, hx = np.asfortranarray(A), np.ascontiguousarray(b), np.empty(len(b))
            st = solver.gesv_host_ptr(len(b), hA.ctypes.data, len(b), hb.ctypes.data, hx.ctypes.data, mplu.default_options(**kw))
            return hx, st
        dA = cm(torch.tensor(A, dtype=torch.float64, device="cuda"))
        x, st = solver.gesv(dA, torch.tensor(b, dtype=torch.float64, device="cuda"), mplu.default_options(**kw))
        return x.cpu().numpy(), st
    x, st = solve(A, b)
    assert st.fp64_fallback == 1 and st.dsgesv_iter == -3 and st.converged == 1
    assert st.backward_error <= 2 * n * EPS
    assert np.abs(x - x_true).max() <= 1e-10 * np.abs(x_true).max()
    # 2. kappa = 1e10: 16-bit factors are no contraction for classic refinement
    A2, b2 = _spd(oracle, n, 1e10)
    x2, st2 = solve(A2, b2, max_iters=8, bf16_fallback=1)
    assert st2.fp64_fallback == 1 and st2.dsgesv_iter in (-9, -2, -3) and st2.converged == 1
    assert st2.backward_error <= 2 * n * EPS
    # 3. healthy matrix: no fallback, ITER counts the refinement iterations
    A3 = oracle.counter_matrix(n, seed=2)
    x3, st3 = solve(A3, A3.sum(axis=1))
    assert st3.fp64_fallback == 0 and st3.dsgesv_iter == st3.iters >= 1 and st3.converged == 1


def test_full_size_properties_n32768(mplu, solver):
    """BASELINE.json configs[2] through size-independent properties: refined solution reproduces x_true = 1,
    fp64 normwise backward error about 1e-15*n or better, in at most 3 refinement iterations."""
    n = 32768
    A, b = mplu.generate(n, seed=1)
    x, st = solver.gesv(A, b, mplu.default_options())
    d = st.as_dict()
    assert d["converged"] == 1 and d["status_bits"] == 0 and d["iters"] <= 3
    assert d["backward_error"] <= 1e-15 * n
    assert (x - 1).abs().max().item() <= 1e-11
    # the backward error recomputed independently (torch fp64 GEMV) agrees with the solver's own figure
    import torch
    r = b - A @ x
    be = (r.abs().max() / (A.abs().sum(dim=1).max() * x.abs().max() + b.abs().max())).item()
    assert be <= 1e-15 * n and be <= 8 * d["backward_error"] + 1e-15  # both are rounding noise of an n-term fp64 sum
    # linearity: same factors, right-hand side 2b - 3e_0 -> 2x - 3 A^-1 e_0, checked through its residual
    b2 = 2.0 * b
    b2[0] -= 3.0
    x2 = torch.empty_like(x)
    st2 = solver.solve_ptr(A.data_ptr(), A.stride(1), b2.data_ptr(), x2.data_ptr())
    r2 = b2 - A @ x2
    assert st2.converged == 1
    assert (r2.abs().max() / (A.abs().sum(dim=1).max() * x2.abs().max() + b2.abs().max())).item() <= 1e-15 * n


@pytest.mark.parametrize("precision", [0, 1])
def test_config2_n8192_factors_reproduce_A(mplu, oracle, solver, record_property, precision):
    """BASELINE.json configs[1] (n=8192, fp16 panel + fp16/fp32-accumulate GEMM + fp64 IR): L*U reproduces A to the
    16-bit operand tolerance, the refined solution to fp64."""
    import torch
    n = 8192
    A, b = mplu.generate(n, seed=3)
    x, st = solver.gesv(A, b, mplu.default_options(precision=precision))
    assert st.converged == 1 and st.iters <= 3 and st.backward_error <= 1e-15 * n
    assert (x - 1).abs().max().item() <= 1e-11
    LU = solver.factors(n)
    L = torch.tril(LU, -1) + torch.eye(n, dtype=torch.float64, device="cuda")
    U = torch.triu(LU)
    E = (L @ U - A).abs().max().item()
    u16 = 2.0 ** -11 if precision == 0 else 2.0 ** -8
    # |A - LU| <= c * u16 * max|A| with a modest constant: the diagonal of this matrix is ~n/2 * 10, kept to fp32 level
    assert E <= 0.05 * u16 * A.abs().max().item(), E
    # and tile by tile against |L||U|: the bound above does not see a wrong off-diagonal tile (entries at most 9.9)
    check_factors(oracle, record_property, A, LU, precision)


# ---- condition-number sweep (BASELINE.json configs[4]) and GMRES-based refinement -----------------------------------
def _spd(oracle, n, kappa):
    A = oracle.spd_kappa_matrix(n, kappa, seed=1)
    return A, A.sum(axis=1)


@pytest.mark.parametrize("kappa,prec,classic_ok", [(1e2, 0, True), (1e4, 0, True), (1e4, 1, True), (1e7, 0, False), (1e6, 1, False)])
def test_kappa_sweep_classic_vs_gmres_refinement(mplu, oracle, solver, kappa, prec, classic_ok):
    """SPD matrices with geometric spectrum.  Classic refinement with 16-bit factors converges while kappa * u16 is
    small and stagnates beyond (SURVEY.md section 8c); GMRES-IR converges on all of them to the fp64 backward error a
    host dgetrf/dgetrs solve (the reference's factors + a solve) reaches."""
    n = 1024
    A, b = _spd(oracle, n, kappa)
    x_ref, _, _ = oracle.lapack_gesv(A, b)
    r = b - A @ x_ref
    be_ref = np.abs(r).max() / (np.abs(A).sum(axis=1).max() * np.abs(x_ref).max() + np.abs(b).max())
    import torch
    dA = cm(torch.tensor(A, dtype=torch.float64, device="cuda"))
    db = torch.tensor(b, dtype=torch.float64, device="cuda")
    x, st = solver.gesv(dA, db, mplu.default_options(precision=prec, fp64_fallback=0), allow_noconv=True)
    assert bool(st.converged) == classic_ok, st.as_dict()
    xg, sg = solver.gesv(dA, db, mplu.default_options(precision=prec, refinement=mplu.REFINE_GMRES), allow_noconv=True)
    assert sg.converged == 1 and sg.gmres_iters >= sg.iters
    assert sg.backward_error <= max(10 * be_ref, 2 * n * EPS)
    if classic_ok:
        assert sg.iters <= st.iters  # never more outer iterations than classic refinement
    # forward error consistent with the conditioning
    assert np.abs(xg.cpu().numpy() - 1).max() <= 100 * kappa * n * EPS


def test_fp16_overflow_falls_back_to_bf16(mplu, oracle, solver):
    """a matrix whose inverse factors leave the scaled fp16 range: reported (status bit 0) and redone in bf16"""
    n = 512
    A, b = _spd(oracle, n, 1e12)
    import torch
    dA = cm(torch.tensor(A, dtype=torch.float64, device="cuda"))
    db = torch.tensor(b, dtype=torch.float64, device="cuda")
    overflowed = False
    try:
        x, st = solver.gesv(dA, db, mplu.default_options(refinement=mplu.REFINE_GMRES, bf16_fallback=0, fp64_fallback=0), allow_noconv=True)
    except mplu.MpluError as e:
        assert e.code == -5  # MPLU_E_OVERFLOW: reported, not silent
        overflowed = True
    x2, st2 = solver.gesv(dA, db, mplu.default_options(refinement=mplu.REFINE_GMRES), allow_noconv=True)
    assert st2.precision_used == (mplu.MPLU_BF16 if overflowed else mplu.MPLU_FP16)
    assert np.isfinite(x2.cpu().numpy()).all()


def test_schedule_options_do_not_change_the_arithmetic(mplu, oracle, record_property):
    """Grouped launches, triangular K-range skipping, lane split, CUDA graph, workspace GETRF, the left-looking schedule
    (schedule=1), chain-lane programmatic launches and the width / grid of the persistent GETRF launches only change WHEN and
    WHERE the same products are formed: the factors are bit-identical within each GETRF arithmetic -- the dataflow launch
    (default; rank-128 updates, the order in which helpers take tasks must not matter), the fused step program (flow_w = 0:
    tensor-core leaf, recursion's products) and one launch per leaf / product (fuse_w = 0: fp32 FMA leaf) -- and agree to
    rounding level between them."""
    import torch
    n = 2304  # not a multiple of the tile size: the last tile is partial
    A = oracle.counter_matrix(n, seed=4)
    dA = cm(torch.tensor(A, dtype=torch.float64, device="cuda"))
    db = torch.tensor(A.sum(axis=1), dtype=torch.float64, device="cuda")
    ref = {}
    s = mplu.Solver(0)
    try:
        common = (dict(), dict(group=0), dict(tri_skip=0), dict(lookahead=0), dict(use_graph=0), dict(gemm_variant=mplu.GEMM_CG2),
                  dict(stream_c=0), dict(fuse_w=0), dict(fuse_w=0, group=0), dict(fuse_w=256), dict(fuse_w=256, fuse_ctas=2),
                  dict(fuse_w=512, fuse_ctas=8, use_graph=0), dict(fuse_w=512, fuse_ctas=32, tri_skip=0), dict(lazy_touch=0),
                  dict(lazy_touch=0, fuse_w=0))
        common = tuple(dict(flow_w=0, **kw) for kw in common) + (
            dict(), dict(flow_ctas=4), dict(flow_ctas=24, flow_merge_ctas=0), dict(flow_merge_ctas=6, use_graph=0),
            dict(flow_w=512, lazy_touch=0), dict(flow_w=512, lookahead=0), dict(flow_w=256), dict(flow_w=256, flow_ctas=6, group=0))
        right = tuple(dict(schedule=0, **kw) for kw in common) + (
            dict(schedule=0, flow_w=0, tile_ws=1), dict(schedule=0, flow_w=0, side_sms=16, side_sms_early=8), dict(schedule=0, flow_w=0, pdl=2),
            dict(schedule=0, tile_ws=1))
        left = tuple(dict(schedule=1, **kw) for kw in common) + (
            dict(schedule=1, flow_w=0, eager=0), dict(schedule=1, flow_w=0, use_graph=0, side_sms_left=64), dict(schedule=1, flow_w=0, side_sms_left=24),
            dict(schedule=1, flow_w=0, early_scale=1, lazy_touch=0), dict(schedule=1, flow_w=0, early_scale=1, lazy_touch=0, use_graph=0),
            dict(schedule=1, eager=0), dict(schedule=1, side_sms_left=32, flow_ctas=32), dict(schedule=1, early_scale=1, lazy_touch=0),
            dict(schedule=1, pair_ts=1), dict(schedule=1, pair_ts=1, eager=0, use_graph=0), dict(schedule=1, pair_ts=1, flow_w=0),
            dict(schedule=1, pair_ts=1, flow_w=0, fuse_w=0, lazy_touch=0))
        for kw in right + left:
            x, st = s.gesv(dA, db, mplu.default_options(nb=512, update_pair=0, **kw))  # paired updates: test_paired_updates
            LU = s.factors(n)
            assert st.converged == 1
            flow_w = kw.get("flow_w", 2048)
            if flow_w >= 512: grp = "flow"          # whole tiles as one dataflow launch
            elif flow_w > 0: grp = "flow256"        # 256-blocks as dataflow launches, the 512-node's products as launches
            else: grp = "unfused" if kw.get("fuse_w", 2048) == 0 else "fused"
            if grp not in ref:
                ref[grp] = LU.clone()
            else:
                assert torch.equal(LU, ref[grp]), kw
        m = ref["unfused"].abs().max().item()
        d = (ref["fused"] - ref["unfused"]).abs().max().item()
        assert 0 <= d <= 1e-5 * m, d
        for g in ("flow", "flow256"):  # another summation order on the same 16-bit operands
            d = (ref[g] - ref["unfused"]).abs().max().item()
            assert 0 <= d <= 2.0 ** -9 * m, (g, d)
        for g, LU in ref.items():
            check_factors(oracle, record_property, dA, LU, 0, f"rho_{g}")
    finally:
        s.close()


@pytest.mark.parametrize("n,nb,fuse_w,ctas", [(4096, 2048, 2048, 16), (4096, 2048, 1024, 8), (4096, 4096, 4096, 16), (3000, 1024, 1024, 4)])
@pytest.mark.parametrize("precision", [0, 1])
def test_fused_getrf_matches_the_launch_per_product_path(mplu, oracle, record_property, n, nb, fuse_w, ctas, precision):
    """opts.fuse_w: the GETRF of a diagonal block (leaves + every product between them) as ONE persistent launch with grid
    barriers between the steps (csrc/getrf_fused.cu) instead of one launch per leaf / product group.  The products
    between the leaves are the same tcgen05 products on the same 16-bit operands in the same order; inside a leaf the
    fused kernel forms the rank-32 updates and the inverse merges on the tensor cores from three-part bf16 splits (fp32-class
    accuracy, another summation order) where the stand-alone leaf uses fp32 FMAs, so the factors agree to rounding level, not bit for bit; fused runs
    agree with each other bit for bit.  nb = 4096 exercises the step program read from global memory (it does not fit the
    shared-memory staging area), n = 3000 the identity padding."""
    import torch
    A, b = mplu.generate(n, seed=6)
    s = mplu.Solver(0)
    try:
        x0, st0 = s.gesv(A, b, mplu.default_options(nb=nb, fuse_w=0, flow_w=0, precision=precision))
        LU0 = s.factors(n).clone()
        LU1 = None
        for rep in range(2):  # second pass replays the cached graph / programs
            x1, st1 = s.gesv(A, b, mplu.default_options(nb=nb, fuse_w=fuse_w, fuse_ctas=ctas, flow_w=0, precision=precision))
            assert st1.converged == 1 and st1.status_bits == 0 and st1.iters <= st0.iters + 1
            assert st1.kernel_launches < st0.kernel_launches
            F = s.factors(n)
            if LU1 is None:
                LU1 = F.clone()
            assert torch.equal(F, LU1)
        dU = (torch.triu(LU1) - torch.triu(LU0)).abs().max().item()
        dL = (torch.tril(LU1, -1) - torch.tril(LU0, -1)).abs().max().item()
        assert dU <= 1e-5 * LU0.abs().max().item(), dU  # a few dozen fp32 ulps of the diagonal: the summation order differs
        # the 16-bit inverse of a diagonal block can round the other way: one fp16 ulp of a multiplier
        assert dL <= (2.0 ** -10 if precision == 0 else 2.0 ** -7) * torch.tril(LU0, -1).abs().max().item(), dL
        check_factors(oracle, record_property, A, LU0, precision, "rho_unfused")
        check_factors(oracle, record_property, A, LU1, precision, "rho_fused")
        assert float((x1 - 1).abs().max()) < 1e-11 and float((x1 - x0).abs().max()) < 1e-11
    finally:
        s.close()


@pytest.mark.parametrize("n,nb", [(8192, 1024), (4096, 512), (6000, 1024), (16384, 2048)])
@pytest.mark.parametrize("kw", [dict(), dict(lazy_touch=0), dict(use_graph=0, precision=1), dict(edge_nb=256, eager=0)])
def test_paired_updates(mplu, oracle, record_property, n, nb, kw):
    """opts.update_pair: two consecutive rank-nb updates of a block-column range applied as ONE product over both panels
    (K = 2 nb).  Same 16-bit products; the two partial sums meet in the TMEM accumulator instead of in fp32 C, so the factors
    agree with the one-update-per-pass schedule to fp32 rounding of the entries (not bit for bit), the refined solution to
    fp64 accuracy, and repeated runs are bit-identical."""
    import torch
    A, b = mplu.generate(n, seed=9)
    s = mplu.Solver(0)
    try:
        x0, st0 = s.gesv(A, b, mplu.default_options(nb=nb, update_pair=0, **kw))
        LU0 = s.factors(n).clone()
        LU1 = None
        for rep in range(2):
            x1, st1 = s.gesv(A, b, mplu.default_options(nb=nb, update_pair=1, **kw))
            assert st1.converged == 1 and st1.status_bits == 0 and st1.iters <= st0.iters + 1
            assert st1.trailing_launches < st0.trailing_launches  # fewer, longer update passes
            F = s.factors(n)
            if LU1 is None:
                LU1 = F.clone()
            assert torch.equal(F, LU1)
        tol = 2.0 ** -8 if kw.get("precision", 0) == 0 else 2.0 ** -5  # a 16-bit shadow may round the other way
        assert (LU1 - LU0).abs().max().item() <= tol * LU0.abs().max().item()
        assert float((x1 - 1).abs().max()) < 1e-11 and float((x1 - x0).abs().max()) < 1e-11
        assert st1.backward_error <= 2 * n * EPS
        check_factors(oracle, record_property, A, LU0, kw.get("precision", 0), "rho_reference")
        check_factors(oracle, record_property, A, LU1, kw.get("precision", 0))
        check_agreement(oracle, record_property, LU1, LU0, kw.get("precision", 0))  # tile by tile, within AGREE
    finally:
        s.close()


@pytest.mark.parametrize("n,nb,edge", [(8192, 1024, 512), (4096, 512, 128), (6000, 1024, 256), (16384, 2048, 1024)])
@pytest.mark.parametrize("kw", [dict(), dict(lazy_touch=0), dict(use_graph=0, precision=1)])
def test_narrow_edge_tiles(mplu, oracle, record_property, n, nb, edge, kw):
    """opts.edge_nb: first and last block column of the left-looking schedule narrower than nb.  Other tile boundaries mean
    other rank-k pieces of the same sums: factors agree with the uniform tiling to a few 16-bit ulps, the refined solution
    is the same to fp64 accuracy, repeated runs are bit-identical."""
    import torch
    A, b = mplu.generate(n, seed=8)
    s = mplu.Solver(0)
    try:
        x0, st0 = s.gesv(A, b, mplu.default_options(nb=nb, edge_nb=0, **kw))
        LU0 = s.factors(n).clone()
        LU1 = None
        for rep in range(2):
            x1, st1 = s.gesv(A, b, mplu.default_options(nb=nb, edge_nb=edge, **kw))
            assert st1.converged == 1 and st1.status_bits == 0 and st1.iters <= st0.iters + 1
            F = s.factors(n)
            if LU1 is None:
                LU1 = F.clone()
            assert torch.equal(F, LU1)
        tol = 2.0 ** -8 if kw.get("precision", 0) == 0 else 2.0 ** -5
        assert (LU1 - LU0).abs().max().item() <= tol * LU0.abs().max().item()
        assert float((x1 - 1).abs().max()) < 1e-11 and float((x1 - x0).abs().max()) < 1e-11
        assert st1.backward_error <= 2 * n * EPS
        check_factors(oracle, record_property, A, LU0, kw.get("precision", 0), "rho_reference")
        check_factors(oracle, record_property, A, LU1, kw.get("precision", 0))
    finally:
        s.close()


@pytest.mark.parametrize("n,nb,flow_w,ctas", [(2048, 512, 256, 4), (4096, 2048, 2048, 16), (4096, 1024, 1024, 8), (4096, 4096, 4096, 16),
                                              (3000, 1024, 1024, 6), (4096, 2048, 512, 8)])
@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.timeout(300)
def test_dataflow_getrf_matches_the_launch_per_product_path(mplu, oracle, record_property, n, nb, flow_w, ctas, precision):
    """opts.flow_w: the GETRF of a diagonal block as ONE dataflow launch (csrc/getrf_flow.cu): right-looking at 128-block
    granularity, leaf CTAs + helper CTAs that pull tile products from a priority-ordered list and hand results over through
    counters.  Same tcgen05 products on the same 16-bit operands as the recursion, but the Schur updates are summed in
    rank-128 pieces and the panel solves use one 128-block inverse at a time, so the factors agree to rounding level;
    repeated runs agree bit for bit (the order in which helpers take tasks does not change any sum).  nb = 4096 exercises
    problem descriptors read from global memory, n = 3000 the identity padding, flow_w < nb the recursion above the
    dataflow blocks."""
    import torch
    A, b = mplu.generate(n, seed=6)
    s = mplu.Solver(0)
    try:
        x0, st0 = s.gesv(A, b, mplu.default_options(nb=nb, fuse_w=0, flow_w=0, precision=precision))
        LU0 = s.factors(n).clone()
        LU1 = None
        for rep in range(3):  # later passes replay the cached graph / programs
            x1, st1 = s.gesv(A, b, mplu.default_options(nb=nb, flow_w=flow_w, flow_ctas=ctas, precision=precision))
            assert st1.converged == 1 and st1.status_bits == 0 and st1.iters <= st0.iters + 1
            assert st1.kernel_launches < st0.kernel_launches
            F = s.factors(n)
            if LU1 is None:
                LU1 = F.clone()
            assert torch.equal(F, LU1)
        dU = (torch.triu(LU1) - torch.triu(LU0)).abs().max().item()
        dL = (torch.tril(LU1, -1) - torch.tril(LU0, -1)).abs().max().item()
        # another summation order on 16-bit operands: a few fp16 / bf16 ulps of the largest entries
        tol = 2.0 ** -8 if precision == 0 else 2.0 ** -5
        assert dU <= tol * LU0.abs().max().item(), dU
        assert dL <= tol * torch.tril(LU0, -1).abs().max().item(), dL
        check_factors(oracle, record_property, A, LU0, precision, "rho_unfused")
        check_factors(oracle, record_property, A, LU1, precision, "rho_dataflow")
        assert float((x1 - 1).abs().max()) < 1e-11 and float((x1 - x0).abs().max()) < 1e-11
    finally:
        s.close()


@pytest.mark.parametrize("n,nb", [(4096, 1024), (2048, 512)])
@pytest.mark.parametrize("precision", [0, 1])
def test_lazy_first_touch_is_bit_identical(mplu, oracle, record_property, n, nb, precision):
    """opts.lazy_touch: no separate fp64 -> fp32 cast pass over A -- every tile's first Schur update takes its addend
    straight from the caller's fp64 matrix (the cast of /root/reference/MPF.cu:20-25,106-121 fused into the GEMM
    epilogue's loads) and ||A||_inf rides in the first residual.  Same arithmetic: identical factors, norms, solutions."""
    import torch
    A, b = mplu.generate(n, seed=8)
    s = mplu.Solver(0)
    try:
        x0, st0 = s.gesv(A, b, mplu.default_options(nb=nb, lazy_touch=0, precision=precision))
        LU0 = s.factors(n).clone()
        check_factors(oracle, record_property, A, LU0, precision)
        for rep in range(2):
            x1, st1 = s.gesv(A, b, mplu.default_options(nb=nb, lazy_touch=1, precision=precision))
            assert torch.equal(s.factors(n), LU0)
            assert torch.equal(x1, x0)
            assert st1.iters == st0.iters and st1.anorm_inf == st0.anorm_inf and st1.backward_error == st0.backward_error
            assert st1.kernel_launches == st0.kernel_launches + 0 or True
        # a second matrix at another address through the same cached graph
        A2, b2 = mplu.generate(n, seed=9)
        x2, st2 = s.gesv(A2, b2, mplu.default_options(nb=nb, lazy_touch=1, precision=precision))
        assert st2.converged == 1 and float((x2 - 1).abs().max()) < 1e-11
    finally:
        s.close()


def test_lazy_first_touch_scale_overflow_is_redone(mplu, oracle, solver, record_property):
    """the fp16 scale of the lazy first touch comes from the first block column / row only; an interior block 2^6 larger
    leaves the fp16 range under it: detected, redone with the global scale, right answer"""
    import torch
    n, nb = 1536, 512
    A = oracle.counter_matrix(n, seed=5)
    A[nb:, nb:] *= 64.0
    b = A.sum(axis=1)
    x, st = run(mplu, solver, A, b, nb=nb, lazy_touch=1)
    if st["status_bits"] == 0:  # an overflow that did not spoil the solve keeps its factors on purpose
        check_factors(oracle, record_property, A, solver.factors(n), 0, "rho_lazy")
    x0, st0 = run(mplu, solver, A, b, nb=nb, lazy_touch=0)
    if st0["status_bits"] == 0:
        check_factors(oracle, record_property, A, solver.factors(n), 0, "rho_eager")
    assert st["converged"] == 1 and st0["converged"] == 1
    np.testing.assert_allclose(x, x0, rtol=0, atol=1e-10)
    np.testing.assert_allclose(x, 1.0, rtol=0, atol=1e-9)
