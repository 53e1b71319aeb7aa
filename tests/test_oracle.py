"""CPU tests: pin the oracle (generator vs libc rand(); factorization vs host LAPACK; restatement of the reference's
MPF vs outputs of the unmodified reference captured on a B200 in tests/golden/)."""
import ctypes
import os

import numpy as np
import pytest

from conftest import GOLDEN


def test_glibc_rand_matches_libc(oracle):
    libc = ctypes.CDLL("libc.so.6")
    libc.srand(1)
    ref = [libc.rand() for _ in range(5000)]
    g = oracle.GlibcRand()
    assert [g.rand() for _ in range(5000)] == ref


def test_matrix_generator_first_matrix(oracle):
    # SURVEY.md section 8b [probe]: first 2x2 emitted by the reference generator is 8.3 8.6 / 7.7 1.5
    n, M = next(oracle.matrix_generator_stream(2))
    assert n == 2
    np.testing.assert_array_equal(M, np.array([[8.3, 8.6], [7.7, 1.5]]))
    assert oracle.matrix_generator_sizes(1024, 2, "exp") == [2 ** k for k in range(1, 11)]
    assert oracle.matrix_generator_sizes(10, 3, "lin") == [2, 5, 8]


def test_double_to_fp16_contract(oracle):
    x = np.array([1e6, -1e6, 65504.0, 6.0e-5, -6.0e-5, 6.2e-5, 0.1, 1.0 + 2 ** -11])
    h = oracle.double_to_fp16(x).astype(np.float64)
    assert h[0] == 65504.0 and h[1] == -65504.0 and h[2] == 65504.0  # saturates (fp16_utils.h:19-20)
    assert h[3] == 0.0 and h[4] == 0.0 and h[5] != 0.0  # flush below 6.10352e-5 (fp16_utils.h:21)
    assert h[6] == np.float64(np.float16(0.1)) and h[7] == 1.0  # RN, ties to even


@pytest.mark.parametrize("n", [33, 64, 256])
def test_mpf_reference_on_dominant_is_nopivot_lu(oracle, n):
    from scipy.linalg import lu_factor
    A = oracle.counter_matrix(n, seed=7)
    LU, ipiv = oracle.mpf_reference(A, 32)
    assert np.array_equal(ipiv, np.arange(1, n + 1))  # diagonal dominance => identity pivots (SURVEY.md section 0)
    lu, piv = lu_factor(A)
    assert np.array_equal(piv, np.arange(n))
    np.testing.assert_allclose(LU, lu, rtol=0, atol=1e-12 * np.abs(lu).max())
    assert oracle.check_correctitude(A, LU, ipiv)
    np.testing.assert_allclose(oracle.lu_nopivot_fp64(A, 32), LU, rtol=0, atol=1e-12 * np.abs(lu).max())


@pytest.mark.parametrize("n", [2, 3, 31, 32, 33, 65])
def test_mpf_reference_random_passes_reference_check(oracle, n):
    # edge sizes around the panel width r = 32, incl. N % r == 1 where MPF leaves IPIV[N-1] untouched (MPF.cu:104)
    rng = np.random.default_rng(n)
    A = (rng.integers(0, 100, size=(n, n)) / 10.0) + 0.0
    LU, ipiv = oracle.mpf_reference(A, 32)
    assert oracle.check_correctitude(A, LU, ipiv, tol=1e-9)
    assert ipiv[n - 1] == n


@pytest.mark.parametrize("n", [128, 256])
def test_golden_dominant_vs_oracle(oracle, n):
    g = np.load(os.path.join(GOLDEN, f"ref_mpf_dd_n{n}.npz"))
    A = oracle.counter_matrix(n, seed=int(g["seed"]))
    LU, ipiv = oracle.mpf_reference(A, int(g["r"]))
    assert np.array_equal(g["ipiv"], ipiv) and np.array_equal(ipiv, np.arange(1, n + 1))
    np.testing.assert_allclose(g["LU"], LU, rtol=0, atol=1e-13 * np.abs(LU).max())
    assert oracle.check_correctitude(A, g["LU"], g["ipiv"])


def _stream_matrix(oracle, n):
    for m_, M in oracle.matrix_generator_stream(n):
        if m_ == n:
            return oracle.as_benchmark_reads(M)
    raise AssertionError


@pytest.mark.parametrize("n", [64, 128])
def test_golden_random_pivoting_vs_oracle(oracle, n):
    # fp16 pivot discovery on the reference generator's own stream: the restated HGETF2 reproduces the reference's
    # pivot sequence exactly at these sizes (fused multiply-subtract, the -O3 code path)
    g = np.load(os.path.join(GOLDEN, f"ref_mpf_rand_n{n}.npz"))
    A = _stream_matrix(oracle, n)
    LU, ipiv = oracle.mpf_reference(A, 32, fused=True)
    assert np.array_equal(g["ipiv"], ipiv)
    np.testing.assert_allclose(g["LU"], LU, rtol=0, atol=1e-11 * np.abs(LU).max())
    assert oracle.check_correctitude(A, g["LU"], g["ipiv"])


def test_golden_random_256_matches_with_the_references_tie_break(oracle):
    # Exact ties of |a| in fp16 are frequent on this value set (k/10); the reference's reduction tree does NOT keep the
    # first maximum but the tied row with the smallest (block, bit-reversed thread index) -- hgetf2_kernel.cu:48-56,72-79.
    # With that rule restated the n = 256 golden output (which "first maximum wins" missed) is reproduced exactly.
    g = np.load(os.path.join(GOLDEN, "ref_mpf_rand_n256.npz"))
    A = _stream_matrix(oracle, 256)
    assert oracle.check_correctitude(A, g["LU"], g["ipiv"])
    LU, ipiv = oracle.mpf_reference(A, 32)
    assert np.array_equal(ipiv, g["ipiv"])
    np.testing.assert_allclose(g["LU"], LU, rtol=0, atol=1e-11 * np.abs(LU).max())


def test_hgetf2_tie_break_is_the_reduction_trees(oracle):
    # column with its maximum at rows 20 and 68: slot 68 % 64 = 4 absorbs row 68 first and later wins the tie against
    # slot 20 (strict '>'), so the pivot is row 68 although row 20 comes first
    P = np.zeros((128, 1), dtype=np.float16)
    P[20, 0] = P[68, 0] = 9.9
    P[5, 0] = 3.0
    _, ip = oracle.hgetf2(P)
    assert ip[0] == 69
    # across blocks of 256 rows the lower block wins
    P = np.zeros((600, 1), dtype=np.float16)
    P[300, 0] = P[255, 0] = 2.5
    _, ip = oracle.hgetf2(P)
    assert ip[0] == 256


def test_emulated_mixed_lu_refines_to_fp64(oracle):
    n = 512
    A = oracle.counter_matrix(n, seed=1)
    b = A.sum(axis=1)
    for bf16 in (False, True):
        W = oracle.lu_mixed_emulated(A, 128, bf16=bf16)
        res = oracle.refine(A, b, W)
        assert res["converged"] and res["iters"] <= 3
        assert res["backward_error"] < 4 * n * 1.1e-16
        x_ref, _, _ = oracle.lapack_gesv(A, b)
        np.testing.assert_allclose(res["x"], x_ref, rtol=1e-12)


@pytest.mark.parametrize("n,dominant", [(300, True), (1025, True), (1025, False)])
def test_blocked_generator_equals_counter_matrix(oracle, n, dominant):
    """bench.py's reference arm builds its full-size input by column blocks: same values bit for bit"""
    A = np.empty((n, n), order="F")
    oracle.counter_matrix_into(A, seed=3, dominant=dominant, block=256)
    assert np.array_equal(A, oracle.counter_matrix(n, seed=3, dominant=dominant))


def _randn_dominant(n, seed):
    """stable without pivoting, and its off-diagonal blocks carry O(1) weight next to a diagonal of 2 sqrt(n)"""
    return np.random.default_rng(seed).standard_normal((n, n)) + 2.0 * np.sqrt(n) * np.eye(n)


@pytest.mark.parametrize("n", [1024, 3000])
@pytest.mark.parametrize("kind", ["counter", "randn"])
def test_factor_tile_ratio_of_the_emulated_factors(oracle, n, kind):
    """the tile-wise componentwise backward error of the emulated 16-bit factorization is a few unit roundoffs of the
    16-bit type (the bound the GPU factor tests use is 3 u), on dominant and on randn + 2 sqrt(n) I inputs"""
    A = oracle.counter_matrix(n, seed=1) if kind == "counter" else _randn_dominant(n, 1)
    for bf16, u in ((False, 2.0 ** -11), (True, 2.0 ** -8)):
        rho = oracle.factor_tile_ratio(A, oracle.lu_mixed_emulated(A, 128, bf16=bf16))
        assert rho.shape == ((n + 127) // 128,) * 2
        assert 0 < rho.max() <= 2 * u, (bf16, rho.max() / u)


def test_factor_tile_ratio_names_a_wrong_tile(oracle):
    """one off-diagonal tile of the factors 1 % off: that tile and only that tile leaves the bound, although the
    refinement still converges and the error is far below the old normwise tolerances (2^-9 max|LU|)"""
    n, u = 1024, 2.0 ** -11
    A = _randn_dominant(n, 2)
    F = oracle.lu_mixed_emulated(A, 128)
    assert oracle.factor_tile_ratio(A, F).max() <= 3 * u
    for I, J in ((1, 4), (5, 1)):  # a tile of U, a tile of L
        G = F.copy()
        G[128 * I:128 * (I + 1), 128 * J:128 * (J + 1)] *= 1.01
        rho = oracle.factor_tile_ratio(A, G)
        bad = np.argwhere(rho > 3 * u)
        assert [tuple(t) for t in bad] == [(I, J)], bad
        assert oracle.refine(A, A.sum(axis=1), G)["converged"]


def test_factor_tile_ratio_edges(oracle):
    # ragged order, exact factors: zero error; a tile whose |L||U| is zero must have zero error too
    A = _randn_dominant(200, 3)
    rho = oracle.factor_tile_ratio(A, oracle.lu_nopivot_fp64(A))
    assert rho.shape == (2, 2) and rho.max() <= 1e-14
    D = np.diag(np.arange(1.0, 257.0))
    assert (oracle.factor_tile_ratio(D, D) == 0).all()  # off-diagonal tiles: M = 0 and E = 0
    D2 = D.copy()
    D2[200, 10] = 1.0  # A has an entry where L U (= D) has none
    rho = oracle.factor_tile_ratio(D2, D)
    assert rho[1, 0] == np.inf and rho[0, 0] == 0 and rho[1, 1] == 0
    try:
        import torch
    except ImportError:
        return
    F = oracle.lu_mixed_emulated(A, 128)
    np.testing.assert_allclose(oracle.factor_tile_ratio(torch.tensor(A), torch.tensor(F.astype(np.float64))),
                               oracle.factor_tile_ratio(A, F), rtol=1e-12)


def _exact_block_inverses(LU, blk=128):
    n = LU.shape[0]
    npad = -(-n // blk) * blk
    F = np.eye(npad)
    F[:n, :n] = LU
    Li, Ui = [], []
    for i in range(npad // blk):
        D = F[i * blk:(i + 1) * blk, i * blk:(i + 1) * blk]
        Li.append(np.linalg.inv(np.tril(D, -1) + np.eye(blk)))
        Ui.append(np.linalg.inv(np.triu(D)))
    return np.array(Li), np.array(Ui)


@pytest.mark.parametrize("n", [1, 127, 129, 1000])
def test_blocked_sweeps_are_the_triangular_solves(oracle, n):
    """with exact block inverses and the solved blocks kept in fp64, the blocked sweeps are L U x = b; with fp32 blocks,
    fp32 factors and an fp32 evaluation they stay within fp32 rounding of it"""
    from scipy.linalg import solve_triangular
    A = _randn_dominant(n, n)
    LU = oracle.lu_nopivot_fp64(A)
    Li, Ui = _exact_block_inverses(LU)
    rng = np.random.default_rng(0)
    B = rng.standard_normal((n, 3)).astype(np.float32).astype(np.float64)  # the sweeps take b in fp32
    y = solve_triangular(LU, B, lower=True, unit_diagonal=True)
    X = solve_triangular(LU, y, lower=False)
    got = oracle.blocked_sweeps(LU, Li, Ui, B, store=np.float64)
    np.testing.assert_allclose(got, X, rtol=0, atol=1e-12 * np.abs(X).max())
    x1 = oracle.blocked_sweeps(LU, Li, Ui, B[:, 1], store=np.float64)
    assert x1.shape == (n,)
    np.testing.assert_allclose(x1, X[:, 1], rtol=0, atol=1e-12 * np.abs(X).max())
    x64 = oracle.blocked_sweeps(LU, Li, Ui, B)  # fp32 blocks
    x32 = oracle.blocked_sweeps(LU, Li, Ui, B, dtype=np.float32)
    assert (x64.astype(np.float32) == x64).all() and (x32.astype(np.float32) == x32).all()
    err = np.abs(x64 - X).max()
    assert 0 < err <= 1e-6 * np.abs(X).max()
    assert np.abs(x32 - X).max() <= 1e-5 * np.abs(X).max()


def test_factor_tile_distance_sees_what_the_backward_error_bound_lets_pass(oracle):
    """an L tile 0.1 % off stays under the 3 u backward-error bound, but against the unperturbed factors it is a
    distance of about one u, located in its own tile; identical factors are at distance 0"""
    n, u = 1024, 2.0 ** -11
    A = _randn_dominant(n, 2)
    F = oracle.lu_mixed_emulated(A, 128)
    assert (oracle.factor_tile_distance(F, F) == 0).all()
    G = F.copy()
    G[640:768, 128:256] *= 1.001
    assert oracle.factor_tile_ratio(A, G).max() <= 3 * u
    d = oracle.factor_tile_distance(G, F)
    assert np.unravel_index(np.argmax(d), d.shape) == (5, 1) and d.max() >= u / 2
    assert d[:5].max() == 0 and d[6:].max() == 0  # only tile row 5 of L U changes
    try:
        import torch
    except ImportError:
        return
    np.testing.assert_allclose(oracle.factor_tile_distance(torch.tensor(G.astype(np.float64)), torch.tensor(F.astype(np.float64))),
                               d, rtol=1e-12)
