"""GPU parity tests of the 2D block-cyclic path (csrc/dist.cu) through the C ABI: the same solve as the single-GPU
path, distributed over P x Q logical ranks.  "local" mode hosts all ranks on cuda:0 (collectives = device copies),
so the block-cyclic logic is covered on a 1-GPU box; the NCCL test needs >= 2 GPUs and is skipped otherwise."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_reference import check_factors

pytestmark = pytest.mark.gpu
EPS = np.finfo(np.float64).eps / 2


@pytest.fixture(scope="module")
def single_ref(mplu, oracle):
    """single-GPU result + LAPACK result for the inputs used below"""
    import torch
    out = {}
    s = mplu.Solver(0)
    for n in (1024, 2048):
        A = oracle.counter_matrix(n, seed=1)
        b = A.sum(axis=1)
        dA = torch.tensor(A, dtype=torch.float64, device="cuda").t().contiguous().t()
        x, st = s.gesv(dA, torch.tensor(b, device="cuda"), mplu.default_options(nb=256))
        x_ref, lu_ref, _ = oracle.lapack_gesv(A, b)
        out[n] = dict(A=A, b=b, x=x.cpu().numpy(), iters=st.iters, be=st.backward_error, x_ref=x_ref, lu_ref=lu_ref,
                      LU=s.factors(n).cpu().numpy())
    s.close()
    return out


@pytest.mark.parametrize("n,nb,P,Q", [(1024, 256, 1, 1), (1024, 256, 1, 2), (1024, 256, 2, 2), (1024, 256, 2, 4),
                                      (2048, 256, 2, 2), (2048, 512, 2, 4), (1024, 128, 3, 2)])
def test_block_cyclic_solve_matches_single_gpu_and_lapack(mplu, oracle, single_ref, record_property, n, nb, P, Q):
    ref = single_ref[n]
    ds = mplu.DistSolver(0, P, Q)
    try:
        As, bs = ds.generate(n, nb, seed=1)
        # the device generator's local tiles are exactly the block-cyclic pieces of the oracle's matrix
        parts = mplu.scatter_block_cyclic(ref["A"], nb, P, Q)
        for i in range(ds.num_local):
            p, q, mloc, nloc = ds.local_shape(i, n, nb)
            if mloc and nloc:
                assert np.array_equal(As[i].cpu().numpy(), parts[p * Q + q])
            np.testing.assert_allclose(bs[i].cpu().numpy(), ref["b"], rtol=1e-14)
        xs, st = ds.gesv(n, nb, As, bs, mplu.default_options())
        assert st.converged == 1 and st.status_bits == 0
        assert st.iters <= ref["iters"]
        assert st.backward_error <= 2 * n * EPS
        for x in xs:  # every rank holds the same full solution
            np.testing.assert_allclose(x.cpu().numpy(), ref["x_ref"], rtol=0, atol=1e-12)
            assert np.array_equal(x.cpu().numpy(), xs[0].cpu().numpy())
        # factors: gather the local L\U pieces and compare with the fp64 no-pivot LU (fp16 tolerance as in
        # test_gpu_solver.py) and with the single-GPU factors (same arithmetic class, different blocking)
        fac = [ds.local_factors(i, n, nb).cpu().numpy() for i in range(ds.num_local)]
        order = [None] * (P * Q)
        for i in range(ds.num_local):
            p, q, mloc, nloc = ds.local_shape(i, n, nb)
            order[p * Q + q] = fac[i][:mloc, :nloc]
        LU = mplu.gather_block_cyclic(order, n, nb, P, Q)
        u16 = 2.0 ** -11
        lu_ref = ref["lu_ref"]
        assert np.abs(np.triu(LU) - np.triu(lu_ref)).max() <= 0.02 * u16 * np.abs(lu_ref).max()
        assert np.abs(np.tril(LU, -1) - np.tril(lu_ref, -1)).max() <= 2 * u16 * np.abs(np.tril(lu_ref, -1)).max()
        assert np.abs(np.triu(LU) - np.triu(ref["LU"])).max() <= 0.02 * u16 * np.abs(lu_ref).max()
        check_factors(oracle, record_property, ref["A"], LU, 0)  # tile by tile: blind to no off-diagonal tile
    finally:
        ds.close()


def test_block_cyclic_bf16_and_no_lookahead(mplu, single_ref):
    n, nb = 1024, 256
    ds = mplu.DistSolver(0, 2, 2)
    try:
        As, bs = ds.generate(n, nb, seed=1)
        for kw in (dict(precision=1), dict(lookahead=0)):
            xs, st = ds.gesv(n, nb, As, bs, mplu.default_options(**kw))
            assert st.converged == 1 and st.backward_error <= 2 * n * EPS
            np.testing.assert_allclose(xs[0].cpu().numpy(), single_ref[n]["x_ref"], rtol=0, atol=1e-12)
        # b = 0: x = 0 solves it exactly, so the backward error is 0, as in the single-GPU path
        xs, st = ds.gesv(n, nb, As, [b.new_zeros(n) for b in bs], mplu.default_options())
        assert st.converged == 1 and st.backward_error == 0.0 and st.first_backward_error == 0.0
        assert all((x == 0).all() for x in xs)
    finally:
        ds.close()


def test_dist_argument_errors(mplu):
    import ctypes
    lib = mplu.load_library()
    d = ctypes.c_void_p()
    assert lib.mplu_dist_create_local(ctypes.byref(d), 0, 0, 2) == -1
    ds = mplu.DistSolver(0, 1, 2)
    try:
        with pytest.raises(mplu.MpluError):
            ds.local_shape(0, 1000, 256)  # n % nb != 0
    finally:
        ds.close()


@pytest.mark.parametrize("peer_exchange", ["0", "1"])
def test_nccl_two_ranks(mplu, peer_exchange):
    """Two processes over NCCL.  peer_exchange = 1: the partial sums of the triangular solves travel through CUDA-IPC-mapped
    peer memory (px_send_kernel, the tile sweep waits for the slots itself) instead of ncclAllReduce: same iterations."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tools", "dist_nccl.py"), "4096", "512", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, MASTER_ADDR="127.0.0.1", MPLU_DIST_PEER_EXCHANGE=peer_exchange))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("DIST")][0]
    assert "conv 1" in line and "iters 2" in line
