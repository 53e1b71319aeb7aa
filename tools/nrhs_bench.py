#!/usr/bin/env python
"""Several right-hand sides: the batched solve against a loop of single-vector solves.

    python tools/nrhs_bench.py [--n 32768] [--nrhs 1,2,4,8,16,32,64] [--reps 3] [--out FILE] [--profile]

Synthetic diagonally dominant system (mplu_generate, seed 1), B = A X_true with standard-normal X_true columns.
Per nrhs, with the factors stored once (mplu_factor_device), device events on the solver's stream around
  loop:    mplu_solve_device over the columns, one after the other
  batched: mplu_solve_device_nrhs on the whole block
and the whole call mplu_gesv_device_nrhs (factor + batched solve).  Median of --reps timed runs after one warm-up.
One JSON line per nrhs on stdout (and appended to --out), with the card's name and power limit read in the same run.
bytes_per_s: the algorithmic traffic of the solve phase -- 8 n^2 per residual pass and 4 n^2 per triangular-solve pair,
per column block (16 columns per residual launch, 8 per solve launch; one column each in the loop) -- over the time.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
PKG_NAME = "mixed-precision_lu_factorization_b200"
RES_BLOCK, SOLVE_BLOCK = 16, 8  # kResidualBlock / kSolveBlock of csrc/kernels.h


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else (None, None, None)
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def solve_bytes(n, nrhs, iters, batched):
    """first solve + `iters` (residual + solve) + the final residual: iters + 1 of each"""
    res_blocks = -(-nrhs // RES_BLOCK) if batched else nrhs
    sol_blocks = -(-nrhs // SOLVE_BLOCK) if batched else nrhs
    return (iters + 1) * (8.0 * n * n * res_blocks + 4.0 * n * n * sol_blocks)


def profile_kernels(fn):
    """{kernel name: [launches, summed device ms]} of one call of fn"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if us > 0 and "Memset" not in e.key and "Memcpy" not in e.key:
            # "void mplu::(anonymous namespace)::name<args>(params)" -> "name<args>"
            name = e.key.replace("(anonymous namespace)::", "").split("(")[0].replace("void ", "").split("::")[-1]
            cnt, ms = out.get(name, [0, 0.0])
            out[name] = [cnt + e.count, ms + us / 1e3]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=32768)
    ap.add_argument("--nrhs", default="1,2,4,8,16,32,64")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also append the JSON lines to this file")
    ap.add_argument("--profile", action="store_true", help="add the per-kernel device time of one batched solve "
                    "(torch.profiler, after the timed runs) to each line")
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("nrhs_bench.py needs a CUDA device")
    m = importlib.import_module(PKG_NAME)
    n = args.n
    info = card()
    s = m.Solver(0)
    A, _ = m.generate(n, seed=1, with_rhs=False)
    lda = A.stride(1)
    opts = m.default_options()
    stream = torch.cuda.ExternalStream(s.stream)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            e0.record()
            out = fn()
            e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    out = open(args.out, "a") if args.out else None
    for k in [int(v) for v in args.nrhs.split(",")]:
        g = torch.Generator(device="cuda").manual_seed(k)
        Xt = torch.randn(k, n, dtype=torch.float64, device="cuda", generator=g).t()  # column-major n x k
        B = torch.empty(k, n, dtype=torch.float64, device="cuda").t()
        B.copy_(A @ Xt)
        X = torch.empty(k, n, dtype=torch.float64, device="cuda").t()
        cols = [B[:, j].contiguous() for j in range(k)]
        torch.cuda.synchronize()
        s.factor_ptr(n, A.data_ptr(), lda, opts)

        def loop():
            its = []
            for j in range(k):
                its.append(s.solve_ptr(A.data_ptr(), lda, cols[j].data_ptr(), X[:, j].data_ptr()).iters)
            return its

        def batched():
            st, berr = s.solve_nrhs_ptr(k, A.data_ptr(), lda, B.data_ptr(), n, X.data_ptr(), n)
            return st, berr

        def whole():
            return s.gesv_nrhs_ptr(n, k, A.data_ptr(), lda, B.data_ptr(), n, X.data_ptr(), n, opts)

        res = {}
        for name, fn in (("loop", loop), ("batched", batched)):
            fn()  # warm-up
            runs = [timed(fn) for _ in range(args.reps)]
            res[name] = (statistics.median(r[0] for r in runs), runs[-1][1])
        loop_ms, loop_iters = res["loop"]
        bat_ms, (bst, bberr) = res["batched"]
        fwd_err = float(((X - Xt).abs().max(dim=0).values / Xt.abs().max(dim=0).values).max().item())
        kernels = profile_kernels(batched) if args.profile else None
        whole()
        wruns = [timed(whole) for _ in range(args.reps)]
        w_ms = statistics.median(r[0] for r in wruns)
        wst, wberr = wruns[-1][1]
        line = dict(
            n=n, nrhs=k, card=info,
            loop=dict(ms=loop_ms, ms_per_col=loop_ms / k, iters=max(loop_iters), iters_min=min(loop_iters),
                      bytes_per_s=sum(solve_bytes(n, 1, it, False) for it in loop_iters) / (loop_ms * 1e-3)),
            batched=dict(ms=bat_ms, ms_per_col=bat_ms / k, iters=bst.iters, worst_backward_error=float(np.max(bberr)),
                         converged=bst.converged, max_rel_fwd_err=fwd_err,
                         bytes_per_s=solve_bytes(n, k, bst.iters, True) / (bat_ms * 1e-3)),
            speedup=loop_ms / bat_ms,
            gesv=dict(ms=w_ms, ms_per_col=w_ms / k, factor_ms=wst.factor_ms, iters=wst.iters,
                      worst_backward_error=float(np.max(wberr)), converged=wst.converged),
            kernels=kernels,
            what="solve phase with stored factors: loop of mplu_solve_device vs mplu_solve_device_nrhs (device events on "
                 "the solver's stream, median of %d); gesv = whole mplu_gesv_device_nrhs call" % args.reps)
        js = json.dumps(line)
        print(js, flush=True)
        if out:
            out.write(js + "\n")
            out.flush()
        del Xt, B, X, cols
    s.close()


if __name__ == "__main__":
    main()
