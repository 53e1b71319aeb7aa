#!/usr/bin/env python
"""Equilibration (opts.equilibrate): its cost on a well-scaled system and what it saves on badly scaled ones.

    python tools/equilibrate_bench.py [--reps 5] [--out profiles/r04_equilibrate.json]

Cases, each solved with equilibrate = 0 and 1 in alternation (one warm-up call each first, then --reps pairs; medians
with min / max of the device time of the whole mplu_gesv_device call, stats.total_ms):
  dominant_n32768       the synthetic dominant system (mplu_generate, seed 1): EQUED = N, the cost of the two passes
  rows2pm6_n32768       the same matrix with its rows scaled by seeded powers of two in 2^+-6
  spd1e6_2pm6_n16384    generate_spd(16384, 1e6) with rows and columns scaled by powers of two in 2^+-6
For each case the path that ran (EQUED, precision_used, fp64_fallback, dsgesv_iter, iterations).
kernels: one equilibrated solve of rows2pm6_n32768 under torch.profiler in a run of its own; row pass, column pass and
scaled first touch with their algorithmic bytes (8 n^2 read each pass; the first touch 8 n^2 read + 4 n^2 written) over
their device time.  ptxas: the -Xptxas -v lines of the new kernels, compiled for sm_100a in a temporary directory.
The card's name, power limit and maximum SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
PKG_NAME = "mixed-precision_lu_factorization_b200"
CSRC = os.path.join(ROOT, PKG_NAME, "csrc")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else (None, None, None)
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def ptxas_lines():
    """registers / shared memory / spills of the equilibration kernels and of both first-touch instantiations"""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    out = []
    with tempfile.TemporaryDirectory() as tmp:
        for src in ("equil.cu", "panel.cu"):
            r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I",
                                os.path.join(ROOT, "include"), "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o",
                                os.path.join(tmp, src + ".o")], capture_output=True, text=True)
            lines = r.stderr.splitlines()
            for i, l in enumerate(lines):
                if "Compiling entry function" in l and ("equil" in l or "diag_scale" in l or "first_touch" in l):
                    out.append(" | ".join(x.strip() for x in lines[i:i + 4] if "ptxas info" in x or "spill" in x))
    return out


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
            name = e.key.replace("(anonymous namespace)::", "").split("(")[0].replace("void ", "").split("::")[-1]
            cnt, ms = out.get(name, [0, 0.0])
            out[name] = [cnt + e.count, ms + us / 1e3]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="write the JSON document to this file as well")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("equilibrate_bench.py needs a CUDA device")
    m = importlib.import_module(PKG_NAME)
    doc = dict(card=card(), reps=args.reps, cases={})
    s = m.Solver(0)

    def pow2(n, spread, seed):
        g = torch.Generator(device="cuda").manual_seed(seed)
        return 2.0 ** torch.randint(-spread, spread + 1, (n,), generator=g, device="cuda").double()

    def run(name, A, b):
        n = A.shape[0]
        x = torch.empty(n, dtype=torch.float64, device="cuda")
        opts = {e: m.default_options(equilibrate=e) for e in (0, 1)}
        last, ms = {}, {0: [], 1: []}
        for e in (0, 1):  # warm-up: graph capture, workspaces
            s.gesv_ptr(n, A.data_ptr(), A.stride(1), b.data_ptr(), x.data_ptr(), opts[e], allow_noconv=True)
        for _ in range(args.reps):
            for e in (0, 1):
                st = s.gesv_ptr(n, A.data_ptr(), A.stride(1), b.data_ptr(), x.data_ptr(), opts[e], allow_noconv=True)
                ms[e].append(st.total_ms)
                last[e] = st
        res = {}
        for e in (0, 1):
            st = last[e]
            res[f"equilibrate{e}"] = dict(
                total_ms_median=statistics.median(ms[e]), total_ms_min=min(ms[e]), total_ms_max=max(ms[e]),
                factor_ms=st.factor_ms, equed=st.equed, precision_used=st.precision_used, fp64_fallback=st.fp64_fallback,
                dsgesv_iter=st.dsgesv_iter, iters=st.iters, converged=st.converged, status_bits=st.status_bits,
                backward_error=st.backward_error)
        res["difference_ms_median"] = res["equilibrate1"]["total_ms_median"] - res["equilibrate0"]["total_ms_median"]
        doc["cases"][name] = res
        print(json.dumps({name: res}), flush=True)

    n = 32768
    A, b = m.generate(n, seed=1)
    run("dominant_n32768", A, b)
    A.mul_(pow2(n, 6, seed=7)[:, None])  # diag(d1) A: rows scaled; b scaled alike keeps the solution
    b.mul_(pow2(n, 6, seed=7))
    run("rows2pm6_n32768", A, b)
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    opts = m.default_options(equilibrate=1)
    kern = profile_kernels(lambda: s.gesv_ptr(n, A.data_ptr(), n, b.data_ptr(), x.data_ptr(), opts, allow_noconv=True))
    gb = {"equil_row_max_kernel": 8.0 * n * n, "equil_col_kernel": 8.0 * n * n, "first_touch_kernel<true>": 12.0 * n * n}
    doc["kernels_rows2pm6_n32768"] = {
        k: dict(launches=v[0], ms=v[1], gbytes=gb[k] / 1e9, tbytes_per_s=gb[k] / (v[1] * 1e-3) / 1e12)
        for k, v in kern.items() if k in gb}
    doc["kernels_rows2pm6_n32768_other"] = {k: dict(launches=v[0], ms=v[1]) for k, v in kern.items()
                                             if k not in gb and ("equil" in k or "scale" in k or "first_touch" in k)}
    print(json.dumps({"kernels": doc["kernels_rows2pm6_n32768"]}), flush=True)
    del A, b, x
    torch.cuda.empty_cache()

    n = 16384
    A0 = m.generate_spd(n, 1e6, seed=1)
    A = (pow2(n, 6, seed=11)[:, None] * A0 * pow2(n, 6, seed=12)[None, :]).t().contiguous().t()
    del A0
    g = torch.Generator(device="cuda").manual_seed(13)
    b = (A @ torch.randn(n, dtype=torch.float64, device="cuda", generator=g)).contiguous()
    run("spd1e6_2pm6_n16384", A, b)
    s.close()
    doc["ptxas"] = ptxas_lines()
    doc["what"] = ("device time of whole mplu_gesv_device calls (stats.total_ms, CUDA events), equilibrate 0 and 1 "
                   "alternating after one warm-up each; kernel times from torch.profiler in a separate call")
    js = json.dumps(doc, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(js + "\n")
    print(js)


if __name__ == "__main__":
    main()
