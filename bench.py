#!/usr/bin/env python
"""bench.py -- LU+IR TFLOP/s (2/3 n^3) of the mixed-precision solver on synthetic diagonally dominant systems.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--n 32768] [--impl reference] [--dump-outputs DIR]

A "step" is one full solve of one n x n system: no-pivot LU in fp16 (fp32 accumulate) on the tcgen05 tensor cores +
fp64 iterative refinement to the dsgesv tolerance, inputs (fp64 A, b) already resident in HBM (`value`).  `e2e` is the
same solve through the C-ABI host entry point mplu_gesv_host(): pinned host A and b copied to the device and x copied
back inside the timed region.  One JSON line on stdout (rank 0).  See DESIGN.md section "Measurement".
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only; a benchmark run leaves nothing in it
PKG_NAME = "mixed-precision_lu_factorization_b200"
METRIC = "LU+IR TFLOP/s (2/3*n^3)"


def flops(n):
    return 2.0 / 3.0 * float(n) ** 3


def measured_traffic():
    """DRAM bytes of one rank-2048 update launch of the bulk lane from the committed ncu --set full capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "traffic_gemm_update.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    return dict(bytes_per_launch=d["dram_bytes_read"] + d["dram_bytes_write"], algorithmic_bytes=d["algorithmic_bytes"],
                shape=d["shape"], tensor_pipe_active_pct=d["tensor_pipe_active_pct"], source=d["source"])


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        # "under load": upper half of the samples
        load = sm[len(sm) // 2:] if sm else []
        return dict(sm_mhz=(load[len(load) // 2] if load else None), sm_max_mhz=(max(mx) if mx else None), reasons=reasons,
                    samples=len(sm))


def dump_outputs(d, **arrays):
    """--dump-outputs: what the timed path returned in its last timed step, one DIR/<name>.npy per array."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------------------
def cpu_lapack_baseline(n_sample):
    """Host LAPACK dgetrf + dgetrs on all host cores (the reference's CPU arm: LAPACKE_dgetrf at benchmark.cpp:240,
    plus the solve the metric adds), on a bounded sample size; TFLOP/s by the same 2/3 n^3 count."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import mplu_oracle as orc
    from scipy.linalg import lu_factor, lu_solve
    A = orc.counter_matrix_into(np.empty((n_sample, n_sample), order="F"), seed=1)
    b = A.sum(axis=1)
    lu_factor(A[:512, :512].copy())  # thread-pool warm-up
    t = time.perf_counter()
    lu, piv = lu_factor(A, check_finite=False)
    x = lu_solve((lu, piv), b, check_finite=False)
    dt = time.perf_counter() - t
    cores = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info
        th = [i["num_threads"] for i in threadpool_info() if i.get("internal_api") == "openblas"]
        cores = max(th) if th else cores
    except Exception:
        pass
    err = float(np.abs(x - 1).max())
    return dict(value=flops(n_sample) / dt / 1e12, unit="TFLOP/s", cores=cores, kind="reference",
                sample=f"scipy/OpenBLAS dgetrf+dgetrs, n={n_sample}, {dt:.2f} s, max|x-1|={err:.1e}")


def mpf_dropin_leg(m, n, reps=2):
    """The repo's drop-in MPF(double *A, int N, int r, int *IPIV) (include/MPF.h; the reference's entry point,
    /root/reference/MPF.h:3, with its semantics: fp16 pivot discovery + fp64 factors) timed the way benchmark.cpp:219-222
    times the reference: the whole call from a host buffer, r = 32.  The reference arm (--impl reference) reports the
    unmodified reference's MPF() at the same n as `reference_arm.mpf_same_n`."""
    import numpy as np
    import torch
    A, _ = m.generate(n, seed=1, with_rhs=False)
    hA0 = A.t().cpu().numpy()  # contiguous storage of A^T = column-major A
    del A
    torch.cuda.empty_cache()
    times = []
    for _ in range(reps + 1):
        hA = np.asfortranarray(hA0.T.copy(order="F"))
        t = time.perf_counter()
        ipiv = m.MPF(hA, 32)
        times.append(time.perf_counter() - t)
    dt = min(times[1:])
    return dict(value=flops(n) / dt / 1e12, unit="TFLOP/s", n=n, r=32, ms=1e3 * dt, what="repo drop-in MPF(), LU only, whole call incl. H2D/D2H",
                identity_pivots=bool((ipiv == np.arange(1, n + 1)).all()))


def run_reference(args):
    """--impl reference: the UNMODIFIED reference MPF() (oracle/_ref/libmpf_ref.so, built from /root/reference by
    oracle/Makefile; CUDA path, r = 32 as benchmark.cpp:220) timed as benchmark.cpp:219-222 times it (whole call,
    host buffers), next to host LAPACK on the box's cores.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import ctypes
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import mplu_oracle as orc
    n = args.n or 32768
    cpu = cpu_lapack_baseline(min(n, args.cpu_n))
    line = dict(impl="reference", metric=METRIC, unit="TFLOP/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=f"n={n} column-diagonally-dominant, reference MPF(A,n,32,ipiv) LU only (it has no solve)"))
    lib_path = os.path.join(ROOT, "oracle", "_ref", "libmpf_ref.so")
    have_gpu = False
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        pass
    if os.path.exists(lib_path) and have_gpu:
        lib = ctypes.CDLL(lib_path)
        f = getattr(lib, "_Z3MPFPdiiPi")
        f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        f.restype = None
        import torch
        n_ref = min(n, args.ref_n) if args.ref_n > 0 else n  # default: the repo arm's own n (same config)
        # the same generated input as the repo arm (mplu_generate == oracle.counter_matrix), built by column blocks
        A0 = np.empty((n_ref, n_ref), dtype=np.float64, order="F")
        orc.counter_matrix_into(A0, seed=1)
        A = np.empty_like(A0, order="F")
        devnull = os.open(os.devnull, os.O_WRONLY)
        times = []
        for it in range(args.warmup + args.steps):
            torch.from_numpy(A.T).copy_(torch.from_numpy(A0.T))  # MPF factors in place: fresh input every call (threaded copy)
            ipiv = np.arange(1, n_ref + 1, dtype=np.int32)
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(devnull, 1)  # MPF prints a line per panel
            t = time.perf_counter()
            f(A.ctypes.data, n_ref, 32, ipiv.ctypes.data)
            dt = time.perf_counter() - t
            os.dup2(saved, 1)
            os.close(saved)
            if it >= args.warmup:
                times.append(dt)
        ms = 1e3 * sum(times) / len(times)
        val = flops(n_ref) / (ms * 1e-3) / 1e12
        same_n = None
        if args.dropin_n > 0 and args.dropin_n != n_ref:  # the size the repo arm's mpf_dropin leg runs
            nd = args.dropin_n
            Ad0 = np.empty((nd, nd), dtype=np.float64, order="F")
            orc.counter_matrix_into(Ad0, seed=1)
            td = []
            for it in range(3):
                Ad = Ad0.copy(order="F")
                ipd = np.arange(1, nd + 1, dtype=np.int32)
                sys.stdout.flush()
                saved = os.dup(1)
                os.dup2(devnull, 1)
                t = time.perf_counter()
                f(Ad.ctypes.data, nd, 32, ipd.ctypes.data)
                td.append(time.perf_counter() - t)
                os.dup2(saved, 1)
                os.close(saved)
            same_n = dict(n=nd, ms=1e3 * min(td[1:]), value=flops(nd) / min(td[1:]) / 1e12, unit="TFLOP/s")
        line.update(value=val, ms_per_step=ms,
                    cpu_baseline=dict(value=val, unit="TFLOP/s", cores=1, kind="reference",
                                      sample=f"unmodified reference MPF() via oracle/_ref/libmpf_ref.so, n={n_ref}, r=32, one host "
                                             f"thread driving the GPU, whole call incl. cudaMalloc/H2D/D2H as benchmark.cpp:219-222"),
                    host_lapack=cpu,
                    e2e=dict(value=val, unit="TFLOP/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    reference_arm=dict(kind="reference CUDA path (unmodified MPF.cu, -O3 sm_100a)", n=n_ref, mpf_same_n=same_n,
                                       non_identity_pivots=int((ipiv != np.arange(1, n_ref + 1)).sum())))
        line["config"]["workload"] = f"n={n_ref} column-diagonally-dominant, reference MPF(A,n,32,ipiv) (LU only; it has no solve)"
    else:
        line.update(value=cpu["value"], ms_per_step=None, cpu_baseline=cpu,
                    e2e=dict(value=cpu["value"], unit="TFLOP/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        line["config"]["workload"] = cpu["sample"]
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
class stdout_to_stderr:
    """NCCL prints its version banner on stdout when it initialises; the contract is ONE JSON line on stdout, so the
    communicator set-up runs with file descriptor 1 pointed at stderr."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def run_distributed(args, m, pk, rank, world, local):
    """N > 1: ONE n x n system, 2D block-cyclic over a P x Q grid (one process per GPU, NCCL over NVLink)."""
    import torch
    import torch.distributed as dist
    n = args.n or 131072
    nb = args.nb or 2048
    P, Q = m.grid_shape(world)
    with stdout_to_stderr():
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.tensor(list(m.DistSolver.unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(uid, 0)
        ds = m.DistSolver(local, P, Q, rank=rank, unique_id=bytes(uid.cpu().tolist()))
        dist.barrier()
        torch.cuda.synchronize()
    opts = m.default_options(precision=1 if args.precision == "bf16" else 0)
    As, bs = ds.generate(n, nb, seed=1)
    p, q, mloc, nloc = ds.local_shape(0, n, nb)
    for _ in range(args.warmup):
        xs, st = ds.gesv(n, nb, As, bs, opts)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev_ms = tr_ms = tr_fl = tr_by = 0.0
    tr_n = launches = iters = 0
    worst_be = 0.0
    for _ in range(args.steps):
        xs, st = ds.gesv(n, nb, As, bs, opts)  # returns after its own stream sync; device time in st.total_ms
        dev_ms += st.total_ms
        tr_ms += st.trailing_ms; tr_fl += st.trailing_flops; tr_by += st.trailing_bytes; tr_n += st.trailing_launches
        launches += st.kernel_launches
        iters = max(iters, st.iters)
        worst_be = max(worst_be, st.backward_error)
    torch.cuda.synchronize()
    dist.barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    t = torch.tensor([dev_ms / args.steps, wall_ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, wall_max = float(t[0].item()), float(t[1].item())
    clocks = sampler.stop() if rank == 0 else None
    fwd_err = float((xs[0] - 1).abs().max().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x=xs[0].cpu().numpy())

    extra = dict(per_gpu_tflops=flops(n) / (ms_max * 1e-3) / 1e12 / world)
    if args.extra_n > 0:
        # the same curve on a system that also fits ONE GPU (bench.py --gpus 1 reports it under the same key)
        n2 = args.extra_n
        As2, bs2 = ds.generate(n2, nb, seed=1)
        best = None
        for i in range(3):
            xs2, st2 = ds.gesv(n2, nb, As2, bs2, opts)
            tt = torch.tensor([st2.total_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            if i and (best is None or float(tt.item()) < best[0]):
                best = (float(tt.item()), st2)
        extra["same_system"] = dict(n=n2, n_gpus=world, value=flops(n2) / (best[0] * 1e-3) / 1e12, unit="TFLOP/s", ms=best[0],
                                    ir_iters=best[1].iters, backward_error=best[1].backward_error,
                                    max_abs_err=float((xs2[0] - 1).abs().max().item()),
                                    what="ONE n x n system that fits a single GPU, 2D block-cyclic on these N GPUs")
        del As2, bs2, xs2
        torch.cuda.empty_cache()
        xs, st = ds.gesv(n, nb, As, bs, opts)  # back to the headline system (workspace sized for it again)

    e2e = None
    if not args.no_e2e:
        try:
            hA = torch.empty(max(nloc, 1), max(mloc, 1), dtype=torch.float64, pin_memory=True)
            hA.copy_(As[0].t())
            hb = bs[0].cpu().pin_memory()
            hx = torch.empty(n, dtype=torch.float64, pin_memory=True)
            del As
            torch.cuda.empty_cache()
            ds.gesv_host(n, nb, [hA.t()], [hb], [hx], opts)  # warm-up (staging allocation)
            torch.cuda.synchronize()
            dist.barrier()
            k_e2e = max(1, min(args.steps, 2))
            t1 = time.perf_counter()
            for _ in range(k_e2e):
                st_h = ds.gesv_host(n, nb, [hA.t()], [hb], [hx], opts)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t1) / k_e2e
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e = dict(value=flops(n) / float(tt.item()) / 1e12, unit="TFLOP/s", h2d_bytes_per_step=8 * n * n + 8 * n * world,
                       d2h_bytes_per_step=8 * n * world, ms_per_step=1e3 * float(tt.item()), h2d_ms=st_h.h2d_ms,
                       max_abs_err=float((hx - 1).abs().max().item()))
        except Exception as ex:  # e.g. not enough pinnable host memory for the local tiles
            e2e = dict(value=None, unit="TFLOP/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0, skipped=repr(ex)[:200])
    if rank == 0:
        value = flops(n) / (ms_max * 1e-3) / 1e12
        ach = (tr_fl / (tr_ms * 1e-3) / 1e12) if tr_ms > 0 else None
        line = dict(metric=METRIC, value=value, unit="TFLOP/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms_max, wall_ms_per_step=wall_max, higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype=args.precision + " operands, f32 accumulate, f64 refinement", data="synthetic",
                    config=dict(workload=f"n={n} 2D block-cyclic LU+IR across {world} B200 (BASELINE.json configs[3]); one system, "
                                         f"value = 2/3 n^3 / time", n=n, nb=nb, rhs=1, grid=f"{P}x{Q}",
                                matrix="column-diagonally-dominant, values k/10 (reference generator distribution), seed=1",
                                l2_policy="inputs larger than L2 (local A is %.1f GiB per GPU)" % (8.0 * mloc * nloc / 2 ** 30),
                                parallelism=f"2D block-cyclic {P}x{Q}, NCCL panel broadcasts, depth-1 look-ahead"),
                    ir_iters=iters, backward_error=worst_be, max_abs_err=fwd_err, factor_ms=st.factor_ms, solve_ms=st.solve_ms,
                    gpu_launches=launches, clocks=clocks, e2e=e2e,
                    roofline=dict(bound="tensor", kernel="gemm_tc_kernel (rank-nb trailing update, rank 0's launches)", achieved=ach,
                                  peak=pk["tc_sustained"], unit="TFLOP/s", frac=(ach / pk["tc_sustained"]) if ach else None,
                                  peak_kind=f"bf16_tflops_sustained ({pk['src']}); burst {pk['tc_burst']}", launches=tr_n,
                                  avg_launch_ms=(tr_ms / tr_n) if tr_n else None,
                                  share_of_step=(tr_ms / args.steps / ms_max) if ms_max > 0 else None,
                                  traffic=(measured_traffic() or {}).get("bytes_per_launch"), traffic_detail=measured_traffic()),
                    headline_frac_of_peak=value / world / pk["tc_sustained"], extra=extra)
        print(json.dumps(line), flush=True)
    ds.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", "--size", dest="n", type=int, default=0,
                    help="matrix order (default: 32768 on 1 GPU, 131072 block-cyclic on N > 1); under torchrun spell it --size (torchrun rejects --n as an ambiguous prefix of its own options)")
    ap.add_argument("--nb", type=int, default=0, help="outer block size (0 = library default for this n)")
    ap.add_argument("--precision", choices=["fp16", "bf16"], default="fp16")
    ap.add_argument("--impl", choices=["mplu", "reference"], default="mplu")
    ap.add_argument("--ref-n", type=int, default=0, help="size the reference arm runs (0 = the same n as the repo arm; the reference needs seconds per call)")
    ap.add_argument("--cpu-n", type=int, default=16384, help="sample size of the host LAPACK cpu_baseline leg (bounded: ~15 s of CPU work)")
    ap.add_argument("--dropin-n", type=int, default=16384, help="size of the mpf_dropin leg: the repo's drop-in MPF() (reference semantics: fp16 pivot search + fp64 factors), whole call from host buffers; 0 = skip")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--extra-n", type=int, default=65536, help="second workload reported under `extra`: ONE system of this order, which fits a single GPU, solved on the same N GPUs -- the 1 -> 8 curve read on one workload (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps write the solution of the last one as DIR/x.npy (float64, "
                    "--impl mplu); the inputs come from fixed seeds, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "mplu":
        ap.error("--dump-outputs needs --impl mplu")
    if args.warmup < 3:
        args.warmup = 3 if args.impl == "mplu" else args.warmup

    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        with stdout_to_stderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    m = importlib.import_module(PKG_NAME)
    pk = peaks()
    if world > 1:
        return run_distributed(args, m, pk, rank, world, local)
    n = args.n or 32768
    opts = m.default_options(precision=1 if args.precision == "bf16" else 0)
    if args.nb:
        opts.nb = args.nb

    solver = m.Solver(local)
    A, b = m.generate(n, seed=1 + rank)
    x = torch.empty(n, dtype=torch.float64, device="cuda")

    def step():
        return solver.gesv_ptr(n, A.data_ptr(), n, b.data_ptr(), x.data_ptr(), opts)

    for _ in range(args.warmup):
        st = step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.ExternalStream(solver.stream)
    tr_ms = tr_fl = tr_by = 0.0
    tr_n = launches = iters = 0
    worst_be = 0.0
    with torch.cuda.stream(stream):
        e0.record()
        for _ in range(args.steps):
            st = step()
            tr_ms += st.trailing_ms; tr_fl += st.trailing_flops; tr_by += st.trailing_bytes; tr_n += st.trailing_launches
            launches += st.kernel_launches
            iters = max(iters, st.iters)
            worst_be = max(worst_be, st.backward_error)
        e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    fwd_err = float((x - 1).abs().max().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x=x.cpu().numpy())

    # ---- e2e: host buffers through mplu_gesv_host (pinned memory), copies inside the timed region
    e2e = None
    if not args.no_e2e:
        hA = torch.empty(n, n, dtype=torch.float64, pin_memory=True)
        hA.copy_(A.t())  # A is column-major n x n: its transpose view is the contiguous storage
        hb = b.cpu().pin_memory()
        hx = torch.empty(n, dtype=torch.float64, pin_memory=True)
        solver.gesv_host_ptr(n, hA.data_ptr(), n, hb.data_ptr(), hx.data_ptr(), opts)  # warm-up (staging alloc)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        k_e2e = max(1, min(args.steps, 3))
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            st_h = solver.gesv_host_ptr(n, hA.data_ptr(), n, hb.data_ptr(), hx.data_ptr(), opts)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / k_e2e
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = dict(value=world * flops(n) / float(t.item()) / 1e12, unit="TFLOP/s", h2d_bytes_per_step=8 * n * n + 8 * n,
                   d2h_bytes_per_step=8 * n, ms_per_step=1e3 * float(t.item()), h2d_ms=st_h.h2d_ms,
                   max_abs_err=float((hx - 1).abs().max().item()))
        del hA

    extra = None
    if args.extra_n > 0 and world == 1:
        # the like-for-like single-GPU point of the multi-GPU curve (bench.py --gpus N reports the same system on N GPUs)
        n2 = args.extra_n
        del A, b, x
        torch.cuda.empty_cache()
        A2, b2 = m.generate(n2, seed=1)
        x2 = torch.empty(n2, dtype=torch.float64, device="cuda")
        best = None
        for i in range(3):  # first call: allocation + schedule capture
            st2 = solver.gesv_ptr(n2, A2.data_ptr(), n2, b2.data_ptr(), x2.data_ptr(), opts)
            if i and (best is None or st2.total_ms < best.total_ms):
                best = st2
        extra = dict(per_gpu_tflops=world * flops(n) / (ms_max * 1e-3) / 1e12 / world,
                     same_system=dict(n=n2, n_gpus=1, value=flops(n2) / (best.total_ms * 1e-3) / 1e12, unit="TFLOP/s", ms=best.total_ms,
                                      ir_iters=best.iters, backward_error=best.backward_error,
                                      max_abs_err=float((x2 - 1).abs().max().item()),
                                      what="ONE n x n system that fits a single GPU; `bench.py --gpus N` solves the same system block-cyclic on N GPUs"))
        del A2, b2, x2

    if rank == 0:
        num_sms = torch.cuda.get_device_properties(local).multi_processor_count
        left = int(opts.schedule) == 1
        bulk_sms = num_sms - (int(opts.side_sms_left) if left else int(opts.side_sms))
        value = world * flops(n) / (ms_max * 1e-3) / 1e12
        ach = (tr_fl / (tr_ms * 1e-3) / 1e12) if tr_ms > 0 else None
        line = dict(metric=METRIC, value=value, unit="TFLOP/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms_max, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype=args.precision + " operands, f32 accumulate, f64 refinement", data="synthetic",
                    config=dict(workload=f"n={n} mixed-precision LU+IR on 1 B200 per rank (BASELINE.json configs[2])" if n == 32768
                                else f"n={n} mixed-precision LU+IR", n=n,
                                nb=int(opts.nb) or (2048 if n >= 12288 else (1024 if n >= 4096 else 512)), rhs=1,
                                schedule="left-looking block columns, look-ahead + eager updates" if int(opts.schedule) == 1
                                else "right-looking, depth-1 look-ahead",
                                host_path="streamed by block columns behind the H2D copy" if int(opts.stream_host) else "copy, then solve",
                                matrix="column-diagonally-dominant, values k/10 (reference generator distribution), seed=1+rank",
                                l2_policy="inputs larger than L2 (A is %.1f GiB)" % (8.0 * n * n / 2 ** 30),
                                parallelism=("replicas x%d" % world) if world > 1 else "single GPU"),
                    ir_iters=iters, backward_error=worst_be, max_abs_err=fwd_err,
                    factor_ms=st.factor_ms, solve_ms=st.solve_ms,
                    gpu_launches=launches, clocks=clocks, e2e=e2e,
                    roofline=dict(bound="tensor", kernel="gemm_tc_kernel (rank-nb Schur updates of the bulk lane)", achieved=ach,
                                  peak=pk["tc_sustained"], unit="TFLOP/s", frac=(ach / pk["tc_sustained"]) if ach else None,
                                  peak_kind=f"bf16_tflops_sustained ({pk['src']}); burst {pk['tc_burst']}",
                                  # these launches run on the bulk lane's SM budget while the chain lane factors the next
                                  # diagonal tile on the other SMs: frac is against the WHOLE GPU's peak
                                  sms=bulk_sms, sms_total=num_sms,
                                  frac_of_lane_peak=(ach / (pk["tc_sustained"] * bulk_sms / num_sms)) if ach else None,
                                  launches=tr_n, avg_launch_ms=(tr_ms / tr_n) if tr_n else None,
                                  share_of_step=(tr_ms / args.steps / ms) if ms > 0 else None,
                                  algorithmic_c_bytes_per_s=(tr_by / (tr_ms * 1e-3) / 1e9) if tr_ms > 0 else None,
                                  traffic=(measured_traffic() or {}).get("bytes_per_launch"), traffic_detail=measured_traffic()),
                    headline_frac_of_peak=value / world / pk["tc_sustained"])
        if extra:
            line["extra"] = extra
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = dict(cpu_lapack_baseline(min(n, args.cpu_n)), kind="port")
        if args.dropin_n > 0:
            line["mpf_dropin"] = mpf_dropin_leg(m, args.dropin_n)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
