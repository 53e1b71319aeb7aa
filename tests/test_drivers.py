"""The two C++ drivers keep the reference's CLI and file formats (SURVEY.md section 8b "Driver formats")."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

GEN = os.path.join(ROOT, "drivers", "matrix_generator")
BENCH = os.path.join(ROOT, "drivers", "benchmark")
REF_GEN = os.path.join(ROOT, "oracle", "_ref", "matgen")  # the unmodified reference generator (oracle/Makefile)


def read_matrices(path):
    """Parse the generator format the way benchmark.cpp:171-194 does: values sequentially, column-major storage."""
    tok = open(path).read().split()
    count, pos, out = int(tok[0]), 1, []
    for _ in range(count):
        n = int(tok[pos]); pos += 1
        vals = np.array(tok[pos:pos + n * n], dtype=np.float64); pos += n * n
        out.append(vals.reshape(n, n).T.copy())  # element e -> column e // n, row e % n
    return out


@pytest.mark.parametrize("args", [["64", "2", "exp"], ["40", "3", "lin"], ["33", "2", "exp", "0.5"], ["20", "7", "lin", "0.9"]])
def test_generator_is_byte_identical_to_the_reference(mplu, tmp_path, args):
    """The expected files are stored in tests/golden/, since the reference generator is not part of the repository: they
    were written by this generator, whose rand path is unchanged since this test compared it with the reference's, and
    the dense ones agree value for value with the oracle's restatement on libc rand().  When oracle/_ref/matgen is
    built, the reference is compared with them as well."""
    with gzip.open(os.path.join(GOLDEN, "matrix_generator_" + "_".join(args) + ".txt.gz")) as fh:
        want = fh.read()
    a = tmp_path / "mine.txt"
    subprocess.run([GEN, str(a), *args], check=True, capture_output=True)
    assert a.read_bytes() == want
    if os.path.exists(REF_GEN):
        b = tmp_path / "ref.txt"
        subprocess.run([REF_GEN, str(b), *args], check=True, capture_output=True)
        assert b.read_bytes() == want


def test_generator_first_matrix_matches_libc_rand_pin(mplu, oracle, tmp_path):
    """SURVEY.md section 8b [probe]: the first 2x2 the generator emits is 8.3 8.6 / 7.7 1.5 (glibc rand(), seed 1)."""
    f = tmp_path / "m.txt"
    subprocess.run([GEN, str(f), "2"], check=True, capture_output=True)
    lines = f.read_text().splitlines()
    assert lines[0].strip() == "1" and lines[1] == "2"
    assert lines[2].split() == ["8.3", "8.6"] and lines[3].split() == ["7.7", "1.5"]


def test_generator_dd_mode_is_column_dominant_as_read_by_the_driver(mplu, tmp_path):
    f, g = tmp_path / "dd.txt", tmp_path / "rand.txt"
    subprocess.run([GEN, str(f), "64", "2", "exp", "0.0", "dd"], check=True, capture_output=True)
    subprocess.run([GEN, str(g), "64", "2", "exp", "0.0", "rand"], check=True, capture_output=True)
    for A, R in zip(read_matrices(f), read_matrices(g)):
        n = A.shape[0]
        off = np.abs(A).sum(axis=0) - np.abs(np.diag(A))
        assert np.all(np.abs(np.diag(A)) > off)           # strictly column diagonally dominant
        mask = ~np.eye(n, dtype=bool)
        assert np.array_equal(A[mask], R[mask])           # same rand() draws off the diagonal


def test_generator_spd_kappa_mode(mplu, tmp_path):
    f = tmp_path / "spd.txt"
    subprocess.run([GEN, str(f), "32", "2", "exp", "0.0", "spd:1e4:7"], check=True, capture_output=True)
    for A in read_matrices(f):
        n = A.shape[0]
        assert np.abs(A - A.T).max() <= 1e-15
        w = np.linalg.eigvalsh(A)
        assert w.min() > 0 and abs(w.max() - 1.0) < 1e-12 and abs(w.max() / w.min() / 1e4 - 1.0) < 1e-6


def test_generator_usage_and_argument_errors(mplu, tmp_path):
    assert subprocess.run([GEN], capture_output=True).returncode != 0
    for bad in (["0"], ["8", "0"], ["8", "2", "cubic"], ["8", "2", "exp", "1.5"], ["8", "2", "exp", "0.0", "spd"]):
        r = subprocess.run([GEN, str(tmp_path / "x.txt"), *bad], capture_output=True, text=True)
        assert r.returncode != 0 and "Invalid" in r.stdout


def test_benchmark_driver_csv_header_is_the_reference_one(mplu, tmp_path):
    """Runs without a GPU too: MPF() then reports the missing device like the reference (MPF.cu:72-75)."""
    f = tmp_path / "m.txt"
    subprocess.run([GEN, str(f), "8"], check=True, capture_output=True)
    r = subprocess.run([BENCH, str(f), "--no-check"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0
    rows = (tmp_path / "benchmark_times.csv").read_text().splitlines()
    assert rows[0] == "matrix_size,mpf_time,lapack_time"
    assert [int(x.split(",")[0]) for x in rows[1:]] == [2, 4, 8]
    assert all(len(x.split(",")[1].split(".")[1]) == 10 for x in rows[1:])  # fixed, 10 decimals (benchmark.cpp:169)


@pytest.mark.gpu
def test_benchmark_driver_end_to_end_on_gpu(mplu, tmp_path):
    f = tmp_path / "dd.txt"
    subprocess.run([GEN, str(f), "1024", "2", "exp", "0.0", "dd"], check=True, capture_output=True)
    r = subprocess.run([BENCH, str(f), "--solve", "--csv", str(tmp_path / "out.csv")], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "incorrect" not in r.stdout, r.stdout          # MPF and LAPACK both pass the P*L*U == A check
    rows = (tmp_path / "out.csv").read_text().splitlines()
    assert rows[0] == "matrix_size,mpf_time,lapack_time,mplu_time,iters,backward_error,mplu_tflops"
    last = rows[-1].split(",")
    assert int(last[0]) == 1024 and int(last[4]) <= 3 and float(last[5]) < 1e-12 and float(last[6]) > 0
    assert "Matriz tamanyo: 1024" in r.stdout  # the reference's own line (benchmark.cpp:236)


@pytest.mark.gpu
def test_benchmark_driver_random_matrices_need_pivoting_and_pass(mplu, tmp_path):
    """reference distribution (not dominant): MPF's fp16 pivot discovery + fp64 factors must pass the 1e-10 check at
    the sizes where the reference passes it"""
    f = tmp_path / "r.txt"
    subprocess.run([GEN, str(f), "64", "2", "exp"], check=True, capture_output=True)
    r = subprocess.run([BENCH, str(f)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0 and "MPF produced incorrect results." not in r.stdout, r.stdout


def test_benchmark_driver_usage_and_exit_codes_are_the_references(mplu, tmp_path):
    """benchmark.cpp:148-151,162-165: usage line / unreadable file -> return -1 (exit status 255)"""
    r = subprocess.run([BENCH], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout.startswith("Usage: ")
    r = subprocess.run([BENCH, str(tmp_path / "missing.txt")], capture_output=True, text=True)
    assert r.returncode == 255 and "Failed to open" in r.stdout
    bad = tmp_path / "bad.txt"
    bad.write_text("0\n")
    r = subprocess.run([BENCH, str(bad)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 255 and "Invalid number of matrices" in r.stdout


@pytest.mark.gpu
def test_benchmark_driver_binary_input_n8192(mplu, tmp_path):
    """--bin: int32 count, then int32 n + n*n float64 (column-major) per matrix -- the input mode that reaches the sizes
    the text format cannot; n = 8192 dominant system through MPF() (checked by the driver) and through LU + IR"""
    import numpy as np
    import torch
    n = 8192
    A, _ = mplu.generate(n, seed=3, with_rhs=False)
    f = tmp_path / "m.bin"
    with open(f, "wb") as fh:
        np.array([1, n], dtype=np.int32).tofile(fh)
        A.t().cpu().numpy().tofile(fh)  # contiguous storage of A^T = column-major A
    # --no-check: the reference's check is an ABSOLUTE 1e-10 on P*L*U - A (benchmark.cpp:97-104), which no fp64 LU of a
    # matrix with entries ~4e4 meets at this size; the refined solve's backward error is the check here
    r = subprocess.run([BENCH, str(f), "--bin", "--no-check", "--solve", "--csv", str(tmp_path / "out.csv")], cwd=tmp_path,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "Matriz tamanyo: 8192" in r.stdout
    last = (tmp_path / "out.csv").read_text().splitlines()[-1].split(",")
    assert int(last[0]) == n and int(last[4]) <= 3 and float(last[5]) < 1e-15 * n


@pytest.mark.gpu
def test_benchmark_driver_generated_on_device(mplu, tmp_path):
    """--gen dd:N: the headline workload without any host copy of A (mplu_generate + mplu_gesv_device)"""
    r = subprocess.run([BENCH, "--gen", "dd:8192:5", "--csv", str(tmp_path / "g.csv")], cwd=tmp_path, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = (tmp_path / "g.csv").read_text().splitlines()
    assert rows[0] == "matrix_size,mpf_time,lapack_time,mplu_time,iters,backward_error,mplu_tflops"
    last = rows[1].split(",")
    assert int(last[0]) == 8192 and int(last[4]) <= 3 and float(last[5]) < 1e-11 and float(last[6]) > 10
