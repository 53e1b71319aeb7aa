"""Host reference of the equilibration (mplu_options::equilibrate, csrc/equil.cu): LAPACK dgeequb's power-of-two scales,
dlaqge's decision (EQUED) and dsgesv refinement with equilibrated factors, for the emulation in mplu_oracle."""
from __future__ import annotations

import math

import numpy as np

SMLNUM = np.finfo(np.float64).tiny          # dlamch('S') = 2^-1022
BIGNUM = 1.0 / SMLNUM
SMALL = SMLNUM / np.finfo(np.float64).eps   # dlaqge: dlamch('S') / dlamch('P') = 2^-970
LARGE = 1.0 / SMALL
THRESH = 0.1
EQUED_CODE = {"N": 0, "R": 1, "C": 2, "B": 3}


def pow2_trunc_log2(m: float) -> float:
    """2^int(log2 m) for a finite m > 0, int() truncating toward zero (dgeequb's RADIX**INT(LOG(m)/LOG(RADIX))), exactly:
    m = f 2^k with f in [0.5, 1) gives the exponent k - 1 if m >= 1, else k if f > 0.5, else k - 1."""
    f, k = math.frexp(m)
    return math.ldexp(1.0, k - 1 if m >= 1.0 else (k if f > 0.5 else k - 1))


def _scales(maxima):
    p = np.array([pow2_trunc_log2(float(v)) if v > 0 else 0.0 for v in maxima])
    rcmin, rcmax = float(p.min()), float(p.max())
    s = 1.0 / np.minimum(np.maximum(p, SMLNUM), BIGNUM)
    return p, s, rcmin, rcmax


def geequb_pow2(A):
    """dgeequb of the square matrix A: (r, c, rowcnd, colcnd, amax, info) like scipy.linalg.lapack.dgeequb.  info = i + 1
    for the first zero row i, n + j + 1 for the first zero column j (r / c are not meaningful then)."""
    A = np.asarray(A, dtype=np.float64)
    n = A.shape[0]
    rm = np.abs(A).max(axis=1)
    p, r, rmin, rmax = _scales(rm)
    amax = rmax
    if rmin == 0.0:
        return r, np.ones(A.shape[1]), 0.0, 0.0, amax, int(np.flatnonzero(p == 0)[0]) + 1
    rowcnd = max(rmin, SMLNUM) / min(rmax, BIGNUM)
    cm = (np.abs(A) * r[:, None]).max(axis=0)
    q, c, cmin, cmax = _scales(cm)
    if cmin == 0.0:
        return r, c, rowcnd, 0.0, amax, n + int(np.flatnonzero(q == 0)[0]) + 1
    return r, c, rowcnd, max(cmin, SMLNUM) / min(cmax, BIGNUM), amax, 0


def laqge_equed(rowcnd: float, colcnd: float, amax: float) -> str:
    """dlaqge's choice: rows when ROWCND < 0.1 or AMAX outside [SMALL, LARGE], columns when COLCND < 0.1."""
    rows = not (rowcnd >= THRESH and SMALL <= amax <= LARGE)
    cols = not (colcnd >= THRESH)
    return "B" if rows and cols else ("R" if rows else ("C" if cols else "N"))


def equilibrate(A):
    """What the solver does with opts.equilibrate = 1: (EQUED code 0..3, r, c) with ones on a side that is not applied.
    A zero row or column (dgeequb INFO > 0) or a non-finite entry: no equilibration."""
    A = np.asarray(A, dtype=np.float64)
    n = A.shape[0]
    one = np.ones(n)
    if not np.isfinite(A).all():
        return 0, one, one.copy()
    r, c, rowcnd, colcnd, amax, info = geequb_pow2(A)
    if info:
        return 0, one, one.copy()
    e = EQUED_CODE[laqge_equed(rowcnd, colcnd, amax)]
    return e, (r if e & 1 else one), (c if e & 2 else one.copy())


def refine_equilibrated(oracle, A, b, r, c, nb: int = 128, bf16: bool = False, max_iters: int = 30):
    """oracle.refine with the emulated factors of diag(r) A diag(c): x0 = c (LU)^-1 (r b), x += c (LU)^-1 (r (b - A x)),
    the residual, norms and stopping rule those of the original A (dsgesv's)."""
    A = np.asarray(A, dtype=np.float64)
    n = A.shape[0]
    with np.errstate(all="ignore"):
        LU = oracle.lu_mixed_emulated(r[:, None] * A * c[None, :], nb=nb, bf16=bf16)
    anorm = np.abs(A).sum(axis=1).max()
    bnorm = np.abs(b).max()
    eps = np.finfo(np.float64).eps / 2
    x = c * oracle.lu_solve(LU, r * b).astype(np.float64)
    iters, conv, first = 0, False, None
    while True:
        res = b - A @ x
        rn, xn = np.abs(res).max(), np.abs(x).max()
        be = rn / (anorm * xn + bnorm)
        first = be if first is None else first
        if not np.isfinite(rn):
            break
        if rn <= xn * anorm * eps * math.sqrt(n):
            conv = True
            break
        if iters >= max_iters:
            break
        x = x + c * oracle.lu_solve(LU, r * res).astype(np.float64)
        iters += 1
    return dict(x=x, iters=iters, converged=conv, backward_error=be, first_backward_error=first)
