"""qrcp_numpy.py — NumPy restatement of the pivoted-QR rescue of csrc/dense.cu (`qrcp_kernel`, `qrcp_solve_kernel`).
TEST INFRASTRUCTURE ONLY.

When the dense LU of a Newton step reports a zero pivot the driver solves the step in the least-squares sense instead
(the reference's default dense solver falls back from a failed LU to a column-pivoted QR).  This file states the same
algorithm step by step, so the tests can hold the kernel's iterate to it:

  * unblocked Householder QR with column pivoting; the squared norms of the trailing columns are recomputed at every step
    (not downdated), and the column with the largest norm is taken, the lowest index winning ties;
  * LAPACK `dlarfg` reflectors: beta = -sign(alpha) ||x||, tau = (beta - alpha) / beta, v = (1, x[1:] / (alpha - beta));
    tau = 0 when the part below the diagonal is exactly zero;
  * numerical rank r = 1 + the last k with |R_kk| > n eps |R_00|;
  * basic solution x = P [R11^-1 (Q'b)(1:r) ; 0].

Every per-column quantity is computed by elementwise operations and reductions along the column, so two identical columns
stay bit-identical here as they do in the kernel, and an exact tie between them is resolved by the index alone."""
import math

import numpy as np


def qrcp(A):
    """Factor a copy of the square matrix A.  Returns (QR, tau, jpvt, rank): R in the upper triangle, the Householder
    vectors below it (v_k = 1 implied), the column permutation (column k of QR came from column jpvt[k] of A)."""
    A = np.array(A, dtype=np.float64, order="F", copy=True)
    n = A.shape[0]
    assert A.shape == (n, n)
    tau = np.zeros(n)
    jpvt = np.arange(n)
    thr = n * np.finfo(np.float64).eps
    r00, rank = 0.0, 0
    for k in range(n):
        T = A[k:, k:]
        cn = np.einsum("ij,ij->j", T, T)
        p = k + int(np.argmax(cn))  # first maximum: the lowest index wins ties
        cn2 = float(cn[p - k])
        if p != k:
            A[:, [k, p]] = A[:, [p, k]]
            jpvt[[k, p]] = jpvt[[p, k]]
        alpha = float(A[k, k])
        xn2 = max(cn2 - alpha * alpha, 0.0)
        beta = t = scal = 0.0
        if xn2 > 0.0 or alpha != 0.0:
            beta = -math.copysign(math.sqrt(alpha * alpha + xn2), alpha)
            t = (beta - alpha) / beta
            scal = 1.0 / (alpha - beta) if xn2 > 0.0 else 0.0
            if xn2 == 0.0:
                beta, t = alpha, 0.0
        A[k, k] = beta
        tau[k] = t
        A[k + 1:, k] *= scal
        if k == 0:
            r00 = abs(beta)
        if abs(beta) > thr * r00:
            rank = k + 1
        if t != 0.0 and k + 1 < n:
            v = A[k + 1:, k]
            S = A[k:, k + 1:]
            w = (S[0] + np.einsum("ij,i->j", S[1:], v)) * t
            S[0] -= w
            S[1:] -= v[:, None] * w[None, :]
    return A, tau, jpvt, rank


def qrcp_solve(QR, tau, jpvt, rank, b):
    """The basic solution x = P [R11^-1 (Q'b)(1:rank) ; 0] from the factors of qrcp()."""
    c = np.array(b, dtype=np.float64, copy=True)
    n = len(c)
    for k in range(n):  # c = Q' b, reflectors in order
        v = QR[k + 1:, k]
        s = (float(v @ c[k + 1:]) + c[k]) * tau[k]
        c[k] -= s
        c[k + 1:] -= s * v
    for k in range(rank - 1, -1, -1):  # R11 y = c(1:rank), column-oriented back substitution
        c[k] /= QR[k, k]
        c[:k] -= QR[:k, k] * c[k]
    x = np.zeros(n)
    x[jpvt[:rank]] = c[:rank]
    return x


def lstsq_basic(A, b):
    """qrcp + qrcp_solve: the basic least-squares solution of A x = b and the numerical rank."""
    QR, tau, jpvt, rank = qrcp(A)
    return qrcp_solve(QR, tau, jpvt, rank, b), rank
