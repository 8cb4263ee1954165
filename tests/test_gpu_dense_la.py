"""Dense linear algebra on the device against exact and high-precision references: `b200_getrf` / `b200_getrs` (every code
path of the blocked LU: both outer-block widths, the full-width cooperative panel, several tile groups in the trailing GEMM,
ld > n, ties in the pivot search, zero and non-finite pivots), `b200_gemv` (its three paths) and the pivoted-QR rescue of a
singular Newton step.

Exact-factor matrices.  A = Pi (I + L0) U0 with L0 strictly lower, entries in {0, +-1/4, +-1/2}; U0 upper with integer
entries in [-8, 8] above a diagonal of +-2^e, e in 0..3; Pi a random row permutation.  Every product and partial sum is a
multiple of 1/4 below 2^17 in magnitude, so A, every Schur complement and every multiplier a * (1 / pivot) are exact whatever
the summation order, and partial pivoting has a unique maximum at every step (|l| = 1 on the intended row, <= 1/2 elsewhere).
getrf must therefore return exactly L0 \\ U0, and the pivot sequence is a replay of the interchanges on Pi (O(n) on the host):
bit-exact at any size without an O(n^3) reference.

The GPU tests allocate through torch and pass data_ptr() to the ABI; torch and the library run on different streams, so both
sides are synchronised explicitly around every library call."""
import ctypes as C
import math

import numpy as np
import pytest

SENTINEL = -12345.5  # written into the padding rows [n, ld) of every column-major buffer; must survive every call
EPS = np.finfo(np.float64).eps
SM_COUNT_B200 = 148


# ============================================================================ generators (CPU and device)
def exact_lu_instance(n, seed, device="cpu", zero_cols=(), tie_cols=None):
    """(E, M, perm): E = L0 \\ U0 (strict lower part L0, upper part U0) as an n x n torch tensor, M = (I + L0) U0 and the row
    permutation perm (numpy int64, row i of M sits at row perm[i] of A).

    zero_cols: columns k with u_kk = 0 and L0[k+1:, k] = 0 (perm fixes position k, so no earlier step moves that row).
    tie_cols: {k: i} (i > k) leaves L0[:, k] zero but for an entry +-1 at row i, and zeroes L0[i, k+1:i]: rows k and i tie
    at step k, and whichever of them comes first the elimination stays exact and the later pivots stay +- powers of two
    (the other row's remainder is then +- row i's, whose only entry past column k is its unit diagonal)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    L = torch.randint(-2, 3, (n, n), generator=g, device=device).double().mul_(0.25).tril_(-1)
    U = torch.randint(-8, 9, (n, n), generator=g, device=device).double().triu_(1)
    e = torch.randint(0, 4, (n,), generator=g, device=device).double()
    s = torch.randint(0, 2, (n,), generator=g, device=device).double().mul_(-2.0).add_(1.0)
    U.diagonal().copy_(torch.pow(2.0, e) * s)
    rng = np.random.default_rng(seed)
    for k, i in (tie_cols or {}).items():
        L[:, k] = 0.0
        L[i, k] = rng.choice([-1.0, 1.0])
        L[i, k + 1:i] = 0.0
    for k in zero_cols:
        U[k, k] = 0.0
        L[k + 1:, k] = 0.0
    perm = rng.permutation(n)
    for k in zero_cols:
        j = int(np.nonzero(perm == k)[0][0])
        perm[j], perm[k] = perm[k], perm[j]
    M = torch.addmm(U, L, U)  # (I + L0) U0: exact
    E = L.add_(U)
    del U
    return E, M, perm


def replay_ipiv(perm):
    """LAPACK ipiv (1-based) of partial pivoting on A = Pi M when the pivot of step k is always M's row k."""
    n = len(perm)
    pos = np.asarray(perm, dtype=np.int64).copy()     # pos[i]: current row of M's row i
    at = np.empty(n, dtype=np.int64)
    at[pos] = np.arange(n)                            # at[r]: which row of M is at row r
    ipiv = np.empty(n, dtype=np.int64)
    for k in range(n):
        p = pos[k]
        ipiv[k] = p + 1
        rk = at[k]
        at[k], at[p] = k, rk
        pos[k], pos[rk] = k, p
    return ipiv


def assemble(M, perm):
    """A = Pi M (numpy, for the CPU oracle)."""
    A = np.empty_like(M)
    A[perm] = M
    return A


def dyadic_exact(A, LU, ipiv, info, q=4):
    """True when the factorisation (LU, ipiv) of A is exact in floating point whatever the order of its sums: no zero pivot,
    every pivot +- a power of two, every factor entry a multiple of 2^-q, and every partial sum of A_ij - sum_k L_ik U_kj
    below 2^(52 - 2q) in magnitude.  Then the computed factors are the exact ones, and any implementation that picks the
    same pivots must return them bit for bit."""
    if info != 0:
        return False
    n = A.shape[0]
    d = np.abs(np.diag(LU))
    if not np.all(np.frexp(d)[0] == 0.5):
        return False
    sc = LU * 2.0 ** q
    if not np.array_equal(sc, np.round(sc)):
        return False
    L = np.tril(LU, -1) + np.eye(n)
    U = np.triu(LU)
    if (np.abs(A).max() + (np.abs(L) @ np.abs(U)).max()) >= 2.0 ** (52 - 2 * q):
        return False
    PA = A.copy()
    for k in range(n):
        p = ipiv[k] - 1
        if p != k:
            PA[[k, p]] = PA[[p, k]]
    return np.array_equal(L @ U, PA)


def panel_cta(n, k, row, sm_count=SM_COUNT_B200):
    """Which CTA of the cooperative panel that factors column k owns `row` (dense.cu: factor_panel's P / rpc)."""
    c0 = (k // 32) * 32
    m = n - c0
    P = min(sm_count, 160, max(1, (m + 127) // 128))
    rpc = (m + P - 1) // P
    return (row - c0) // rpc


def cross_cta_ties(LU, ipiv):
    """Number of pivot steps at which rows owned by different panel CTAs tie at the column maximum.  Replays the row positions
    at the time of each pivot search from the final factors (the entries of L travel with their rows)."""
    n = LU.shape[0]
    at = np.arange(n)                 # at[r]: final row of the row sitting at r
    pos = np.arange(n)
    count = 0
    for k in range(n - 1, -1, -1):    # undo the interchanges k .. n-1: the arrangement at the search of step k
        p = ipiv[k] - 1
        if p != k:
            at[k], at[p] = at[p], at[k]
            pos[at[k]], pos[at[p]] = k, p
        tied = np.nonzero(np.abs(LU[k + 1:, k]) == 1.0)[0] + k + 1
        if len(tied) and len({panel_cta(n, k, pos[r]) for r in [k, *tied]}) > 1:
            count += 1
    return count


def tie_instance(n, seed, po, npairs=48):
    """An exact-factor matrix with `npairs` tied row pairs (exact_lu_instance's tie_cols) on disjoint rows, and the CPU
    oracle's factorisation of it.  Draws again until the oracle's factorisation is exact (dyadic_exact)."""
    for attempt in range(8):
        rng = np.random.default_rng(seed + attempt)
        idx = rng.choice(n, 2 * npairs, replace=False).reshape(npairs, 2)
        ties = {int(min(a, b)): int(max(a, b)) for a, b in idx}
        E, M, perm = exact_lu_instance(n, seed + attempt, tie_cols=ties)
        A = assemble(M.numpy(), perm)
        LU, ipiv, info = po.getrf(A)
        if dyadic_exact(A, LU, ipiv, info):
            return A, LU, ipiv
    raise AssertionError("no exact tie instance drawn")


# ============================================================================ CPU checks of the generators and restatements
def test_exact_instance_reproduced_by_oracle(po):
    for n, zero_cols, info_expected in ((300, (), 0), (1024, (300, 700), 301)):
        E, M, perm = exact_lu_instance(n, 11, zero_cols=zero_cols)
        A = assemble(M.numpy(), perm)
        LU, ipiv, info = po.getrf(A)
        assert info == info_expected
        assert np.array_equal(LU, E.numpy())
        assert np.array_equal(ipiv, replay_ipiv(perm))
        for k in zero_cols:
            assert ipiv[k] == k + 1


def test_tie_generator_acceptance(po):
    A, LU, ipiv = tie_instance(1024, 3, po)
    assert cross_cta_ties(LU, ipiv) >= 4
    # a pivot of 3 makes the multipliers non-dyadic: rejected
    E, M, perm = exact_lu_instance(64, 5)
    M = M.numpy().copy()
    M[:, 10] *= 3.0 / 2.0 ** np.round(np.log2(abs(E[10, 10].item())))
    B = assemble(M, perm)
    LU2, ipiv2, info2 = po.getrf(B)
    assert not dyadic_exact(B, LU2, ipiv2, info2)
    A0 = assemble(exact_lu_instance(64, 5)[1].numpy(), perm)
    assert dyadic_exact(A0, *po.getrf(A0))


def test_qrcp_restatement_vs_scipy():
    import scipy.linalg as sl
    from oracle import qrcp_numpy as qn
    rng = np.random.default_rng(0)
    for n in (1, 2, 33, 300):
        A = rng.standard_normal((n, n))
        b = rng.standard_normal(n)
        QR, tau, jpvt, rank = qn.qrcp(A)
        Q, R, P = sl.qr(A, pivoting=True)
        assert rank == n and np.array_equal(jpvt, P)
        assert np.abs(np.triu(QR) - R).max() <= 1e-13 * np.abs(R).max()
        x = qn.qrcp_solve(QR, tau, jpvt, rank, b)
        assert np.abs(A @ x - b).max() <= 1e-12 * (np.abs(A).max() * np.abs(x).max() * n)
    # rank-deficient: the basic solution is zero off the first `rank` pivot columns and solves the normal equations there
    A = rng.standard_normal((50, 50))
    A[:, 7] = A[:, 3]
    A[:, 9] = 0.0
    x, rank = qn.lstsq_basic(A, rng.standard_normal(50))
    assert rank == 48 and x[9] == 0.0 and (x[3] == 0.0) != (x[7] == 0.0)


# ============================================================================ device helpers
def _torch():
    import torch
    return torch


def padded(n, ld, ncols=None):
    """A column-major n x ncols device buffer with leading dimension ld, as a torch (ncols, ld) tensor; rows [n, ld) hold
    SENTINEL.  buf[:, :n].T is the matrix."""
    torch = _torch()
    buf = torch.empty((ncols or n, ld), dtype=torch.float64, device="cuda")
    buf[:, n:] = SENTINEL
    return buf


def getrf(nls, ctx, buf, n, ld):
    torch = _torch()
    ipiv = torch.empty(n, dtype=torch.int64, device="cuda")
    info = C.c_int32(-7)
    torch.cuda.synchronize()
    nls.abi.check(ctx.handle, nls.abi.lib().b200_getrf(ctx.handle, n, buf.data_ptr(), ld, ipiv.data_ptr(), C.byref(info)))
    ctx.sync()
    return ipiv, info.value


def getrs(nls, ctx, buf, n, ld, ipiv, bbuf, nrhs, ldb):
    torch = _torch()
    torch.cuda.synchronize()
    nls.abi.check(ctx.handle, nls.abi.lib().b200_getrs(ctx.handle, n, nrhs, buf.data_ptr(), ld, ipiv.data_ptr(), bbuf.data_ptr(), ldb))
    ctx.sync()


def exact_on_device(n, ld, seed, zero_cols=()):
    """(buf holding A = Pi M with padding, E, perm) on the device."""
    E, M, perm = exact_lu_instance(n, seed, device="cuda", zero_cols=zero_cols)
    buf = padded(n, ld)
    buf[:, :n].t()[_torch().as_tensor(perm, device="cuda")] = M
    del M
    return buf, E, perm


def pad_intact(buf, n):
    return bool((buf[:, n:] == SENTINEL).all())


# ============================================================================ §1 + §4: exact factors, getrs
@pytest.mark.gpu
@pytest.mark.parametrize("n,ld", [(1, 1), (2, 2), (31, 31), (33, 33), (255, 255), (256, 256), (257, 257), (511, 511), (513, 513),
                                  (2049, 2049), (4097, 4098), (16384, 16391), (20003, 20011)])
def test_getrf_exact_factors(nls, ctx, n, ld):
    """Bit-exact L0 \\ U0 and the replayed pivots.  2049: two tile groups in the first trailing update; 16384: the first
    NBO = 512 size; 20003: 512-wide outer blocks, the full-width panel (148 CTAs), ragged last inner / outer / tile blocks."""
    torch = _torch()
    buf, E, perm = exact_on_device(n, ld, seed=n)
    nrhs, ldb = 3, n + 3
    x0 = torch.randint(-4, 5, (nrhs, n), device="cuda").double()
    bbuf = padded(n, ldb, nrhs)
    bbuf[:, :n] = x0 @ buf[:, :n]            # (A x0)' : exact
    ipiv, info = getrf(nls, ctx, buf, n, ld)
    assert info == 0
    assert np.array_equal(ipiv.cpu().numpy(), replay_ipiv(perm))
    assert torch.equal(buf[:, :n], E.t())
    assert pad_intact(buf, n)
    getrs(nls, ctx, buf, n, ld, ipiv, bbuf, nrhs, ldb)
    assert torch.equal(bbuf[:, :n], x0)
    assert pad_intact(bbuf, n) and pad_intact(buf, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n,nrhs", [(513, 1), (513, 257), (513, 513), (1000, 3)])
def test_getrs_exact_many_rhs(nls, ctx, n, nrhs):
    """getrs on exact factors returns x0 bit for bit: nrhs past the 256 threads of apply_pivots_kernel's first block and
    nrhs = n (Broyden's true_jacobian inverts J that way), ldb = n + 3."""
    torch = _torch()
    buf, E, perm = exact_on_device(n, n, seed=7 * n + nrhs)
    ldb = n + 3
    x0 = torch.randint(-4, 5, (nrhs, n), device="cuda").double()
    bbuf = padded(n, ldb, nrhs)
    bbuf[:, :n] = x0 @ buf[:, :n]
    ipiv, info = getrf(nls, ctx, buf, n, n)
    assert info == 0 and torch.equal(buf[:, :n], E.t())
    getrs(nls, ctx, buf, n, n, ipiv, bbuf, nrhs, ldb)
    assert torch.equal(bbuf[:, :n], x0)
    assert pad_intact(bbuf, n)


# ============================================================================ §2: ties across panel CTAs
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1024, 2048])
def test_getrf_ties_across_panel_ctas(nls, ctx, po, n):
    """Rows tie at the column maximum in different CTAs of the cooperative panel (8 / 16 CTAs): the first row wins, as in
    LAPACK.  The oracle's factorisation is exact (checked by the generator), so the kernel must match it bit for bit."""
    torch = _torch()
    A, LU, ipiv_o = tie_instance(n, 100 + n, po)
    nties = cross_cta_ties(LU, ipiv_o)
    assert nties >= 4, nties
    ld = n + 1
    buf = padded(n, ld)
    buf[:, :n] = torch.as_tensor(A.T, device="cuda")
    ipiv, info = getrf(nls, ctx, buf, n, ld)
    assert info == 0
    assert np.array_equal(ipiv.cpu().numpy(), ipiv_o)
    assert np.array_equal(buf[:, :n].cpu().numpy().T, LU)
    assert pad_intact(buf, n)


# ============================================================================ §3: zero and non-finite pivots
@pytest.mark.gpu
def test_getrf_zero_pivots(nls, ctx, po):
    """u_kk = 0 at k = 300 (inside the look-ahead panel of the second outer block, factored on the second stream) and 700:
    info = 301, the row at position k stays (ipiv[k] = k + 1), LAPACK carries on past the zero pivot, and the factors are
    still L0 \\ U0 bit for bit; the CPU oracle gives the same bits."""
    torch = _torch()
    n = 1024
    buf, E, perm = exact_on_device(n, n, seed=21, zero_cols=(300, 700))
    A = buf[:, :n].cpu().numpy().T.copy()
    ipiv, info = getrf(nls, ctx, buf, n, n)
    assert info == 301
    ip = ipiv.cpu().numpy()
    assert ip[300] == 301 and ip[700] == 701
    assert np.array_equal(ip, replay_ipiv(perm))
    assert torch.equal(buf[:, :n], E.t())
    LUo, ipo, infoo = po.getrf(A)
    assert infoo == 301 and np.array_equal(ipo, ip) and np.array_equal(LUo, E.cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["nan_col0", "inf_interior"])
def test_getrf_non_finite_entries(nls, ctx, case):
    """A NaN is not a zero pivot (LAPACK): getrf returns OK with info = 0, and the non-finite value reaches the factors and
    the solution.  NaN in column 0 at row 500 (panel CTA 3 of 8); Inf above the diagonal at (200, 600) of an exact-factor
    matrix, so U[200, 600] is infinite and the update below it turns column 600 into Inf / NaN."""
    torch = _torch()
    n = 1024
    if case == "nan_col0":
        g = torch.Generator(device="cuda").manual_seed(5)
        buf = padded(n, n)
        buf[:, :n] = torch.randn((n, n), generator=g, device="cuda", dtype=torch.float64)
        buf[0, 500] = float("nan")
        assert panel_cta(n, 0, 500) == 3
    else:
        buf, E, perm = exact_on_device(n, n, seed=9)
        buf[600, perm[200]] = float("inf")
    ipiv, info = getrf(nls, ctx, buf, n, n)
    assert info == 0
    ip = ipiv.cpu().numpy()
    assert ip.min() >= 1 and ip.max() <= n and np.all(ip >= np.arange(1, n + 1))
    assert not bool(torch.isfinite(buf).all())
    b = torch.ones((1, n), dtype=torch.float64, device="cuda")
    getrs(nls, ctx, buf, n, n, ipiv, b, 1, n)
    assert not bool(torch.isfinite(b).all())


# ============================================================================ §5: parity with LAPACK / cuSOLVER on random data
@pytest.mark.gpu
@pytest.mark.parametrize("n,ld", [(2049, 2051), (4097, 4099)])
def test_getrf_lapack_parity_random(nls, ctx, n, ld):
    import scipy.linalg as sl
    torch = _torch()
    rng = np.random.default_rng(n)
    A = rng.standard_normal((n, n))
    b = rng.standard_normal(n)
    buf = padded(n, ld)
    buf[:, :n] = torch.as_tensor(A.T, device="cuda")
    ipiv, info = getrf(nls, ctx, buf, n, ld)
    assert info == 0
    LUs, pivs = sl.lu_factor(A)
    assert np.array_equal(ipiv.cpu().numpy(), pivs + 1)  # LAPACK's pivot sequence, bit-exact
    LU = buf[:, :n].cpu().numpy().T
    dev = np.abs(LU - LUs).max() / np.abs(LUs).max()
    assert dev <= 1e-9, dev
    bb = padded(n, n + 1, 1)
    bb[0, :n] = torch.as_tensor(b, device="cuda")
    getrs(nls, ctx, buf, n, ld, ipiv, bb, 1, n + 1)
    x = bb[0, :n].cpu().numpy()
    berr = np.abs(A @ x - b).max() / (np.abs(A).sum(axis=1).max() * np.abs(x).max() + np.abs(b).max())
    assert berr <= n * EPS, berr  # normwise backward error; LU with partial pivoting on Gaussian data sits far below this
    assert pad_intact(buf, n) and pad_intact(bb, n)


@pytest.mark.gpu
def test_getrf_cusolver_parity_n20003(nls, ctx):
    """n = 20003, ld = 20011 on Gaussian data: the pivots equal cuSOLVER's (torch.linalg.lu_factor on the same matrix), and
    the backward error ||PA - LU||_max / ||A||_max is no worse than 4x cuSOLVER's own.  Everything stays on the device."""
    torch = _torch()
    n, ld = 20003, 20011
    g = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn((n, n), generator=g, device="cuda", dtype=torch.float64)
    buf = padded(n, ld)
    buf[:, :n] = A.t()
    ipiv, info = getrf(nls, ctx, buf, n, ld)
    assert info == 0 and pad_intact(buf, n)
    LUc, pivc = torch.linalg.lu_factor(A)
    assert torch.equal(ipiv, pivc.to(torch.int64))
    perm = np.arange(n)
    for k, p in enumerate(ipiv.cpu().numpy() - 1):
        perm[k], perm[p] = perm[p], perm[k]
    PA = A[torch.as_tensor(perm, device="cuda")]
    del A
    anorm = PA.abs().max().item()

    def backward_error(LU):
        L = LU.tril(-1)
        L.diagonal().fill_(1.0)
        R = torch.matmul(L, LU.triu())
        del L
        return (R.sub_(PA)).abs().max().item() / anorm

    e_dev = backward_error(buf[:, :n].t())
    e_cus = backward_error(LUc)
    assert e_dev <= 4.0 * e_cus, (e_dev, e_cus)


# ============================================================================ §6: b200_gemv
def _gemv(nls, ctx, trans, m, n, Abuf, ld, x, y):
    torch = _torch()
    torch.cuda.synchronize()
    nls.abi.check(ctx.handle, nls.abi.lib().b200_gemv(ctx.handle, trans, m, n, Abuf.data_ptr(), ld, x.data_ptr(), y.data_ptr()))
    ctx.sync()


GEMV_SHAPES = ([(0, m, n) for m in (1, 257, 100003) for n in (1, 5, 300)]
               + [(1, m, n) for n in (4097, 9000) for m in (3, 1000, 70001)]                      # CTA per column, grid-stride
               + [(1, m, n) for m in (32768, 2100001) for n in (1, 16, 17, 33, 64)]               # tall and skinny
               + [(1, 32768, 65), (1, 40000, 65), (1, 32767, 64), (1, 32767, 17)])                # just outside the tall path


@pytest.mark.gpu
@pytest.mark.parametrize("trans,m,n", GEMV_SHAPES)
def test_gemv_paths(nls, ctx, trans, m, n):
    """Integer-valued A and x: every summation order is exact, so y must equal the exact product bit for bit; then a
    Gaussian A against |y - y_ref| <= 2 K eps (|A| |x|), K the length of the sums.  ld = m + 1 (odd for even m) with
    NaN padding: a read past row m poisons the result."""
    torch = _torch()
    ld = m + 1 if m % 2 == 0 else m + 2
    g = torch.Generator(device="cuda").manual_seed(m * 7 + n)
    buf = torch.empty((n, ld), dtype=torch.float64, device="cuda")
    buf[:, m:] = float("nan")
    A = buf[:, :m].t()                                   # m x n view
    kx, ky = (m, n) if trans else (n, m)
    for kind in ("int", "gauss"):
        if kind == "int":
            buf[:, :m] = torch.randint(-8, 9, (n, m), generator=g, device="cuda").double()
            x = torch.randint(-8, 9, (kx,), generator=g, device="cuda").double()
        else:
            buf[:, :m] = torch.randn((n, m), generator=g, device="cuda", dtype=torch.float64)
            x = torch.randn((kx,), generator=g, device="cuda", dtype=torch.float64)
        y = torch.full((ky,), float("nan"), dtype=torch.float64, device="cuda")
        _gemv(nls, ctx, trans, m, n, buf, ld, x, y)
        Aop = A.t() if trans else A
        ref = Aop @ x
        if kind == "int":
            assert torch.equal(y, ref), (kind, (y - ref).abs().max().item())
        else:
            bound = 2.0 * kx * EPS * (Aop.abs() @ x.abs())
            assert bool(((y - ref).abs() <= bound).all()), kind


# ============================================================================ §7: the pivoted-QR rescue through the driver
def rescue_problem(n, seed):
    """Integer A with a dominant diagonal (well conditioned) made singular on purpose: one zero column, duplicated columns
    (exact ties in the column-norm search, resolved by the index alone) and columns that are exact combinations of two others.  Returns A, b and the groups of
    dependent columns (in each group at least one column must be left out of the basic solution)."""
    rng = np.random.default_rng(seed)
    A = rng.integers(-3, 4, (n, n)).astype(np.float64)
    A[np.arange(n), np.arange(n)] += 8 * math.ceil(math.sqrt(n)) * rng.choice([-1.0, 1.0], n)
    cols = rng.permutation(n)
    z = int(cols[0])
    A[:, z] = 0.0
    groups = []
    for i in range(4):  # duplicates
        a, d = int(cols[1 + 2 * i]), int(cols[2 + 2 * i])
        A[:, d] = A[:, a]
        groups.append((a, d))
    for i in range(3):  # exact combinations; 2 a + 3 c2 rather than a + c2, whose remainders after eliminating a would be
        a, c2, c = (int(v) for v in cols[9 + 3 * i: 12 + 3 * i])   # equal in exact arithmetic: a tie left to rounding
        A[:, c] = 2.0 * A[:, a] + 3.0 * A[:, c2]
        groups.append((a, c2, c))
    b = rng.standard_normal(n)
    return A, b, z, groups


def rescue_solve(nls, ctx, A, b):
    torch = _torch()
    n = len(b)
    Ad = torch.as_tensor(A, device="cuda")
    bd = torch.as_tensor(b, device="cuda")

    def F(du, u, _p):
        torch.as_tensor(du, device="cuda").copy_(Ad @ torch.as_tensor(u, device="cuda") - bd)
        torch.cuda.synchronize()

    def JAC(J, u, _p):
        torch.as_tensor(J, device="cuda").view(n, n).copy_(Ad.t())   # column-major: J_t[c, r] = A[r, c]
        torch.cuda.synchronize()

    prob = nls.NonlinearProblem(nls.NonlinearFunction(F, n=n, jac=JAC), np.zeros(n), None, ctx=ctx)
    return nls.solve(prob, nls.NewtonRaphson(), abstol=1e-12, maxiters=1, termination_condition=nls.AbsNormTerminationMode())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [300, 1500, 4096, 4097])
def test_singular_lu_rescued_by_pivoted_qr(nls, ctx, n):
    """One Newton step from u0 = 0 on f(u) = A u - b with a singular A: getrf reports the zero column, the driver refills J and
    takes the basic least-squares solution from the column-pivoted QR (one CTA of 1024 threads; 1500 has more rows than
    threads; 4096 is the largest size the rescue takes, 4097 must end in InternalLinearSolveFailed).  The iterate matches the
    NumPy restatement (oracle/qrcp_numpy.py) to 1e-10 where that is affordable (n <= 1500) and, at every size and
    independently of it, is zero off a basic set of columns and solves the normal equations on that set."""
    A, b, z, groups = rescue_problem(n, seed=n)
    sol = rescue_solve(nls, ctx, A, b)
    if n > 4096:
        assert sol.retcode == nls.ReturnCode.InternalLinearSolveFailed
        return
    assert sol.retcode == nls.ReturnCode.MaxIters and sol.stats.nsteps == 1
    u = sol.u.to_host() if hasattr(sol.u, "to_host") else np.asarray(sol.u)
    rank = n - 1 - len(groups)
    basic = np.nonzero(u)[0]
    assert u[z] == 0.0 and len(basic) == rank
    for grp in groups:
        assert any(u[c] == 0.0 for c in grp), grp
    r = A @ u - b
    AB = A[:, basic]
    assert np.abs(AB.T @ r).max() <= 1e-10 * np.linalg.norm(AB) * np.linalg.norm(r)
    if n <= 1500:
        from oracle import qrcp_numpy as qn
        x, rank_ref = qn.lstsq_basic(A, -b)   # the step solves J x = f(u0) = -b and takes u1 = u0 - x
        assert rank_ref == rank
        uref = -x
        assert np.abs(u - uref).max() <= 1e-10 * np.abs(uref).max()
