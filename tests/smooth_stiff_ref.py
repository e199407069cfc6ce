"""Reference solution of the smoothing system at large smoothing_time / dx^2, where oracle/smooth_oracle.py's Jacobi-preconditioned
GMRES does not reach its 1e-14 tolerance.  The operator is still the oracle's independent restatement (SmoothOracle.apply); only
the preconditioner differs: a sparse LU factorisation of I - beta * Lap on the uncovered cells, with each level's own 7-point
neighbours (periodic images included; neighbours outside the level, across walls or covered, dropped).  It carries the stiff part
of the operator, so the outer loop needs few GMRES iterations.  TEST INFRASTRUCTURE ONLY."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla


def _level_laplacian_coupling(so):
    """rows, cols, weights dxi^2 of every (uncovered cell, uncovered same-level neighbour) pair, in uncovered numbering"""
    unc = np.full(so.total, -1, dtype=np.int64)
    unc[so.uncovered] = np.arange(len(so.uncovered))
    rows, cols, w = [], [], []
    for l in range(so.nlev):
        lv = so.pf.levels[l]
        dlo, dhi = np.array(lv.domain_lo), np.array(lv.domain_hi)
        n = dhi - dlo + 1
        a, b = so.lev_range[l]
        ijk = so.cell_ijk[l]
        me = unc[a:b]
        for d in range(3):
            for s in (-1, 1):
                q = ijk.copy()
                q[:, d] += s
                rel = q - dlo
                if so.is_per[d]:
                    rel[:, d] %= n[d]
                ok = (rel[:, d] >= 0) & (rel[:, d] < n[d]) & (me >= 0)
                idx = np.nonzero(ok)[0]
                nb = so.owner[l][rel[idx, 2], rel[idx, 1], rel[idx, 0]]
                keep = nb >= 0
                idx, nb = idx[keep], nb[keep]
                nu = unc[nb]
                keep = nu >= 0
                rows.append(me[idx[keep]])
                cols.append(nu[keep])
                w.append(np.full(int(keep.sum()), so.dxi[l][d] ** 2))
    return np.concatenate(rows), np.concatenate(cols), np.concatenate(w)


def stiff_solve(so, c, beta, rounds=30):
    """phi on every valid cell (covered cells = fine averages) with max|c - A phi| <= tol * max|c| over uncovered cells,
    tol = max(1e-14, 1e-15 * (1 + 2 beta sum dxi_finest^2)): the rounding of A phi grows with the operator's diagonal, so a
    fixed 1e-14 is out of reach at large beta.  A = I - beta * Lap with Lap close to a negative semidefinite operator, so the
    error of phi is of the order of that residual, far below the 1e-9 the tests compare at."""
    c = np.asarray(c, dtype=np.float64)
    tol = max(1e-14, 1e-15 * (1.0 + 2.0 * beta * float(np.sum(so.dxi[-1] ** 2))))
    u = so.uncovered
    N = len(u)
    r_, c_, w_ = _level_laplacian_coupling(so)
    off = sp.csr_matrix((-beta * w_, (r_, c_)), shape=(N, N))
    diag = 1.0 - np.asarray(off.sum(axis=1)).ravel()
    M = (off + sp.diags(diag)).tocsc()
    lu = spla.splu(M)

    def mv(y):
        phi = np.zeros(so.total)
        phi[u] = y
        return so.apply(phi, beta)[u]
    A = spla.LinearOperator((N, N), matvec=mv, dtype=np.float64)
    P = spla.LinearOperator((N, N), matvec=lu.solve, dtype=np.float64)
    x = c[u].copy()
    cmax = float(np.max(np.abs(c[u])))
    for _ in range(rounds):
        r = c[u] - mv(x)
        if np.max(np.abs(r)) <= tol * cmax:
            break
        dx, info = spla.gmres(A, r, M=P, rtol=1e-13, atol=0.0, restart=100, maxiter=5)
        x = x + dx
    else:
        raise RuntimeError("stiff reference solve: no convergence to %g" % tol)
    phi = np.zeros(so.total)
    phi[u] = x
    so.average_down(phi)
    return phi
