"""CPU restatement of curvature's do_smooth solve (R/Src/curvature.cpp:328-406) for the tests: the composite AMR system

    phi - beta * div(grad phi) = c,   beta = smoothing_time,

solved to 1e-14 (max norm, relative to max|c|) with SciPy.  TEST INFRASTRUCTURE ONLY: the product never imports this.

The operator is written out here independently of the library's tables (DESIGN.md section 10):
  * 7-point operator on every valid cell; ghost cells from the C oracle's fill (filled_fabs_order below): same-level and
    periodic copies, the hierarchy's wall kinds, the coarse-fine polynomial of order MAXORDER through the o3-interpolated
    coarse value;
  * the coarse side of every coarse-fine face takes the average of the fine face fluxes (reflux), found from the fine boxes'
    face ghost cells that no fine box covers (periodic images included);
  * covered coarse cells hold the average of their 8 fine cells; they are not unknowns of the solve.
Refinement ratio 2 only.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse.linalg as spla

from .oracle import OracleHier

MAXORDER = 3          # AMReX's MLLinOp default maxorder; see DESIGN.md section 10, point 1


def poly_interp_coeff(x_int, x, n):
    """poly_interp_coeff (AMReX_LOUtil_K.H:24-37), the C oracle's loop order"""
    c = []
    for j in range(n):
        num, den = 1.0, 1.0
        for i in range(n):
            if i != j:
                num *= x_int - x[i]
                den *= x[j] - x[i]
        c.append(num / den)
    return c


def filled_fabs_order(O: OracleHier, lev: int, s: np.ndarray, maxorder: int):
    """OracleHier.filled_fabs (one ghost layer) with the coarse-fine polynomial of order `maxorder` instead of the tools' 4.

    The C oracle writes a coarse-fine ghost cell as g4 = sum_{m>=1} coef4[m] * phi_{m-1} + coef4[0] * bc (apply_bc, the
    Dirichlet polynomial of AMReX_MLLinOp_K.H through the o3-interpolated coarse value bc).  bc is recovered from g4 and the
    interior cells, and the ghost cell rewritten with the order-`maxorder` coefficients.  The cells are the ones apply_bc
    writes: faces that are not physical walls, mask value m_maskvals > 0 (OracleHier.mask kind 0).  The recovery moves the
    value by a few units in the last place, far below what the solve's tolerance resolves."""
    fabs = O.filled_fabs(lev, s, ng=1)
    if lev == 0 or maxorder == 4:
        return fabs
    lv = O.pf.levels[lev]
    r = O.ratios[lev - 1]
    for b, (lo, hi) in enumerate(lv.boxes):
        F = fabs[b]
        for face in range(6):
            d = face % 3
            islo = face < 3
            if not _periodic(O, d) and (lo[d] == lv.domain_lo[d] if islo else hi[d] == lv.domain_hi[d]):
                continue                                             # a physical wall: not coarse-fine
            pb, mv = O.mask(lev, b, face, 0)
            if not np.any(mv > 0):
                continue
            blen = hi[d] - lo[d] + 1
            x = [-0.5 * r, 0.5, 1.5, 2.5]                            # -bcl * dxinv with bcl = 0.5 * ratio * dx
            n4, nk = min(blen + 1, 4), min(blen + 1, maxorder)
            c4 = poly_interp_coeff(-0.5, x, n4)
            ck = poly_interp_coeff(-0.5, x, nk)
            s_in = 1 if islo else -1
            # index arrays of the face plane inside the grown fab ([z][y][x], ghost layer at index 0 / n+1)
            kk, jj, ii = np.nonzero(mv > 0)
            g = [ii + pb[0] - lo[0] + 1, jj + pb[1] - lo[1] + 1, kk + pb[2] - lo[2] + 1]

            def at(m):
                q = list(g)
                q[d] = q[d] + m * s_in
                return F[q[2], q[1], q[0]]
            tmp = np.zeros(len(ii))
            for m in range(1, n4):
                tmp = tmp + at(m) * c4[m]
            bc = (at(0) - tmp) / c4[0]
            v = np.zeros(len(ii))
            for m in range(1, nk):
                v = v + at(m) * ck[m]
            F[g[2], g[1], g[0]] = v + bc * ck[0]
    return fabs


def _periodic(O: OracleHier, d: int) -> bool:
    return bool(O._keep[5][d])


class SmoothOracle:
    def __init__(self, pf, is_per=(1, 1, 1), sym_dir=(0, 0, 0)):
        self.pf = pf
        self.O = OracleHier(pf, is_per, sym_dir)
        self.is_per = tuple(int(v) for v in is_per)
        L = pf.levels
        self.nlev = len(L)
        for l in range(1, self.nlev):
            n0 = L[l - 1].domain_hi[0] - L[l - 1].domain_lo[0] + 1
            n1 = L[l].domain_hi[0] - L[l].domain_lo[0] + 1
            if n1 != 2 * n0:
                raise ValueError("the smoothing oracle supports refinement ratio 2 only")
        self.total = int(self.O.total)
        self.dxi = [np.array([1.0 / v for v in lv.dx]) for lv in L]
        # flat layout: levels, boxes, [nz][ny][nx]; grown layout (one ghost layer) per level, boxes concatenated
        self.flat_off, self.grown_off = [], []
        self.cell_ijk = []            # per level: (ncells, 3) global i, j, k
        self.cell_grown = []          # per level: index of each valid cell in the grown concatenation
        self.strides = []             # per level: (ncells, 3) grown strides along x, y, z
        self.owner = []               # per level: dense [z][y][x] over the domain: flat index or -1
        o = 0
        for l, lv in enumerate(L):
            dlo, dhi = np.array(lv.domain_lo), np.array(lv.domain_hi)
            own = -np.ones(tuple((dhi - dlo + 1)[::-1]), dtype=np.int64)
            ijk, grown, strd, go = [], [], [], 0
            offs, goffs = [], []
            for lo, hi in lv.boxes:
                n = [hi[d] - lo[d] + 1 for d in range(3)]
                m = n[0] * n[1] * n[2]
                k, j, i = np.meshgrid(np.arange(n[2]), np.arange(n[1]), np.arange(n[0]), indexing="ij")
                i, j, k = i.ravel(), j.ravel(), k.ravel()
                ijk.append(np.stack([i + lo[0], j + lo[1], k + lo[2]], axis=1))
                P, PS = n[0] + 2, (n[0] + 2) * (n[1] + 2)
                grown.append(go + (k + 1) * PS + (j + 1) * P + (i + 1))
                strd.append(np.tile(np.array([1, P, PS]), (m, 1)))
                own[k + lo[2] - dlo[2], j + lo[1] - dlo[1], i + lo[0] - dlo[0]] = o + np.arange(m)
                offs.append(o)
                goffs.append(go)
                o += m
                go += PS * (n[2] + 2)
            self.flat_off.append(offs)
            self.grown_off.append(goffs)
            self.cell_ijk.append(np.concatenate(ijk))
            self.cell_grown.append(np.concatenate(grown))
            self.strides.append(np.concatenate(strd))
            self.owner.append(own)
        self.lev_range = []
        o = 0
        for l in range(self.nlev):
            n = len(self.cell_ijk[l])
            self.lev_range.append((o, o + n))
            o += n
        # covered coarse cells and their 8 fine cells
        self.cov, self.cov_fine = [], []
        uncovered = np.ones(self.total, dtype=bool)
        for l in range(self.nlev - 1):
            ijk = self.cell_ijk[l]
            fown = self.owner[l + 1]
            flo = np.array(L[l + 1].domain_lo)
            f0 = 2 * ijk - flo
            inside = np.all((f0 >= 0) & (f0 + 1 < np.array(fown.shape[::-1])), axis=1)
            q = np.nonzero(inside)[0]
            cov = q[fown[f0[q, 2], f0[q, 1], f0[q, 0]] >= 0]
            fine = np.stack([fown[f0[cov, 2] + kk, f0[cov, 1] + jj, f0[cov, 0] + ii]
                             for kk in (0, 1) for jj in (0, 1) for ii in (0, 1)], axis=1)
            if np.any(fine < 0):
                raise ValueError("fine boxes are not aligned to the refinement ratio")
            self.cov.append(cov + self.lev_range[l][0])
            self.cov_fine.append(fine)
            uncovered[cov + self.lev_range[l][0]] = False
        self.uncovered = np.nonzero(uncovered)[0]
        self._build_reflux()

    def _build_reflux(self):
        """one row per coarse-fine ghost cell of a fine box: (coarse flat cell, its grown index, its neighbour's grown
        index towards the fine region, dir, side, fine inside / ghost grown indices)"""
        L = self.pf.levels
        self.rf = []
        for lf in range(1, self.nlev):
            lc = lf - 1
            fdom_lo, fdom_hi = np.array(L[lf].domain_lo), np.array(L[lf].domain_hi)
            cdom_lo = np.array(L[lc].domain_lo)
            fown, cown = self.owner[lf], self.owner[lc]
            rows = []
            for b, (lo, hi) in enumerate(L[lf].boxes):
                n = [hi[d] - lo[d] + 1 for d in range(3)]
                P, PS = n[0] + 2, (n[0] + 2) * (n[1] + 2)
                go = self.grown_off[lf][b]
                for face in range(6):
                    d = face % 3
                    lo_face = face < 3
                    rng = [np.arange(lo[e], hi[e] + 1) for e in range(3)]
                    rng[d] = np.array([lo[d] - 1 if lo_face else hi[d] + 1])
                    k, j, i = np.meshgrid(rng[2], rng[1], rng[0], indexing="ij")
                    g = np.stack([i.ravel(), j.ravel(), k.ravel()], axis=1)
                    w = g.copy()
                    nd = fdom_hi[d] - fdom_lo[d] + 1
                    out_lo, out_hi = w[:, d] < fdom_lo[d], w[:, d] > fdom_hi[d]
                    if (out_lo.any() or out_hi.any()) and not self.is_per[d]:
                        continue                                     # a wall
                    w[out_lo, d] += nd
                    w[out_hi, d] -= nd
                    rel = w - fdom_lo
                    keep = fown[rel[:, 2], rel[:, 1], rel[:, 0]] < 0     # not covered by a fine box: coarse-fine
                    if not keep.any():
                        continue
                    g, w = g[keep], w[keep]
                    cc = w // 2
                    crel = cc - cdom_lo
                    qc = cown[crel[:, 2], crel[:, 1], crel[:, 0]]
                    if np.any(qc < 0):
                        raise ValueError("level %d is not properly nested" % lf)
                    side = 1 if lo_face else 0
                    inside = g.copy()
                    inside[:, d] += 1 if lo_face else -1
                    s = np.array([1, P, PS])
                    gi = go + (inside[:, 2] - lo[2] + 1) * PS + (inside[:, 1] - lo[1] + 1) * P + (inside[:, 0] - lo[0] + 1)
                    gg = gi - s[d] if lo_face else gi + s[d]
                    # coarse cell and its neighbour towards the fine region, in the coarse grown concatenation
                    qloc = qc - self.lev_range[lc][0]
                    cgi = self.cell_grown[lc][qloc]
                    cst = self.strides[lc][qloc, d]
                    cn = cgi + cst if side else cgi - cst
                    rows.append((qc, cgi, cn, np.full(len(qc), d), np.full(len(qc), side), gi, gg))
            if rows:
                self.rf.append(tuple(np.concatenate([r[m] for r in rows]) for m in range(7)))
            else:
                self.rf.append(None)

    # ---- the operator --------------------------------------------------------------------------------------------
    def average_down(self, phi: np.ndarray) -> None:
        for l in range(self.nlev - 2, -1, -1):
            phi[self.cov[l]] = 0.125 * phi[self.cov_fine[l]].sum(axis=1)

    def apply(self, phi: np.ndarray, beta: float) -> np.ndarray:
        """A phi on every valid cell (covered coarse cells of phi are overwritten with fine averages first)"""
        phi = np.array(phi, dtype=np.float64)
        self.average_down(phi)
        out = np.empty_like(phi)
        grown = []
        for l in range(self.nlev):
            G = np.concatenate([f.ravel() for f in filled_fabs_order(self.O, l, phi, MAXORDER)])
            grown.append(G)
            c, S = self.cell_grown[l], self.strides[l]
            v = G[c]
            lap = 0.0
            for d in range(3):
                h = self.dxi[l][d]
                lap = lap + ((G[c + S[:, d]] - v) * h - (v - G[c - S[:, d]]) * h) * h
            a, b = self.lev_range[l]
            out[a:b] = v - beta * lap
        for lf in range(1, self.nlev):
            R = self.rf[lf - 1]
            if R is None:
                continue
            qc, cgi, cn, d, side, gi, gg = R
            Gc, Gf = grown[lf - 1], grown[lf]
            hc, hf = self.dxi[lf - 1][d], self.dxi[lf][d]
            F = np.where(side == 1, (Gc[cn] - Gc[cgi]) * hc, (Gc[cgi] - Gc[cn]) * hc)
            g = np.where(side == 1, (Gf[gi] - Gf[gg]) * hf, (Gf[gg] - Gf[gi]) * hf)
            sgn = np.where(side == 1, -1.0, 1.0)
            np.add.at(out, qc, sgn * beta * 0.25 * (g - F) * hc)
        return out

    def residual(self, c: np.ndarray, phi: np.ndarray, beta: float) -> float:
        """max |c - A phi| over uncovered cells"""
        r = np.asarray(c) - self.apply(phi, beta)
        return float(np.max(np.abs(r[self.uncovered]))) if len(self.uncovered) else 0.0

    def solve(self, c: np.ndarray, beta: float, tol: float = 1e-14, rounds: int = 20) -> np.ndarray:
        """phi on every valid cell (covered cells = fine averages), max|c - A phi| <= tol * max|c| over uncovered cells"""
        c = np.asarray(c, dtype=np.float64)
        if beta == 0.0:
            return c.copy()
        u = self.uncovered
        N = len(u)
        diag = np.empty(self.total)
        for l in range(self.nlev):
            a, b = self.lev_range[l]
            diag[a:b] = 1.0 + 2.0 * beta * float(np.sum(self.dxi[l] ** 2))
        dinv = 1.0 / diag[u]

        def mv(y):
            phi = np.zeros(self.total)
            phi[u] = y
            return self.apply(phi, beta)[u]
        A = spla.LinearOperator((N, N), matvec=mv, dtype=np.float64)
        M = spla.LinearOperator((N, N), matvec=lambda y: dinv * y, dtype=np.float64)
        x = c[u].copy()
        cmax = float(np.max(np.abs(c[u]))) if N else 0.0
        for _ in range(rounds):
            r = c[u] - mv(x)
            if np.max(np.abs(r)) <= tol * cmax:
                break
            dx, info = spla.gmres(A, r, M=M, rtol=1e-12, atol=0.0, restart=60, maxiter=200)
            x = x + dx
        else:
            raise RuntimeError("smoothing oracle: no convergence to %g" % tol)
        phi = np.zeros(self.total)
        phi[u] = x
        self.average_down(phi)
        return phi
