"""CPU tier: the do_smooth oracle (oracle/smooth_oracle.py) -- the composite system phi - t * div(grad phi) = c of
R/Src/curvature.cpp:328-406 -- against closed forms on one level (FFT on a periodic domain, DCT-II with Neumann walls), and
the properties of its composite solution: conservation on periodic / Neumann domains, covered cells = fine averages,
t = 0 gives c."""
import numpy as np
import pytest
import scipy.fft as sfft

from helpers import load_golden
from oracle.smooth_oracle import SmoothOracle
from peleanalysis_b200.plotfile import Plotfile


def _one_level(name):
    pf, z = load_golden(name)
    return Plotfile(pf.names, pf.prob_lo, pf.prob_hi, [], pf.levels[:1])


def _dense(pf, flat):
    lv = pf.levels[0]
    n = [lv.domain_hi[d] - lv.domain_lo[d] + 1 for d in range(3)]
    out = np.empty(n[::-1])
    o = 0
    for lo, hi in lv.boxes:
        m = [hi[d] - lo[d] + 1 for d in range(3)]
        k = m[0] * m[1] * m[2]
        out[lo[2]:hi[2] + 1, lo[1]:hi[1] + 1, lo[0]:hi[0] + 1] = flat[o:o + k].reshape(m[2], m[1], m[0])
        o += k
    return out


def _eig(n, dx, t, per):
    """eigenvalues of I - t * Laplacian_h, axes (z, y, x)"""
    lam = 1.0
    for ax, d in enumerate((2, 1, 0)):
        k = np.arange(n[ax])
        th = 2 * np.pi * k / n[ax] if per else np.pi * k / n[ax]
        shape = [1, 1, 1]
        shape[ax] = n[ax]
        lam = lam + t * ((2 - 2 * np.cos(th)) / dx[d] ** 2).reshape(shape)
    return lam


@pytest.mark.parametrize("t", [1e-5, 1e-3])
def test_oracle_periodic_matches_fft(t):
    pf = _one_level("c1_periodic")
    rng = np.random.default_rng(1)
    so = SmoothOracle(pf, (1, 1, 1))
    c = rng.random(so.total)
    phi = so.solve(c, t)
    C = _dense(pf, c)
    ref = np.real(sfft.ifftn(sfft.fftn(C) / _eig(C.shape, pf.levels[0].dx, t, True)))
    assert np.max(np.abs(_dense(pf, phi) - ref)) <= 1e-12 * np.max(np.abs(C))


@pytest.mark.parametrize("t", [1e-5, 1e-3])
def test_oracle_neumann_matches_dct(t):
    pf = _one_level("c1_walls")
    rng = np.random.default_rng(2)
    so = SmoothOracle(pf, (0, 0, 0))
    c = rng.random(so.total)
    phi = so.solve(c, t)
    C = _dense(pf, c)
    ref = sfft.idctn(sfft.dctn(C, type=2, norm="ortho") / _eig(C.shape, pf.levels[0].dx, t, False), type=2, norm="ortho")
    assert np.max(np.abs(_dense(pf, phi) - ref)) <= 1e-12 * np.max(np.abs(C))


def _vol(so, pf):
    return np.concatenate([np.full(b - a, np.prod(pf.levels[l].dx)) for l, (a, b) in enumerate(so.lev_range)])


@pytest.mark.parametrize("name,per", [("c1_periodic", (1, 1, 1)), ("c1_walls", (0, 0, 0)), ("c3_three_levels", (1, 1, 1)),
                                      ("mixed_boxes", (1, 1, 1))])
def test_oracle_composite_conserves(name, per):
    """no flux leaves a periodic or Neumann domain and the coarse side of every coarse-fine face takes the fine fluxes:
    sum(vol * phi) = sum(vol * c) over the uncovered cells"""
    pf, z = load_golden(name)
    so = SmoothOracle(pf, per)
    c = np.random.default_rng(3).random(so.total)
    phi = so.solve(c, 1e-4)
    v = _vol(so, pf)
    u = so.uncovered
    assert abs(np.sum(v[u] * phi[u]) - np.sum(v[u] * c[u])) <= 1e-12 * np.sum(v[u] * c[u])


def test_oracle_covered_cells_are_fine_averages():
    pf, z = load_golden("c3_three_levels")
    so = SmoothOracle(pf, (1, 1, 1))
    c = np.random.default_rng(4).random(so.total)
    phi = so.solve(c, 1e-4)
    for l in range(so.nlev - 1):
        assert len(so.cov[l]) > 0
        assert np.allclose(phi[so.cov[l]], 0.125 * phi[so.cov_fine[l]].sum(axis=1), rtol=0, atol=1e-15)
    assert np.max(np.abs(phi - c)) > 1e-3          # the step did smooth


def test_oracle_zero_time_is_identity():
    pf, z = load_golden("c3_three_levels")
    so = SmoothOracle(pf, (1, 1, 1))
    c = np.random.default_rng(5).random(so.total)
    phi = so.solve(c, 0.0)
    assert np.array_equal(phi.view(np.int64), c.view(np.int64))
