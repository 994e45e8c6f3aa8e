"""Specification checks of B7, off-grid sources and receivers (tests/offgrid_reference.py), in float64, 2-D and 3-D.

B7 is the unchanged B1-B6 problem on the tap cells with the tap matrices around it, so its checks are: integral positions
are B2 bit for bit, the window parameter is the recorded minimiser, the operator with the matrices applied stays the
derivative and the adjoint of the forward (B3, B5), the free-surface fold is the doubled grid's image point, and - the
physical anchor - a point between cells moves the modelled arrival to where the analytic Green's function has it."""
import os
import sys

import numpy as np
import pytest

from oracle import fd_oracle as fo
from oracle import fd_oracle_c as foc
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))     # the B5 - B7 references live beside the tests
import born_reference as br  # noqa: E402
import free_surface_reference as fsr  # noqa: E402
import offgrid_reference as ogr  # noqa: E402
from test_fd_analytic import C, _exact, _rel, _ricker, _setup  # noqa: E402


def _case(ndim, seed=0):
    """Points within 4 cells of every edge, a receiver line at fractional x (shared taps), 0 < z < 1 for the surface."""
    rng = np.random.default_rng(seed)
    if ndim == 2:
        shape, nt, nabs = (30, 46), 120, 6
        src = [(0.6, 14.25), (5.5, 1.3), (27.2, 43.7)]
        rec = [(0.35, x + 0.4) for x in range(2, 42, 2)] + [(26.0, 40.0), (28.9, 0.0), (3.0, 44.6)]
    else:
        shape, nt, nabs = (14, 13, 18), 50, 3
        src = [(0.7, 6.2, 5.5), (3.0, 2.0, 12.4)]
        rec = [(0.45, y + 0.3, x + 0.6) for y in range(1, 12, 4) for x in range(1, 16, 3)] + [(10.0, 7.0, 9.0), (12.5, 11.8, 0.2)]
    v = fo.layered_model(shape, 1700.0, 2900.0, 3) + 40.0 * rng.standard_normal(shape)
    h = 10.0
    dt = fo.stable_dt(v.max(), h, ndim)
    wav = np.stack([fo.ricker(nt, dt, 25.0), 0.7 * fo.ricker(nt, dt, 19.0), -0.4 * fo.ricker(nt, dt, 21.0)], 1)[:, :len(src)]
    return v, h, dt, src, rec, wav, nabs


def _blobs(shape, centres, width):
    grids = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    return sum(np.exp(-sum((g - c) ** 2 for g, c in zip(grids, ctr)) / (2.0 * width ** 2)) for ctr in centres)


def test_window_parameter_is_the_recorded_minimiser():
    e = ogr.window_error(ogr.B)
    print("\nE(%.2f) = %.4e; E(b - 0.01) = %.4e, E(b + 0.01) = %.4e" % (ogr.B, e, ogr.window_error(ogr.B - 0.01), ogr.window_error(ogr.B + 0.01)))
    assert abs(e - ogr.E_B) <= 5e-3 * ogr.E_B
    assert ogr.window_error(ogr.B - 0.01) > e and ogr.window_error(ogr.B + 0.01) > e
    # a coarse scan finds nothing better elsewhere
    assert min(ogr.window_error(b, 40, 40) for b in np.arange(1.0, 10.0, 0.25)) >= 0.99 * ogr.window_error(ogr.B, 40, 40)


def test_taps():
    w = ogr.weights(0.5)
    assert np.allclose(w, w[::-1]) and abs(w.sum() - 1.0) < 1e-2
    assert np.allclose(ogr.weights(1e-12), [0, 0, 0, 1, 0, 0, 0, 0], atol=1e-10)      # continuous at f -> 0
    assert ogr.axis_taps(7.0, 20) == {7: 1.0}
    assert sorted(ogr.axis_taps(1.3, 20)) == list(range(0, 6))                          # taps below 0 dropped
    t = ogr.axis_taps(0.4, 20, fold=True)                                               # -3..-1 fold onto 3..1, row 0 dropped
    assert sorted(t) == [1, 2, 3, 4]
    full = dict(zip(range(-3, 5), ogr.weights(0.4)))
    assert t[2] == full[2] - full[-2]


@pytest.mark.parametrize("ndim,fs", [(2, False), (2, True), (3, False), (3, True)])
def test_integral_positions_are_the_plain_oracle(ndim, fs):
    v, h, dt, _, _, wav, nabs = _case(ndim)
    if ndim == 2:
        src, rec = [(3, 14), (5, 2)], [(1, x) for x in range(2, 44, 3)] + [(26, 40)]
    else:
        src, rec = [(3, 6, 5), (2, 2, 12)], [(1, y, x) for y in range(1, 12, 4) for x in range(1, 16, 3)]
    wav = wav[:, :2]
    plain = (fsr.Problem if fs else fo.Problem)(v, h, dt, src, rec, nabs=nabs)
    off = ogr.Problem(v, h, dt, np.asarray(src, float), np.asarray(rec, float), nabs=nabs, free_surface=fs)
    tr = plain.forward(wav)
    assert np.array_equal(off.forward(wav), tr)
    obs = 0.8 * tr
    J, g, _ = plain.misfit_and_gradient(wav, obs)
    J2, g2, _ = off.misfit_and_gradient(wav, obs)
    assert J == J2 and np.array_equal(g, g2)


@pytest.mark.parametrize("ndim,fs", [(2, False), (2, True), (3, False), (3, True)])
def test_adjoint_and_gauss_newton_identities(ndim, fs):
    """<J dv, r> = <dv, (2/v) adjoint(W_r^T r)> and <dv1, H dv2> = <J dv1, J dv2> = <dv2, H dv1> to 1e-12."""
    v, h, dt, src, rec, wav, nabs = _case(ndim, seed=3)
    p = ogr.Problem(v, h, dt, src, rec, nabs=nabs, free_surface=fs)
    rng = np.random.default_rng(4)
    dv1, dv2 = rng.standard_normal(v.shape), rng.standard_normal(v.shape)
    b1, _ = p.born(wav, dv1)
    b2, _ = p.born(wav, dv2)
    _, ws = p.base.forward(p.cell_wavelet(wav), save=True)
    r = rng.standard_normal(b1.shape)
    lhs = float(np.sum(b1 * r))
    rhs = float(np.sum(dv1 * (2.0 / p.v) * p.base.adjoint(r @ p.Wr, ws)))
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs), (lhs, rhs)
    mid = float(np.sum(b1 * b2))
    a = float(np.sum(dv1 * p.gauss_newton(wav, dv2)))
    b = float(np.sum(dv2 * p.gauss_newton(wav, dv1)))
    assert abs(a - mid) <= 1e-12 * abs(mid) and abs(b - mid) <= 1e-12 * abs(mid), (a, b, mid)


@pytest.mark.parametrize("fs", [False, True])
def test_gradient_matches_finite_differences(fs):
    v, h, dt, src, rec, wav, nabs = _case(2, seed=6)
    vt = v.copy()
    vt[8:14, 10:30] += 60.0
    obs = ogr.Problem(vt, h, dt, src, rec, nabs=nabs, free_surface=fs).forward(wav)
    J, g, _ = ogr.Problem(v, h, dt, src, rec, nabs=nabs, free_surface=fs).misfit_and_gradient(wav, obs)
    assert J > 0
    dv = _blobs(v.shape, [(3, 20), (12, 30)], 3.0)
    eps = 0.05
    Jp = fo.misfit(ogr.Problem(v + eps * dv, h, dt, src, rec, nabs=nabs, free_surface=fs).forward(wav), obs)
    Jm = fo.misfit(ogr.Problem(v - eps * dv, h, dt, src, rec, nabs=nabs, free_surface=fs).forward(wav), obs)
    fd = (Jp - Jm) / (2.0 * eps)
    an = float(np.sum(g * dv))
    assert abs(fd - an) <= 1e-5 * abs(an), (fd, an)


@pytest.mark.parametrize("fs", [False, True])
def test_born_is_the_derivative_of_the_forward(fs):
    v, h, dt, src, rec, wav, nabs = _case(2, seed=7)
    dv = _blobs(v.shape, [(15, 23), (2, 15)], 2.5)
    dtr, _ = ogr.Problem(v, h, dt, src, rec, nabs=nabs, free_surface=fs).born(wav, dv)
    errs = []
    for eps in (5.0, 2.5):
        tp = ogr.Problem(v + eps * dv, h, dt, src, rec, nabs=nabs, free_surface=fs).forward(wav)
        tm = ogr.Problem(v - eps * dv, h, dt, src, rec, nabs=nabs, free_surface=fs).forward(wav)
        errs.append(np.linalg.norm((tp - tm) / (2.0 * eps) - dtr) / np.linalg.norm(dtr))
    assert 3.0 <= errs[0] / errs[1] <= 5.0, errs          # falls as eps^2 (measured 1.4e-4 / 3.4e-5 with the surface)
    assert errs[1] <= 1e-4, errs


@pytest.mark.parametrize("ndim", [2, 3])
def test_free_surface_fold_is_the_doubled_grid(ndim):
    """The folded problem equals the plain problem on the grid doubled about row 0 with image points at -z (negated
    wavelets; for the gradient also negated observed data), to 1e-12."""
    v, h, dt, src, rec, wav, nabs = _case(ndim, seed=8)
    nz = v.shape[0]
    assert nz - 1 >= nabs
    p = ogr.Problem(v, h, dt, src, rec, nabs=nabs, free_surface=True)
    v2 = np.concatenate([v[:0:-1], v], 0)

    def doubled(pts):
        q = np.array(pts, np.float64)
        im = q.copy()
        q[:, 0] = nz - 1 + q[:, 0]
        im[:, 0] = nz - 1 - im[:, 0]
        return np.concatenate([q, im], 0)
    q = ogr.Problem(v2, h, dt, doubled(src), doubled(rec), nabs=nabs)
    tr, _, (cur, old) = p.forward(wav, return_state=True)
    tr2, _, (cur2, old2) = q.forward(np.concatenate([wav, -wav], 1), return_state=True)
    nrec = len(rec)
    scale = np.abs(tr).max()
    assert np.abs(tr - tr2[:, :nrec]).max() <= 1e-12 * scale and np.abs(tr + tr2[:, nrec:]).max() <= 1e-12 * scale
    assert np.abs(cur - cur2[nz - 1:]).max() <= 1e-12 * np.abs(cur).max()
    obs = 0.8 * tr + 0.05 * scale * np.random.default_rng(1).standard_normal(tr.shape)
    J, g, _ = p.misfit_and_gradient(wav, obs)
    J2, g2, _ = q.misfit_and_gradient(np.concatenate([wav, -wav], 1), np.concatenate([obs, -obs], 1))
    assert abs(2.0 * J - J2) <= 1e-12 * J2
    assert np.abs(g - g2[nz - 1:]).max() <= 1e-12 * np.abs(g).max()


def test_points_are_checked():
    shape = (30, 46)
    with pytest.raises(ValueError, match="source 1 .* not finite"):
        ogr.operator([(3.0, 4.0), (np.nan, 2.0)], shape, what="source")
    with pytest.raises(ValueError, match="outside the grid"):
        ogr.operator([(3.0, 45.01)], shape)
    with pytest.raises(ValueError, match="outside the grid"):
        ogr.operator([(-0.01, 5.0)], shape)
    with pytest.raises(ValueError, match="free surface"):
        ogr.operator([(0.0, 5.0)], shape, free_surface=True)
    cells, W = ogr.operator([(29.0, 45.0), (0.0, 0.5)], shape)          # the last cell; a point on the top edge
    assert W.shape == (2, len(cells)) and W[0].tolist().count(1.0) == 1
    assert set(cells[W[1] != 0][:, 0].tolist()) == {0} and cells[:, 1].min() == 0


# ------------------------------------------------------------------------------------------------ physical anchor
def _trace(h, dt, r, src_off, rec_off, rounded):
    """test_fd_analytic's 2-D set-up with the source and the receiver moved by the given cell offsets (z, x), modelled off
    grid or with both points rounded to the nearest cell.  Returns (trace, exact trace at the true distance)."""
    shape, src, rec, nt = _setup(2, h, dt, r + h)
    s = np.array(src[0], float) + src_off
    q = np.array(rec[0], float) + rec_off
    r_true = h * float(np.linalg.norm(q - s))
    if rounded:
        s, q = np.round(s), np.round(q)
    sc, Ws = ogr.operator([s], shape)
    rc, Wr = ogr.operator([q], shape)
    wav = _ricker(np.arange(nt) * dt)[:, None] @ Ws
    tr = foc.forward(np.full(shape, C), h, dt, sc, rc, wav, nabs=0, alpha=0.0, dtype=np.float64) @ Wr.T
    return tr[:, 0], _exact(2, h, dt, nt, r_true)


def test_offgrid_points_meet_the_analytic_greens_function():
    """Source at +0.37 cells and receiver at +0.61 cells on both axes, homogeneous 2-D medium, 480 m apart on the grid;
    rel-L2 error against the analytic trace at the true distance after Richardson extrapolation in time.  Printed;
    measured at h = 16 / 12 / 8 m: off grid 6.93e-03 / 8.02e-03 / 1.13e-02, both points rounded to the nearest cell
    4.59e-01 / 3.45e-01 / 2.30e-01 (on the grid, at integral offsets: 2.9e-03 / 3.4e-04 / 1.6e-05).  The off-grid error
    does not fall with h: it is the window's amplitude error at low wavenumbers, sum_k w_k - 1 = -0.42 % per fractional
    axis at these offsets (four such factors here), the price of the minimax b that E(b) bounds."""
    dt, r = 4e-4, 480.0
    src_off, rec_off = np.array([0.37, 0.37]), np.array([0.61, 0.61])
    errs = {}
    for rounded in (False, True):
        e = []
        for h in (16.0, 12.0, 8.0):
            tr1, ex = _trace(h, dt, r, src_off, rec_off, rounded)
            tr2, _ = _trace(h, dt / 2, r, src_off, rec_off, rounded)
            e.append(_rel((4.0 * tr2[1::2] - tr1) / 3.0, ex))
        errs[rounded] = e
    print("\noff-grid analytic check: rel-L2 at h = 16 / 12 / 8 m: off grid %s, rounded %s"
          % (["%.2e" % x for x in errs[False]], ["%.2e" % x for x in errs[True]]))
    for a, b in zip(errs[False], errs[True]):
        assert 10.0 * a <= b
    assert max(errs[False]) <= 1.5e-2
