"""Specification checks of B6, the free-surface top boundary (tests/free_surface_reference.py), in float64, 2-D and 3-D.

The anchor ties the new boundary to the unchanged B1 oracle: a free surface is the plain problem on a grid doubled about
row 0 with image sources (and image receivers for gradients).  The rest checks the consequences the spec states: a
zero surface row, a symmetric operator (so the B3 adjoint and the B5 identities hold unchanged) and the gradient against
finite differences of the misfit."""
import os
import sys

import numpy as np
import pytest

from oracle import fd_oracle as fo
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))     # the B5 / B6 references live beside the tests
import born_reference as br  # noqa: E402
import free_surface_reference as fs  # noqa: E402


def _case(ndim, seed=0):
    rng = np.random.default_rng(seed)
    if ndim == 2:
        shape, nt, nabs = (30, 46), 120, 6
        src = [(2, 14), (4, 30)]                           # inside the mirrored halo
        rec = [(1, x) for x in range(2, 44, 3)] + [(26, 40)]
    else:
        shape, nt, nabs = (14, 14, 18), 60, 3
        src = [(1, 7, 6), (3, 4, 12)]
        rec = [(1, y, x) for y in range(2, 13, 4) for x in range(2, 17, 4)] + [(10, 7, 9)]
    v = fo.layered_model(shape, 1700.0, 2900.0, 3) + 40.0 * rng.standard_normal(shape)
    h = 10.0
    dt = fo.stable_dt(v.max(), h, ndim)
    wav = np.stack([fo.ricker(nt, dt, 25.0), 0.7 * fo.ricker(nt, dt, 19.0)], 1)
    return v, h, dt, src, rec, wav, nabs


def _blobs(shape, centres, width):
    grids = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    return sum(np.exp(-sum((g - c) ** 2 for g, c in zip(grids, ctr)) / (2.0 * width ** 2)) for ctr in centres)


@pytest.mark.parametrize("ndim", [2, 3])
def test_free_surface_off_is_the_plain_oracle(ndim):
    """Flag off: B1 bit for bit, and points at z = 0 are allowed."""
    v, h, dt, src, rec, wav, nabs = _case(ndim)
    src = [(0,) + tuple(src[0][1:]), src[1]]
    a = fs.Problem(v, h, dt, src, rec, nabs=nabs, free_surface=False)
    b = fo.Problem(v, h, dt, src, rec, nabs=nabs)
    assert np.array_equal(a.g, b.g)
    assert np.array_equal(a.forward(wav), b.forward(wav))


@pytest.mark.parametrize("ndim", [2, 3])
def test_anchor_doubled_grid_with_image_sources(ndim):
    """Traces, final wavefields (rows >= 0), misfit and gradient equal the doubled plain grid's to float64 rounding."""
    v, h, dt, src, rec, wav, nabs = _case(ndim)
    nz = v.shape[0]
    assert nz - 1 >= nabs
    p = fs.Problem(v, h, dt, src, rec, nabs=nabs)
    tr, _, (cur, old) = p.forward(wav, return_state=True)
    v2, s2, r2 = fs.doubled(v, src, rec)
    q = fo.Problem(v2, h, dt, s2, r2, nabs=nabs)
    tr2, _, (cur2, old2) = q.forward(np.concatenate([wav, -wav], 1), return_state=True)
    scale = np.abs(tr).max()
    assert np.abs(tr - tr2).max() <= 1e-12 * scale
    assert np.abs(cur - cur2[nz - 1:]).max() <= 1e-12 * np.abs(cur).max()
    assert np.abs(old - old2[nz - 1:]).max() <= 1e-12 * np.abs(old).max()
    # gradients: image receivers with negated observed data
    obs = 0.8 * tr + 0.05 * scale * np.random.default_rng(1).standard_normal(tr.shape)
    J, g, _ = p.misfit_and_gradient(wav, obs)
    v2, s2, r2 = fs.doubled(v, src, rec, image_receivers=True)
    J2, g2, _ = fo.Problem(v2, h, dt, s2, r2, nabs=nabs).misfit_and_gradient(np.concatenate([wav, -wav], 1),
                                                                            np.concatenate([obs, -obs], 1))
    assert abs(2.0 * J - J2) <= 1e-12 * J2
    assert np.abs(g - g2[nz - 1:]).max() <= 1e-12 * np.abs(g).max()


@pytest.mark.parametrize("ndim", [2, 3])
def test_surface_row_and_gradient_row_are_zero(ndim):
    v, h, dt, src, rec, wav, nabs = _case(ndim, seed=2)
    p = fs.Problem(v, h, dt, src, rec, nabs=nabs)
    cur = np.zeros_like(p.v)
    old = np.zeros_like(p.v)
    for n in range(wav.shape[0]):
        new, w = p.step(cur, old, p.src, wav[n])
        assert not np.any(new[0]) and not np.any(w[0])
        old, cur = cur, new
    assert np.abs(cur).max() > 0
    tr = p.forward(wav)
    _, g, _ = p.misfit_and_gradient(wav, 0.5 * tr)
    assert not np.any(g[0]) and np.abs(g).max() > 0


def test_sponge_leaves_the_top_face_undamped():
    nabs, alpha = 5, 0.3
    g = fs.sponge((14, 12), nabs, alpha, True)
    plain = fo.sponge((14, 12), nabs, alpha)
    gx = fo.sponge_profile(12, nabs, alpha)
    assert np.array_equal(g[:nabs], np.broadcast_to(gx, (nabs, 12)))
    assert np.array_equal(g[-nabs:], plain[-nabs:])


def test_points_on_the_surface_are_rejected():
    v, h, dt, src, rec, wav, nabs = _case(2)
    with pytest.raises(ValueError, match="source 1 at \\(0, 9\\)"):
        fs.Problem(v, h, dt, [(3, 3), (0, 9)], rec, nabs=nabs)
    with pytest.raises(ValueError, match="receiver 0 at \\(0, 2\\)"):
        fs.Problem(v, h, dt, src, [(0, 2)], nabs=nabs)


@pytest.mark.parametrize("ndim", [2, 3])
def test_adjoint_identity(ndim):
    """<J dv, r> = <dv, (2/v) adjoint(r, ws)> with the free surface: the B3 adjoint is the transpose of the FS step."""
    v, h, dt, src, rec, wav, nabs = _case(ndim, seed=3)
    p = fs.Problem(v, h, dt, src, rec, nabs=nabs)
    dv = np.random.default_rng(4).standard_normal(v.shape)
    dtr, _ = br.born(p, wav, dv)
    _, ws = p.forward(wav, save=True)
    r = np.random.default_rng(5).standard_normal(dtr.shape)
    lhs = float(np.sum(dtr * r))
    rhs = float(np.sum(dv * (2.0 / p.v) * p.adjoint(r, ws)))
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs), (lhs, rhs)


def test_gradient_matches_finite_differences():
    """Directional derivative of the FS misfit along a perturbation near the surface vs <grad, dv>."""
    v, h, dt, src, rec, wav, nabs = _case(2, seed=6)
    tr = fs.Problem(v, h, dt, src, rec, nabs=nabs).forward(wav)
    vt = v.copy()
    vt[8:14, 10:30] += 60.0
    obs = fs.Problem(vt, h, dt, src, rec, nabs=nabs).forward(wav)
    J, g, _ = fs.Problem(v, h, dt, src, rec, nabs=nabs).misfit_and_gradient(wav, obs)
    assert J > 0 and np.abs(tr - obs).max() > 0
    dv = _blobs(v.shape, [(3, 20), (12, 30)], 3.0)
    eps = 0.05
    Jp = fo.misfit(fs.Problem(v + eps * dv, h, dt, src, rec, nabs=nabs).forward(wav), obs)
    Jm = fo.misfit(fs.Problem(v - eps * dv, h, dt, src, rec, nabs=nabs).forward(wav), obs)
    fd = (Jp - Jm) / (2.0 * eps)
    an = float(np.sum(g * dv))
    assert abs(fd - an) <= 1e-5 * abs(an), (fd, an)


# eps in m/s for a dv of peak ~1 m/s with one blob at the surface (errors at these eps, in float64: 2-D 5.2e-5 / 1.3e-5,
# 3-D 2.6e-6 / 6.5e-7)
@pytest.mark.parametrize("ndim,eps_pair,bound", [(2, (5.0, 2.5), 2e-5), (3, (2.5, 1.25), 1e-6)])
def test_born_is_the_derivative_of_the_forward(ndim, eps_pair, bound):
    v, h, dt, src, rec, wav, nabs = _case(ndim, seed=7)
    dv = _blobs(v.shape, [tuple(n // 2 for n in v.shape), (2,) + tuple(n // 3 for n in v.shape[1:])], 2.5)
    dtr, tr = br.born(fs.Problem(v, h, dt, src, rec, nabs=nabs), wav, dv)
    errs = []
    for eps in eps_pair:
        tp = fs.Problem(v + eps * dv, h, dt, src, rec, nabs=nabs).forward(wav)
        tm = fs.Problem(v - eps * dv, h, dt, src, rec, nabs=nabs).forward(wav)
        errs.append(np.linalg.norm((tp - tm) / (2.0 * eps) - dtr) / np.linalg.norm(dtr))
    assert 3.0 <= errs[0] / errs[1] <= 5.0, errs
    assert errs[1] <= bound, errs


@pytest.mark.parametrize("ndim", [2, 3])
def test_gauss_newton_is_symmetric(ndim):
    v, h, dt, src, rec, wav, nabs = _case(ndim, seed=8)
    rng = np.random.default_rng(9)
    dv1, dv2 = rng.standard_normal(v.shape), rng.standard_normal(v.shape)
    p = fs.Problem(v, h, dt, src, rec, nabs=nabs)
    b1, _ = br.born(p, wav, dv1)
    b2, _ = br.born(p, wav, dv2)
    mid = float(np.sum(b1 * b2))
    a = float(np.sum(dv1 * br.gauss_newton(p, wav, dv2)))
    b = float(np.sum(dv2 * br.gauss_newton(p, wav, dv1)))
    assert abs(a - mid) <= 1e-12 * abs(mid), (a, mid)
    assert abs(b - mid) <= 1e-12 * abs(mid), (b, mid)
