"""Specification checks of B5, Born modelling and the Gauss-Newton Hessian (tests/born_reference.py), in float64, 2-D and 3-D.

Born is the exact derivative of the discrete forward, so it must match centred finite differences of
`fd_oracle.Problem.forward` with an error that falls as eps^2; the dot-product test ties it to the B3 adjoint (which
tests/test_fd_oracle.py ties to the misfit), and the Gauss-Newton product must be symmetric."""
import os
import sys

import numpy as np
import pytest

from oracle import fd_oracle as fo
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))     # the B5 reference lives beside the tests
import born_reference as br  # noqa: E402


def _blobs(shape, centres, width, rng):
    grids = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    dv = np.zeros(shape)
    for c in centres:
        r2 = sum((g - ci) ** 2 for g, ci in zip(grids, c))
        dv += rng.uniform(0.5, 1.0) * np.exp(-r2 / (2.0 * width ** 2))
    return dv


def _case(ndim, seed=0):
    rng = np.random.default_rng(seed)
    if ndim == 2:
        shape, nt, nabs = (34, 46), 90, 6
        src = [(5, 14)]
        rec = [(4, x) for x in range(2, 44, 3)] + [(30, 40)]
        centres = [(18, 23), (3, 40), (30, 10)]           # one inside the sponge strip
    else:
        shape, nt, nabs = (16, 14, 18), 50, 3
        src = [(4, 7, 6)]
        rec = [(3, y, x) for y in range(2, 13, 4) for x in range(2, 17, 4)]
        centres = [(9, 7, 9), (14, 2, 15)]
    v = fo.layered_model(shape, 1700.0, 2900.0, 3) + 40.0 * rng.standard_normal(shape)
    h = 10.0
    dt = fo.stable_dt(v.max(), h, ndim)
    wav = fo.ricker(nt, dt, 25.0 if ndim == 2 else 30.0)[:, None]
    dv = _blobs(shape, centres, 2.5, rng)
    return v, h, dt, src, rec, wav, dv, nabs


# eps pairs (m/s, dv peaks at ~1 m/s) where the eps^2 truncation error is above the float64 cancellation error of the
# difference (measured: 2-D 7.8e-8 / 2.0e-8 at eps 160 / 80; 3-D 1.1e-7 / 2.8e-8 at 10 / 5; below them cancellation wins)
@pytest.mark.parametrize("ndim,eps_pair", [(2, (160.0, 80.0)), (3, (10.0, 5.0))])
def test_born_is_the_derivative_of_the_forward(ndim, eps_pair):
    v, h, dt, src, rec, wav, dv, nabs = _case(ndim)
    dtr, tr = br.born(fo.Problem(v, h, dt, src, rec, nabs=nabs), wav, dv)
    assert np.array_equal(tr, fo.Problem(v, h, dt, src, rec, nabs=nabs).forward(wav))
    errs = []
    for eps in eps_pair:
        tp = fo.Problem(v + eps * dv, h, dt, src, rec, nabs=nabs).forward(wav)
        tm = fo.Problem(v - eps * dv, h, dt, src, rec, nabs=nabs).forward(wav)
        fd = (tp - tm) / (2.0 * eps)
        errs.append(np.linalg.norm(fd - dtr) / np.linalg.norm(dtr))
    # second order: halving eps divides the error by ~4
    assert 3.0 <= errs[0] / errs[1] <= 5.0, errs
    assert errs[1] <= 1e-7, errs


@pytest.mark.parametrize("ndim", [2, 3])
def test_born_is_the_adjoint_of_the_gradient(ndim):
    """<J dv, r> = <dv, (2/v) adjoint(r, ws)> for a random r."""
    v, h, dt, src, rec, wav, dv, nabs = _case(ndim, seed=1)
    p = fo.Problem(v, h, dt, src, rec, nabs=nabs)
    dtr, _ = br.born(p, wav, dv)
    _, ws = p.forward(wav, save=True)
    r = np.random.default_rng(2).standard_normal(dtr.shape)
    lhs = float(np.sum(dtr * r))
    rhs = float(np.sum(dv * (2.0 / p.v) * p.adjoint(r, ws)))
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs), (lhs, rhs)


@pytest.mark.parametrize("ndim", [2, 3])
def test_gauss_newton_is_symmetric_and_matches_born(ndim):
    """<dv1, H dv2> = <J dv1, J dv2> = <dv2, H dv1>."""
    v, h, dt, src, rec, wav, dv1, nabs = _case(ndim, seed=3)
    dv2 = np.random.default_rng(4).standard_normal(v.shape)
    p = fo.Problem(v, h, dt, src, rec, nabs=nabs)
    b1, _ = br.born(p, wav, dv1)
    b2, _ = br.born(p, wav, dv2)
    mid = float(np.sum(b1 * b2))
    a = float(np.sum(dv1 * br.gauss_newton(p, wav, dv2)))
    b = float(np.sum(dv2 * br.gauss_newton(p, wav, dv1)))
    assert abs(a - mid) <= 1e-12 * abs(mid), (a, mid)
    assert abs(b - mid) <= 1e-12 * abs(mid), (b, mid)
