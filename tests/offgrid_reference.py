"""Float64 reference of off-grid sources and receivers ("spec B7"), built on oracle/fd_oracle.py's Problem (B1-B4) and
tests/free_surface_reference.py's (B6): a point between cells is a short weighted list of cells, and the reference runs the
unchanged problem on those cells with the tap matrices applied around it, so there is no second propagator.  Test
infrastructure only.

B7  off-grid points   a position is a float coordinate per axis in cell units, (z, x) in 2-D and (z, y, x) in 3-D;
                      10.5 lies half-way between rows 10 and 11.
    taps per axis     i = floor(x), f = x - i.  f == 0: one tap at i, weight 1.  Otherwise 8 taps at i + k, k = -3 .. 4,
                      d = k - f,  w = sinc(d) I0(b sqrt(1 - (d/4)^2)) / I0(b),  sinc(d) = sin(pi d) / (pi d): Hicks' (2002)
                      Kaiser-windowed sinc with half-width r = 4, the stencil's halo.  2-D / 3-D weights are the tensor
                      product of the per-axis weights, computed in float64.
    window b          b = 4.06, the b on a 0.01 grid that minimises
                      E(b) = max |sum_k w_k(f) exp(i kappa d_k) - 1| over kappa in [0, 2 pi / 3], f in [0, 1)
                      (how well the taps represent a shifted delta for the wavenumbers the 8th-order stencil carries);
                      E(4.06) = 8.79e-3, attained at f = 1/2, kappa = 2 pi / 3.
    sources           a source injects wavelet x weight at each of its tap cells: B2 on the cells, wavelet matrix W_s^T w.
    receivers         trace[n, r] = sum_taps w u_{n+1}[cell].
    misfit / adjoint  J = 1/2 sum (W_r syn_cells - obs)^2; the adjoint injects W_r^T r at the cells, so B3, dJ/dv = (2/v) I
                      and B5 hold as written (born_reference's `born` / `gauss_newton` with W_s, W_r around them).
    edges             taps outside the grid are dropped (exact with B1's zero halo); a point must lie in [0, n - 1] on
                      every axis.
    free surface (B6) a point needs z > 0 (so 0 < z < 1 is allowed).  A tap at row -k folds onto row +k with its weight
                      negated (the odd mirror); a tap at row 0 is dropped.  Taps of one point on one cell are merged in
                      float64 (the CUDA path then rounds the merged weight to float32).
"""
from __future__ import annotations

import numpy as np

from oracle import fd_oracle as fo

B = 4.06
E_B = 8.79e-3
R = 4


def weights(f, b=B):
    """The 8 Kaiser-windowed sinc weights of taps k = -3 .. 4 for fractional parts f (any shape) -> (..., 8)."""
    d = np.arange(-R + 1, R + 1) - np.asarray(f, np.float64)[..., None]
    return np.sinc(d) * np.i0(b * np.sqrt(np.clip(1.0 - (d / R) ** 2, 0.0, None))) / np.i0(b)


def window_error(b, nf=200, nk=200):
    """E(b) on an f grid of step 1/nf over [0, 1) and nk wavenumbers over [0, 2 pi / 3] (both grids hold the maximiser)."""
    f = np.arange(nf) / nf
    kappa = np.linspace(0.0, 2.0 * np.pi / 3.0, nk)
    d = np.arange(-R + 1, R + 1)[None, :] - f[:, None]
    s = np.einsum("fk,fkq->fq", weights(f, b), np.exp(1j * kappa[None, None, :] * d[:, :, None]))
    return float(np.abs(s - 1.0).max())


def axis_taps(x, n, fold=False):
    """{index: weight} of one coordinate on an axis of n cells; `fold`: the free-surface z axis."""
    i = int(np.floor(x))
    f = x - i
    if f == 0.0:
        return {i: 1.0}
    out = {}
    for k, w in zip(range(-R + 1, R + 1), weights(f)):
        j = i + k
        if fold and j < 0:
            j, w = -j, -w
        if (fold and j == 0) or j < 0 or j >= n:
            continue
        out[j] = out.get(j, 0.0) + float(w)
    return out


def check_points(pts, shape, free_surface, what):
    pts = np.asarray(pts, np.float64).reshape(-1, len(shape))
    for i, p in enumerate(pts):
        if not np.all(np.isfinite(p)):
            raise ValueError("%s %d at %s is not finite" % (what, i, tuple(p)))
        if np.any(p < 0) or np.any(p > np.asarray(shape) - 1):
            raise ValueError("%s %d at %s is outside the grid" % (what, i, tuple(p)))
        if free_surface and p[0] <= 0:
            raise ValueError("%s %d at %s lies on the free surface" % (what, i, tuple(p)))
    return pts


def operator(pts, shape, free_surface=False, what="point"):
    """(cells (ncells, ndim) int, W (npts, ncells) float64): the unique tap cells in ascending linear order and the weights."""
    pts = check_points(pts, shape, free_surface, what)
    taps = []
    for p in pts:
        axes = [axis_taps(c, n, free_surface and a == 0) for a, (c, n) in enumerate(zip(p, shape))]
        t = {(): 1.0}
        for ax in axes:
            t = {key + (j,): w * wj for key, w in t.items() for j, wj in ax.items()}
        taps.append(t)
    cells = sorted({c for t in taps for c in t})
    col = {c: k for k, c in enumerate(cells)}
    W = np.zeros((len(pts), len(cells)))
    for i, t in enumerate(taps):
        for c, w in t.items():
            W[i, col[c]] += w
    return np.array(cells, dtype=np.int64).reshape(-1, len(shape)), W


class Problem:
    """One shot with off-grid points: the cell-level `base` problem (fd_oracle.Problem, or free_surface_reference.Problem
    with `free_surface`) and the tap matrices Ws (nsrc x source cells), Wr (nrec x receiver cells)."""

    def __init__(self, v, h, dt, src, rec, nabs=20, alpha=0.3, dtype=np.float64, free_surface=False):
        shape = np.shape(v)
        src_cells, self.Ws = operator(src, shape, free_surface, "source")
        rec_cells, self.Wr = operator(rec, shape, free_surface, "receiver")
        if free_surface:
            import free_surface_reference as fsr
            self.base = fsr.Problem(v, h, dt, src_cells, rec_cells, nabs, alpha, dtype)
        else:
            self.base = fo.Problem(v, h, dt, src_cells, rec_cells, nabs, alpha, dtype)
        self.v = self.base.v

    def cell_wavelet(self, wavelet):
        return np.asarray(wavelet, np.float64).reshape(len(wavelet), -1) @ self.Ws

    def forward(self, wavelet, return_state=False):
        out = self.base.forward(self.cell_wavelet(wavelet), return_state=return_state)
        if return_state:
            tr, ws, state = out
            return tr @ self.Wr.T, ws, state
        return out @ self.Wr.T

    def misfit_and_gradient(self, wavelet, obs):
        tr, ws = self.base.forward(self.cell_wavelet(wavelet), save=True)
        tr = tr @ self.Wr.T
        res = tr - np.asarray(obs, np.float64)
        J = 0.5 * float(np.sum(res ** 2))
        return J, (2.0 / self.v) * self.base.adjoint(res @ self.Wr, ws), tr

    def born(self, wavelet, dv):
        import born_reference as br
        dtr, tr = br.born(self.base, self.cell_wavelet(wavelet), dv)
        return dtr @ self.Wr.T, tr @ self.Wr.T

    def gauss_newton(self, wavelet, dv):
        import born_reference as br
        dtr, _, ws = br._born(self.base, self.cell_wavelet(wavelet), dv)
        return (2.0 / self.v) * self.base.adjoint((dtr @ self.Wr.T) @ self.Wr, ws)
