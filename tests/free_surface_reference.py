"""Float64 reference of the free-surface top boundary ("spec B6"), built on oracle/fd_oracle.py's Problem (B1-B4): the
subclass below changes only the Laplacian's values above row 0 and the sponge's top strip, so B1-B5 are untouched when
the flag is off, and tests/born_reference.py's `born` / `gauss_newton` give B5 with a free surface unchanged (they only
call `step`, `forward` and `adjoint`).  Test infrastructure only.

B6  free surface  flag `free_surface`, off by default (off: B1-B5 bit for bit).
    surface      grid row z = 0 (axis 0 in 2-D and 3-D).  Above the grid on the z axis the values are the odd mirror
                 u[-k] = -u[k], k = 1..4, instead of 0; rows k >= nz read 0.  Every other face keeps the zero halo.
    sponge       the top face is not damped: the z profile leaves out the strip at index 0 (so it is 1 on the first nabs
                 rows when nz >= 2 nabs); the bottom, x and y faces are unchanged.
    points       sources and receivers need z >= 1; a point at z = 0 is an error that names the point.
    consequences u_n[0] = 0 exactly for every n: the z terms of lap at row 0 cancel pairwise and nothing is injected there.
                 On rows >= 1 the Laplacian's z entries are c_|i-j| - c_(i+j): the operator is symmetric, so B3 (the same
                 step run on the time-reversed residual), dJ/dv = (2 / v) I and B5 hold as written.
                 The gradient is 0 on row 0 (w_n[0] = 0).
    anchor       for nz - 1 >= nabs the FS problem on nz rows equals, on rows >= 0, the plain B1 problem on 2 nz - 1 rows
                 with v mirrored about row 0 and, for every source at depth z, an image source at -z (row nz - 1 - z of
                 the doubled grid) with the negated wavelet; for gradients also image receivers with negated observed
                 data (the doubled misfit is 2 J, the gradient on rows >= 0 is the FS gradient).  Exact in exact
                 arithmetic, and bit for bit in float32 when the per-point operation order is the same: IEEE negation
                 commutes with rounding and the stencil's pairwise sums are commutative.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import fd_oracle as fo


def laplacian(u, free_surface=False):
    """fd_oracle.laplacian; with `free_surface` the 4 values above row 0 are the odd mirror of rows 1..4."""
    if not free_surface:
        return fo.laplacian(u)
    H = fo.HALO
    out = (fo.COEF[0] * u.ndim) * u
    p = np.pad(u, H)
    for k in range(1, H + 1):
        p[H - k] = -p[H + k]
    core = tuple(slice(H, H + n) for n in u.shape)
    for ax in range(u.ndim):
        for r in range(1, H + 1):
            lo = list(core)
            hi = list(core)
            lo[ax] = slice(H - r, H - r + u.shape[ax])
            hi[ax] = slice(H + r, H + r + u.shape[ax])
            out = out + fo.COEF[r] * (p[tuple(lo)] + p[tuple(hi)])
    return out


def sponge_profile(n, nabs, alpha, free_surface=False):
    """fd_oracle.sponge_profile; with `free_surface` the strip at index 0 is left out."""
    if not free_surface:
        return fo.sponge_profile(n, nabs, alpha)
    prof = np.ones(n)
    for i in range(min(nabs, n)):
        val = math.exp(-((alpha * (nabs - i) / nabs) ** 2))
        prof[n - 1 - i] = min(prof[n - 1 - i], val)
    return prof


def sponge(shape, nabs, alpha, free_surface=False):
    g = np.ones(shape)
    for ax, n in enumerate(shape):
        sh = [1] * len(shape)
        sh[ax] = n
        g = g * sponge_profile(n, nabs, alpha, free_surface and ax == 0).reshape(sh)
    return g


class Problem(fo.Problem):
    """fd_oracle.Problem with the B6 flag (on by default here)."""

    def __init__(self, v, h, dt, src, rec, nabs=20, alpha=0.3, dtype=np.float64, free_surface=True):
        super().__init__(v, h, dt, src, rec, nabs, alpha, dtype)
        self.free_surface = bool(free_surface)
        if self.free_surface:
            for what, pts in (("source", src), ("receiver", rec)):
                for i, pt in enumerate(np.asarray(pts, dtype=np.int64).reshape(-1, self.v.ndim)):
                    if pt[0] == 0:
                        raise ValueError("%s %d at %s lies on the free surface; sources and receivers need z >= 1"
                                         % (what, i, tuple(int(c) for c in pt)))
            self.g = sponge(self.v.shape, nabs, alpha, True).astype(dtype)

    def step(self, cur, old, inj_idx=None, inj_val=None):
        if not self.free_surface:
            return super().step(cur, old, inj_idx, inj_val)
        w = laplacian(cur, True)
        if inj_idx is not None:
            np.add.at(w, inj_idx, inj_val)
        new = self.g * (2.0 * cur - self.g * old + self.m * w)
        return new.astype(self.dtype), w.astype(self.dtype)


def doubled(v, src, rec, image_receivers=False):
    """The anchor's plain B1 problem: (v on 2 nz - 1 rows, sources + image sources, receivers [+ image receivers]).
    Row z of the FS grid is row nz - 1 + z of the doubled one; the images of the point lists follow the originals, so
    their wavelet / observed columns are the originals' negated: `np.concatenate([w, -w], 1)`."""
    v = np.asarray(v)
    nz = v.shape[0]
    v2 = np.concatenate([v[:0:-1], v], axis=0)

    def shift(pts, image):
        p = np.array(pts, dtype=np.int64).reshape(-1, v.ndim)
        q = p.copy()
        q[:, 0] = nz - 1 + p[:, 0]
        if not image:
            return q
        im = p.copy()
        im[:, 0] = nz - 1 - p[:, 0]
        return np.concatenate([q, im], 0)
    return v2, shift(src, True), shift(rec, image_receivers)
