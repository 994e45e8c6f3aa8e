"""Pointwise comparison of the CUDA propagators with a float64 reference (TEST INFRASTRUCTURE ONLY).

A global rel-L2 is blind wherever the field is weak (far receivers, late samples, deep gradient, sponge strips, the last
tiles), because the strong arrivals next to the sources dominate the norm.  The checks here bound the error at every grid
point instead, by a scale that is large only where float32 rounding can be large:

  one step   |got - ref| <= K1 eps32 S,   S = g (2|u_n| + g|u_{n-1}| + m (sum_k |c_k| |u_k| + |f|))
             (the float64 result of one step from the same float32 inputs; S is the sum of the magnitudes that the
             float32 update rounds, so a correct float32 step stays within a few eps32 S at every point)
  a sweep    |got - ref| <= K2 eps32 max_9x9|ref|   (local maximum of the float64 result over the 9-point neighbourhood
             per axis, for each step's field and for the gradient)

A failure names the worst points: (z, [y,] x), the step, the tile of the plan's decomposition that owns the point and a
region label (sponge strip, last tile row / column / y-row, z-chunk boundary, interior).  `region_table` gives rel-L2 per
selection (receiver group x time window, gradient region) next to the float32 port's, for long sweeps.
"""
from __future__ import annotations

import math

import numpy as np

from . import fd_oracle as fo

EPS32 = float(np.finfo(np.float32).eps)
HALO = 4
STEP_TILES = ((32, 4), (28, 4), (42, 6), (56, 8))        # the one-step kernel's built (rows, warps); csrc/fd2d.cu kTileShapes
TB2_CORE_X = 120                                         # two-steps-per-pass kernel: 120-column core tiles (fd2d_tb2.cuh)
TILE_X = 128                                             # one-step 2-D and 3-D kernels: 128-column tiles


# ------------------------------------------------------------------------------------------------ decomposition
def pick_tile(nz, nx, sms):
    """The one-step kernel's tile height for a grid (csrc/fd2d.cu pick_tile): fewest waves x (rows + 4)."""
    tx = -(-nx // TILE_X)
    best, out = 1e300, STEP_TILES[0]
    for bz, nw in STEP_TILES:
        cost = (-(-(tx * -(-nz // bz)) // sms)) * (bz + 4)
        if cost < best - 1e-9:
            best, out = cost, (bz, nw)
    return out


def zchunks_3d(nz, ny, nx, by, sms):
    """z-chunk length of a single-GPU 3-D plan with tile height `by` (csrc/fd2d.cu make_tmaps3)."""
    txy = -(-nx // TILE_X) * -(-ny // by)
    best, best_n = 1e300, 1
    for nzch in range(1, max(1, nz // 8) + 1):
        zc = -(-nz // nzch)
        real = -(-nz // zc)
        cost = math.ceil(txy * real / sms) * (zc + 2 * HALO) * by
        if cost < best - 1e-9:
            best, best_n = cost, nzch
    return -(-nz // best_n)


class Decomp:
    """The tiles of a plan: kind 'tile' (one-step 2-D kernel, bz x 128), 'tb2' (two-steps-per-pass, cz x 120 cores) or
    '3d' (by x 128 columns, z chunks of `zchunk` planes)."""

    def __init__(self, shape, kind, tz=None, ty=None, tx=TILE_X, zchunk=None, nabs=0):
        self.shape, self.kind, self.nabs = tuple(shape), kind, nabs
        self.tz, self.ty, self.tx, self.zchunk = tz, ty, tx, zchunk
        self.px = -(-self.shape[-1] // 32) * 32

    @classmethod
    def for_plan(cls, shape, sms, nabs, tile=None, tb2=None, by=None):
        """The decomposition fwi_fd2d_create / fwi_fd3d_create choose (or the forced tile / tb2 / BY)."""
        shape = tuple(shape)
        if len(shape) == 3:
            by = by or 16
            return cls(shape, "3d", ty=by, zchunk=zchunks_3d(*shape, by, sms), nabs=nabs)
        nz, nx = shape
        if tile is None and tb2 is None and nz >= 32 and nx >= 128:
            tb2 = 24 if nz * nx <= 2.0e6 else (32 if nz * nx > 7.5e6 else None)
        if tile is None and tb2 is not None:
            return cls(shape, "tb2", tz=tb2, tx=TB2_CORE_X, nabs=nabs)
        bz = tile[0] if tile is not None else (pick_tile(nz, nx, sms)[0] if nz >= 32 else 32)
        return cls(shape, "tile", tz=bz, nabs=nabs)

    def __repr__(self):
        if self.kind == "3d":
            return "3d(by=%d, zchunk=%d)" % (self.ty, self.zchunk)
        return "%s(%d x %d)" % (self.kind, self.tz, self.tx)

    def tile_of(self, idx):
        """Tile index of a grid point: (tile row, tile column) in 2-D, (z chunk, y tile, x tile) in 3-D."""
        if self.kind == "3d":
            z, y, x = (int(i) for i in idx)
            return (z // self.zchunk, y // self.ty, x // self.tx)
        z, x = (int(i) for i in idx)
        return (z // self.tz, x // self.tx)

    def _axes(self):
        """(axis name, axis length, tile length along it, 'last tile' label) per axis."""
        if self.kind == "3d":
            nz, ny, nx = self.shape
            return (("z", nz, self.zchunk, "last-z-chunk"), ("y", ny, self.ty, "last-tile-y"), ("x", nx, self.tx, "last-tile-col"))
        nz, nx = self.shape
        return (("z", nz, self.tz, "last-tile-row"), ("x", nx, self.tx, "last-tile-col"))

    def label(self, idx):
        """Region label of a grid point, e.g. 'sponge-right+last-tile-col' or 'interior'."""
        names = {"z": ("top", "bottom"), "y": ("front", "back"), "x": ("left", "right")}
        out = []
        for (ax, n, t, last), i in zip(self._axes(), idx):
            if ax == "x" and i >= n:
                return "pad"
            if i < self.nabs:
                out.append("sponge-" + names[ax][0])
            elif i >= n - self.nabs:
                out.append("sponge-" + names[ax][1])
            if i >= (n - 1) // t * t and n > t:
                out.append(last + ("" if n % t == 0 else "(partial)"))
            if self.kind == "3d" and ax == "z" and n > t and (i % t < HALO or i % t >= t - HALO):
                out.append("z-chunk-edge")
        return "+".join(out) or "interior"

    def masks(self):
        """Boolean masks of the regions a long sweep is checked on: sponge strips, last tile row / column, interior."""
        full = np.zeros(self.shape, dtype=bool)
        out = {}
        for k, (ax, n, t, last) in enumerate(self._axes()):
            idx = np.arange(n).reshape([-1 if j == k else 1 for j in range(len(self.shape))])
            if self.nabs:
                out["sponge-" + {"z": "top", "y": "front", "x": "left"}[ax]] = np.broadcast_to(idx < self.nabs, self.shape)
                out["sponge-" + {"z": "bottom", "y": "back", "x": "right"}[ax]] = np.broadcast_to(idx >= n - self.nabs, self.shape)
            if n > t:
                out[last] = np.broadcast_to(idx >= (n - 1) // t * t, self.shape)
        for m in out.values():
            full = full | m
        out["interior"] = ~full
        return out


# ------------------------------------------------------------------------------------------------ references
def abs_laplacian(a):
    """sum_k |c_k| |u_k| over the 8th-order star of every point (a = |u|; zero outside the grid)."""
    out = (abs(fo.COEF[0]) * a.ndim) * a
    p = np.pad(a, HALO)
    core = [slice(HALO, HALO + n) for n in a.shape]
    for ax in range(a.ndim):
        for r in range(1, HALO + 1):
            lo, hi = list(core), list(core)
            lo[ax] = slice(HALO - r, HALO - r + a.shape[ax])
            hi[ax] = slice(HALO + r, HALO + r + a.shape[ax])
            out += abs(fo.COEF[r]) * (p[tuple(lo)] + p[tuple(hi)])
    return out


def model(v, h, dt, nabs, alpha):
    """(m, g) of the specification in float64 (fd_oracle B1)."""
    v = np.asarray(v, np.float64)
    return (v * (dt / h)) ** 2, fo.sponge(v.shape, nabs, alpha)


def step64(cur, old, m, g, inj=None):
    """One step in float64 from (float32) inputs -> (u_{n+1}, w_n, S, A_w).  inj = (index tuple, values) adds f_n to w_n.
    S bounds what float32 rounds in u_{n+1}; A_w = sum_k |c_k| |u_k| + |f| does the same for w_n."""
    cur = np.asarray(cur, np.float64)
    old = np.asarray(old, np.float64)
    w = fo.laplacian(cur)
    aw = abs_laplacian(np.abs(cur))
    if inj is not None:
        np.add.at(w, inj[0], np.asarray(inj[1], np.float64))
        np.add.at(aw, inj[0], np.abs(np.asarray(inj[1], np.float64)))
    new = g * (2.0 * cur - g * old + m * w)
    S = g * (2.0 * np.abs(cur) + g * np.abs(old) + m * aw)
    return new, w, S, aw


def local_max(a, size=9):
    """Maximum of |a| over the size^ndim neighbourhood of every point (zero outside the grid)."""
    from scipy.ndimage import maximum_filter
    return maximum_filter(np.abs(np.asarray(a, np.float64)), size=size, mode="constant", cval=0.0)


# ------------------------------------------------------------------------------------------------ checks and reports
class Result:
    """Outcome of one pointwise check: worst ratio err / (eps32 scale) and the report of the worst points."""

    def __init__(self, name, K, worst, lines, first_fail=None):
        self.name, self.K, self.worst, self.lines, self.first_fail = name, K, worst, lines, first_fail

    @property
    def ok(self):
        return self.worst <= self.K

    @property
    def where(self):
        """(step, index, label) of the first failing point (earliest step, worst point there), or of the worst point."""
        return self.first_fail

    def summary(self):
        step, idx, lab = self.first_fail
        return "%s: worst err/(eps*scale) = %.3g (K = %g); %s %s%s [%s]" % (
            self.name, self.worst, self.K, "worst point" if self.ok else "first failure at", tuple(int(i) for i in idx),
            "" if step is None else " step %d" % step, lab)

    def report(self):
        return "\n".join([self.summary()] + self.lines)

    def check(self):
        assert self.ok, self.report()
        return self


def _ratio(got, ref, scale):
    err = np.abs(np.asarray(got, np.float64) - np.asarray(ref, np.float64))
    with np.errstate(divide="ignore", invalid="ignore"):
        r = err / (EPS32 * scale)
    r[err == 0] = 0.0
    r[np.isnan(r)] = np.inf
    return r, err


def _worst_lines(r, err, ref, scale, decomp, step, k):
    flat = np.argsort(r, axis=None)[::-1][:k]
    lines = []
    for f in flat:
        idx = np.unravel_index(f, r.shape)
        if r[idx] == 0:
            break
        lines.append("  %s%s  err %.3e  ref %.3e  scale %.3e  ratio %.3g  tile %s  %s" % (
            "" if step is None else "step %d  " % step, tuple(int(i) for i in idx), err[idx], ref[idx], scale[idx], r[idx],
            decomp.tile_of(idx) if decomp else "-", decomp.label(idx) if decomp else ""))
    return lines


def check_points(name, got, ref, scale, K, decomp=None, step=None, k=5):
    """|got - ref| <= K eps32 scale at every point."""
    r, err = _ratio(got, ref, scale)
    idx = np.unravel_index(int(np.argmax(r)), r.shape)
    return Result(name, K, float(r[idx]), _worst_lines(r, err, np.asarray(ref), scale, decomp, step, k),
                  (step, idx, decomp.label(idx) if decomp else ""))


def check_sweep(name, got_steps, ref_steps, K, decomp=None, size=9, k=5, scales=None):
    """Sweep bound for a sequence of fields (e.g. every step's wavefield): |got - ref| <= K eps32 max_local|ref| per
    step (`scales`: the local maxima, if already computed).  The report names the worst points of the first failing
    step (where a bug shows first, before the error has spread) and the worst ratio overall."""
    worst, first, lines, worst_at = 0.0, None, [], None
    for n, (got, ref) in enumerate(zip(got_steps, ref_steps)):
        res = check_points(name, got, ref, local_max(ref, size) if scales is None else scales[n], K, decomp, step=n, k=k)
        if res.worst > worst:
            worst, worst_at = res.worst, res.first_fail
        if first is None and not res.ok:
            first, lines = res.first_fail, ["  first failing step %d:" % n] + res.lines
    out = Result(name, K, worst, lines, first or worst_at or (0, (0,) * np.ndim(ref_steps[0]), ""))
    if first is not None and worst_at != first:
        out.lines.append("  worst overall: step %d %s [%s]" % (worst_at[0], tuple(int(i) for i in worst_at[1]), worst_at[2]))
    return out


def check_field(name, got, ref, K, decomp=None, size=9, k=5):
    """Sweep bound for one field (final state, gradient)."""
    return check_points(name, got, ref, local_max(ref, size), K, decomp, k=k)


# ------------------------------------------------------------------------------------------------ long sweeps
def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    nb = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / nb) if nb > 0 else (0.0 if not np.any(a) else math.inf)


def trace_selections(groups, nt, windows):
    """{'group t0:t1': (row slice, column indices)} for every receiver group x time window."""
    return {"%s t%d:%d" % (g, t0, t1): (slice(t0, t1), np.asarray(cols)) for g, cols in groups.items() for t0, t1 in windows}


def region_table(got, f32, ref, selections):
    """Rows (name, rel-L2 of got, rel-L2 of the float32 port, share of the float64 norm) per selection; a selection is
    an index usable on the arrays (a (rows, cols) tuple for traces, a boolean mask for a gradient)."""
    total = np.linalg.norm(np.asarray(ref, np.float64))
    rows = []
    for name, sel in selections.items():
        b = np.asarray(ref[sel], np.float64)
        rows.append((name, rel_l2(got[sel], b), rel_l2(f32[sel], b), float(np.linalg.norm(b) / total)))
    return rows


def format_table(title, rows):
    out = ["%s\n  %-36s %12s %12s %12s" % (title, "selection", "GPU rel-L2", "fp32 port", "norm share")]
    out += ["  %-36s %12.3e %12.3e %12.3e" % r for r in rows]
    return "\n".join(out)
