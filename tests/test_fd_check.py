"""The pointwise comparator of oracle/fd_check.py on the CPU: the float32 C port of the self-oracle must pass it against
the float64 build, and float32 runs with one planted bug (a sponge value off by one cell in the last column, one stencil
neighbour read from the wrong row in the last partial tile row, one injection dropped next to a tile corner) must fail
it at the planted place.  The grid has 70 x 300 points, so in the 32 x 128 tiles of the one-step kernel the last tile row
(z >= 64) and the last tile column (x >= 256) are partial."""
import numpy as np
import pytest

from oracle import fd_check as fc
from oracle import fd_oracle as fo
from oracle import fd_oracle_c as foc

# the bounds of test_fd_fullgrid_gpu.py (the float32 C port measures 1.5 for one step, 5.9 for the fields, 11.1 for the
# gradient here)
K1, K2, K2_GRAD = 16.0, 128.0, 256.0
NZ, NX, NT, NABS, ALPHA, H = 70, 300, 9, 10, 0.3, 10.0
DEC = fc.Decomp((NZ, NX), "tile", tz=32, nabs=NABS)


def lattice(nz, nx, every=3):
    """Points every `every` cells plus every edge row and column (corners included)."""
    zz, xx = np.meshgrid(np.union1d(np.arange(0, nz, every), [nz - 1]), np.union1d(np.arange(0, nx, every), [nx - 1]), indexing="ij")
    return np.stack([zz.ravel(), xx.ravel()], 1)


@pytest.fixture(scope="module")
def case():
    rng = np.random.default_rng(11)
    v = (fo.layered_model((NZ, NX), 1500.0, 4500.0, 4) + 60.0 * rng.standard_normal((NZ, NX))).astype(np.float32)
    dt = fo.stable_dt(float(v.max()), H, 2)
    src = lattice(NZ, NX)
    rec = np.stack(np.meshgrid(np.arange(NZ), np.arange(NX), indexing="ij"), -1).reshape(-1, 2)
    wav = rng.standard_normal((NT, len(src))).astype(np.float32)
    ref = foc.forward(v, H, dt, src, rec, wav, nabs=NABS, alpha=ALPHA, dtype=np.float64).reshape(NT, NZ, NX)
    return dict(v=v, dt=dt, src=src, rec=rec, wav=wav, ref=ref)


def sweep32(c, g=None, lap=fo.laplacian, drop=None):
    """Float32 NumPy sweep with dense injection (every step's field), optionally with a planted bug:
    g = a wrong sponge, lap = a wrong stencil, drop = (step, source) whose injection is skipped."""
    P = fo.Problem(c["v"], H, c["dt"], c["src"], [(0, 0)], NABS, ALPHA, dtype=np.float32)
    gg = P.g if g is None else g.astype(np.float32)
    cur = np.zeros((NZ, NX), np.float32)
    old = np.zeros_like(cur)
    out = []
    for n in range(NT):
        vals = c["wav"][n].copy()
        if drop is not None and drop[0] == n:
            vals[drop[1]] = 0.0
        w = lap(cur)
        np.add.at(w, P.src, vals)
        new = gg * (2.0 * cur - gg * old + P.m * w)
        assert new.dtype == np.float32
        out.append(new)
        old, cur = cur, new
    return np.stack(out)


def test_float32_port_passes_the_sweep_bound(case):
    """Every step's field and the gradient of the float32 C port against the float64 build, and the final state."""
    c = case
    got = foc.forward(c["v"], H, c["dt"], c["src"], c["rec"], c["wav"], nabs=NABS, alpha=ALPHA, dtype=np.float32)
    res = fc.check_sweep("fp32 port fields", got.reshape(NT, NZ, NX), c["ref"], K2, DEC)
    print("\n" + res.summary())
    res.check()
    obs = np.random.default_rng(3).standard_normal((NT, len(c["rec"]))).astype(np.float32)
    _, g64, _ = foc.misfit_and_gradient(c["v"], H, c["dt"], c["src"], c["rec"], c["wav"], obs, NABS, ALPHA, dtype=np.float64)
    _, g32, _ = foc.misfit_and_gradient(c["v"], H, c["dt"], c["src"], c["rec"], c["wav"], obs, NABS, ALPHA, dtype=np.float32)
    res = fc.check_field("fp32 port gradient", g32, g64, K2_GRAD, DEC)
    print(res.summary())
    res.check()
    assert res.worst > 0.0                                    # the comparison is not vacuous


def test_numpy_float32_sweep_passes_too(case):
    """The float32 NumPy sweep the planted-bug tests start from is itself within the bound."""
    res = fc.check_sweep("fp32 numpy", sweep32(case), case["ref"], K2, DEC).check()
    assert 0.0 < res.worst


def test_one_step_bound_on_random_fields(case):
    """One float32 step from random fields (with injection at the lattice) against step64 with its scale S."""
    rng = np.random.default_rng(4)
    c = case
    cur, old = (rng.standard_normal((NZ, NX)).astype(np.float32) for _ in range(2))
    P = fo.Problem(c["v"], H, c["dt"], c["src"], [(0, 0)], NABS, ALPHA, dtype=np.float32)
    new32, w32 = P.step(cur, old, P.src, c["wav"][0])
    m, g = fc.model(c["v"], H, c["dt"], NABS, ALPHA)
    new, w, S, aw = fc.step64(cur, old, m, g, (P.src, c["wav"][0]))
    res = fc.check_points("one step", new32, new, S, K1, DEC)
    print("\n" + res.summary())
    res.check()
    fc.check_points("one step w", w32, w, aw, K1, DEC).check()
    assert res.worst > 0.1


def test_sponge_misindex_in_the_last_column_is_caught(case):
    """gx[nx-1] takes the profile value of nx-2 (about 4e-3 relative, ~3e4 eps): fails, at column nx-1."""
    gx = fo.sponge_profile(NX, NABS, ALPHA)
    gx[NX - 1] = gx[NX - 2]
    g = fo.sponge_profile(NZ, NABS, ALPHA)[:, None] * gx[None, :]
    res = fc.check_sweep("sponge misindex", sweep32(case, g=g), case["ref"], K2, DEC)
    print("\n" + res.report())
    assert not res.ok
    step, idx, label = res.where
    assert step == 0 and idx[1] == NX - 1 and "sponge-right" in label and "last-tile-col" in label


def test_wrong_neighbour_in_the_last_partial_tile_row_is_caught(case):
    """Row 66 (in the last tile row, 64..69) reads its z+1 neighbour from z+2: fails, in row 66."""
    z0 = 66

    def lap_bad(u):
        w = fo.laplacian(u)
        w[z0] += np.float32(fo.COEF[1]) * (u[z0 + 2] - u[z0 + 1])
        return w
    res = fc.check_sweep("neighbour offset", sweep32(case, lap=lap_bad), case["ref"], K2, DEC)
    print("\n" + res.report())
    assert not res.ok
    step, idx, label = res.where
    assert idx[0] == z0 and "last-tile-row(partial)" in label


def test_dropped_injection_in_a_tile_halo_is_caught(case):
    """The source at (30, 129), within the 4-cell halo of the tile corner (32, 128), skips its injection at step 4:
    fails at that point and step."""
    c = case
    s = int(np.nonzero((c["src"][:, 0] == 30) & (c["src"][:, 1] == 129))[0][0])
    res = fc.check_sweep("dropped injection", sweep32(c, drop=(4, s)), c["ref"], K2, DEC)
    print("\n" + res.report())
    assert not res.ok
    step, idx, label = res.where
    assert step == 4 and tuple(int(i) for i in idx) == (30, 129)
    assert DEC.tile_of(idx) == (0, 1)


def test_decomposition_and_labels():
    """pick_tile's choice at the benchmark size on 148 SMs, the tb2 defaults by size, region labels."""
    d = fc.Decomp.for_plan((1000, 3000), 148, 40)
    assert (d.kind, d.tz) == ("tile", 56)
    assert d.label((999, 3000)) == "pad"
    assert d.label((960, 2999)) == "sponge-bottom+last-tile-row(partial)+sponge-right+last-tile-col(partial)"
    assert d.label((500, 1500)) == "interior" and d.tile_of((500, 1500)) == (8, 11)
    d = fc.Decomp.for_plan((751, 2301), 148, 40)
    assert (d.kind, d.tz, d.tx) == ("tb2", 24, 120) and d.label((750, 2300)).count("(partial)") == 2
    assert fc.Decomp.for_plan((2503, 3001), 148, 40).tz == 32
    d = fc.Decomp.for_plan((64, 512, 512), 148, 16, by=14)
    assert d.ty == 14 and "last-tile-y(partial)" in d.label((30, 511, 30))
    m = d.masks()
    assert m["interior"].sum() > 0 and not (m["interior"] & m["sponge-back"]).any()


def test_region_table():
    rng = np.random.default_rng(0)
    ref = rng.standard_normal((40, 6))
    got = ref * (1 + 1e-6)
    sel = fc.trace_selections({"a": [0, 1], "b": [5]}, 40, [(0, 20), (20, 40)])
    rows = fc.region_table(got, ref, ref, sel)
    assert len(rows) == 4 and all(abs(r[1] - 1e-6) < 1e-9 and r[2] == 0.0 for r in rows)
    assert abs(sum(r[3] ** 2 for r in rows) - 0.5) < 0.2
    print("\n" + fc.format_table("demo", rows))
