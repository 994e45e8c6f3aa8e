"""Born modelling (J dv) and Gauss-Newton Hessian-vector products (J^T J dv) on the GPU (spec B5, tests/born_reference.py).

Parity is against the float64 self-oracle (the reference has no propagator, SURVEY 0): Born traces rel-L2 <= 1e-5 and
Hessian products rel-L2 <= 1e-4, the north_star tolerances of traces and gradients.  The adjoint test ties the new STEP_BORN
kernels to the existing gradient kernels, which share no code path with them.

Measured worst cases on a B200 (each test prints its own): Born vs oracle 3.0e-6 (2-D, 33x129) and 6.9e-7 (3-D);
Gauss-Newton vs oracle 4.9e-6 (2-D) and 1.3e-6 (3-D); adjoint test 2.7e-6 (2-D 500x1500) and 1.8e-7 (3-D); directional
derivative 1.8e-4; born(2 dv) vs 2 born(dv) 3.7e-7 (bound 1e-6, see that test)."""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fd_oracle as fo  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))     # the B5 reference lives beside the tests
import born_reference as br  # noqa: E402


@pytest.fixture(scope="module")
def ac():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from full_waveform_inversion_b200 import acoustic
    return acoustic


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def blobs(shape, centres, width, amps=None):
    """Sum of Gaussian blobs (peak ~1 m/s each) -> float32-exact float64 grid."""
    grids = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    dv = np.zeros(shape)
    for i, c in enumerate(centres):
        r2 = sum((g - ci) ** 2 for g, ci in zip(grids, c))
        dv += (1.0 if amps is None else amps[i]) * np.exp(-r2 / (2.0 * width ** 2))
    return dv.astype(np.float32).astype(np.float64)


def case2d(nz, nx, nt, seed=0, nsrc=1, f0=18.0):
    """test_fd2d_gpu's geometry, plus dv: a blob inside, one inside the sponge strip, one on the last (partial) tile."""
    rng = np.random.default_rng(seed)
    v = fo.layered_model((nz, nx), 1600.0, 3200.0, 4) + 60.0 * rng.standard_normal((nz, nx))
    v = v.astype(np.float32).astype(np.float64)
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 2)
    src = [(6 + 3 * i, nx // 3 + 11 * i) for i in range(nsrc)]
    rec = [(5, x) for x in range(2, nx - 2, 3)] + [(nz - 7, nx // 2)]
    wav = np.stack([fo.ricker(nt, dt, f0 * (1 + 0.2 * i)) for i in range(nsrc)], 1).astype(np.float32).astype(np.float64)
    dv = blobs((nz, nx), [(nz // 2, nx // 2), (3, 2 * nx // 3), (nz - 2, nx - 3)], 3.0, [1.0, -0.7, 0.8])
    return v, h, dt, src, rec, wav, dv


def case3d(shape, nt, seed=0):
    """test_fd3d_gpu's geometry, plus blob perturbations (one in the sponge, one at the far corner)."""
    rng = np.random.default_rng(seed)
    nz, ny, nx = shape
    v = fo.layered_model(shape, 1700.0, 3000.0, 3) + 50.0 * rng.standard_normal(shape)
    v = v.astype(np.float32).astype(np.float64)
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 3)
    src = [(5, ny // 2, nx // 3), (7, ny // 3, nx // 2)]
    rec = [(4, y, x) for y in range(2, ny - 2, 5) for x in range(2, nx - 2, 7)] + [(nz - 6, ny // 2, nx // 2)]
    wav = np.stack([fo.ricker(nt, dt, 22.0), 0.6 * fo.ricker(nt, dt, 17.0)], 1).astype(np.float32).astype(np.float64)
    dv = blobs(shape, [(nz // 2, ny // 2, nx // 2), (2, 2, nx // 4), (nz - 2, ny - 2, nx - 2)], 2.5, [1.0, 0.6, -0.8])
    return v, h, dt, src, rec, wav, dv


def plan(ac, shape, h, dt, v, src, rec, nabs, **kw):
    p = ac.Propagator(shape, h, dt, nabs=nabs, **kw)
    p.set_model(v)
    p.set_geometry(src, rec)
    return p


def plane_bytes(shape):
    return int(np.prod(shape[:-1])) * ((shape[-1] + 31) // 32 * 32) * 4


CASES_2D = [(70, 150, 260, 1), (33, 129, 150, 2), (130, 64, 200, 1), (40, 300, 120, 3)]
PLANS_2D = [dict(), dict(tile=(32, 4)), dict(tb2=24), dict(tb2=32), dict(graphs=False)]
_oracle = {}


def born_oracle_2d(nz, nx, nt, nsrc):
    key = (nz, nx, nt, nsrc)
    if key not in _oracle:
        v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=nz, nsrc=nsrc)
        _oracle[key] = br.born(fo.Problem(v, h, dt, src, rec, nabs=12), wav, dv)[0]
    return _oracle[key]


# ------------------------------------------------------------------------------------------------ 1. Born vs oracle
@pytest.mark.parametrize("kw", PLANS_2D)
@pytest.mark.parametrize("nz,nx,nt,nsrc", CASES_2D)
def test_born_traces_vs_oracle_2d(ac, nz, nx, nt, nsrc, kw):
    """J dv vs born_reference.born (float64), rel-L2 <= 1e-5; the background traces the call returns are forward()'s bit for bit."""
    v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=nz, nsrc=nsrc)
    want = born_oracle_2d(nz, nx, nt, nsrc)
    p = plan(ac, (nz, nx), h, dt, v, src, rec, 12, **kw)
    dtr, tr = p.born(wav, dv, want_traces=True)
    e = rel_l2(dtr.cpu().numpy(), want)
    print("\n[born 2-D %dx%d nt=%d %s] rel-L2 vs float64 oracle %.3e" % (nz, nx, nt, kw, e))
    assert e <= 1e-5
    assert np.array_equal(tr.cpu().numpy(), p.forward(wav).cpu().numpy())
    p.close()


@pytest.mark.parametrize("shape,nt", [((40, 37, 150), 90), ((18, 50, 131), 60)])
def test_born_traces_vs_oracle_3d(ac, shape, nt):
    v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=shape[0])
    want = br.born(fo.Problem(v, h, dt, src, rec, nabs=8), wav, dv)[0]
    p = plan(ac, shape, h, dt, v, src, rec, 8)
    dtr, tr = p.born(wav, dv, want_traces=True)
    e = rel_l2(dtr.cpu().numpy(), want)
    print("\n[born 3-D %s nt=%d] rel-L2 vs float64 oracle %.3e" % (shape, nt, e))
    assert e <= 1e-5
    assert np.array_equal(tr.cpu().numpy(), p.forward(wav).cpu().numpy())
    p.close()


# ------------------------------------------------------------------------------------------------ 2. Gauss-Newton vs oracle
@pytest.mark.parametrize("kw", [dict(), dict(tile=(32, 4)), dict(tb2=24)])
def test_gauss_newton_vs_oracle_2d(ac, kw):
    nz, nx, nt = 70, 150, 260
    v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=5)
    want = br.gauss_newton(fo.Problem(v, h, dt, src, rec, nabs=12), wav, dv)
    p = plan(ac, (nz, nx), h, dt, v, src, rec, 12, **kw)
    hv, dtr = p.gauss_newton(wav, dv, want_dtraces=True)
    e = rel_l2(hv.cpu().numpy(), want)
    print("\n[gauss-newton 2-D %s] rel-L2 vs float64 oracle %.3e" % (kw, e))
    assert e <= 1e-4
    assert np.array_equal(dtr.cpu().numpy(), p.born(wav, dv)[0].cpu().numpy())    # the same J dv as born()
    hv2, _ = p.gauss_newton(wav, dv, hv=hv.clone())                                 # accumulates
    assert rel_l2(hv2.cpu().numpy(), 2 * want) <= 1e-4
    p.close()


def test_gauss_newton_vs_oracle_3d(ac):
    shape, nt = (36, 30, 140), 70
    v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=5)
    want = br.gauss_newton(fo.Problem(v, h, dt, src, rec, nabs=8), wav, dv)
    p = plan(ac, shape, h, dt, v, src, rec, 8)
    hv, _ = p.gauss_newton(wav, dv)
    e = rel_l2(hv.cpu().numpy(), want)
    print("\n[gauss-newton 3-D %s] rel-L2 vs float64 oracle %.3e" % (shape, e))
    assert e <= 1e-4
    p.set_memory_limit(40 * plane_bytes(shape))          # 70 snapshots do not fit -> checkpointed
    hv_c, _ = p.gauss_newton(wav, dv)
    assert rel_l2(hv_c.cpu().numpy(), hv.cpu().numpy()) <= 1e-6
    p.close()


# ------------------------------------------------------------------------------------------------ 3. adjoint test
def _dot_test(ac, shape, v, h, dt, src, rec, wav, dv, nabs):
    """<J dv, syn> vs <dv, J^T syn>; J^T syn is the existing gradient with obs = 0 (residual = synthetics)."""
    import torch
    p = plan(ac, shape, h, dt, v, src, rec, nabs)
    dtr, tr = p.born(wav, dv, want_traces=True)
    _, g, _ = p.gradient(wav, torch.zeros_like(tr))
    p.close()
    lhs = float(np.sum(dtr.cpu().numpy().astype(np.float64) * tr.cpu().numpy().astype(np.float64)))
    rhs = float(np.sum(dv * g.cpu().numpy().astype(np.float64)))
    return lhs, rhs


def test_born_is_the_adjoint_of_the_gradient_2d_500x1500(ac):
    nz, nx, nt = 500, 1500, 700
    rng = np.random.default_rng(5)
    v = (fo.layered_model((nz, nx), 1600.0, 3800.0, 5) + 40.0 * rng.standard_normal((nz, nx))).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(float(v.max()), h, 2)
    src = [(5, 300), (40, 700)]
    rec = [(4, x) for x in range(10, nx - 10, 7)] + [(300, 600), (499, 1499)]
    wav = np.stack([fo.ricker(nt, dt, 12.0), fo.ricker(nt, dt, 15.0)], 1).astype(np.float32)
    dv = blobs((nz, nx), [(60, 400), (150, 900), (20, 1200), (nz - 3, nx - 5)], 12.0, [1.0, -0.8, 0.6, 0.5])
    lhs, rhs = _dot_test(ac, (nz, nx), v, h, dt, src, rec, wav, dv, 30)
    print("\n[born adjoint 2-D 500x1500 nt=700] <J dv, d> = %.9e  <dv, J^T d> = %.9e  rel diff %.2e" % (lhs, rhs, abs(lhs - rhs) / abs(lhs)))
    assert abs(lhs - rhs) <= 1e-5 * abs(lhs)


def test_born_is_the_adjoint_of_the_gradient_3d(ac):
    shape, nt = (64, 64, 128), 150
    v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=2)
    lhs, rhs = _dot_test(ac, shape, v, h, dt, src, rec, wav, dv, 10)
    print("\n[born adjoint 3-D %s nt=%d] <J dv, d> = %.9e  <dv, J^T d> = %.9e  rel diff %.2e" % (shape, nt, lhs, rhs, abs(lhs - rhs) / abs(lhs)))
    assert abs(lhs - rhs) <= 1e-5 * abs(lhs)


# ------------------------------------------------------------------------------------------------ 4. directional derivative
def test_born_is_the_directional_derivative_at_500x1500(ac):
    """J dv vs (forward(v + e dv) - forward(v - e dv)) / 2e through the CUDA path, with test_fd_scale_gpu's choice: dv =
    the box-smoothed gradient scaled to 1 m/s, e = 2 m/s.  Tolerance rel-L2 1e-3."""
    from scipy.ndimage import uniform_filter
    nz, nx, nt = 500, 1500, 600
    v = fo.layered_model((nz, nx), 1600.0, 3800.0, 5).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(3900.0, h, 2)
    wav = fo.ricker(nt, dt, 12.0).astype(np.float32)
    src, rec = [(4, 500)], [(4, x) for x in range(0, nx, 2)]
    p = ac.Propagator2D((nz, nx), h, dt, nabs=30)
    p.set_geometry(src, rec)
    p.set_model(v * np.float32(1.03))
    obs = p.forward(wav).clone()
    p.set_model(v)
    _, g, _ = p.gradient(wav, obs)
    dv = uniform_filter(g.cpu().numpy().astype(np.float64), 9)
    dv = (dv / np.abs(dv).max()).astype(np.float32)
    dtr = p.born(wav, dv)[0].cpu().numpy().astype(np.float64)
    eps = 2.0
    tr = []
    for s in (+1.0, -1.0):
        p.set_model(v + np.float32(s * eps) * dv)
        tr.append(p.forward(wav).cpu().numpy().astype(np.float64))
    p.close()
    fd = (tr[0] - tr[1]) / (2 * eps)
    e = rel_l2(dtr, fd)
    print("\n[born directional derivative 500x1500 nt=600] rel-L2 vs centred difference %.3e" % e)
    assert e <= 1e-3


# ------------------------------------------------------------------------------------------------ 5. exact properties
@pytest.mark.parametrize("kw", [dict(tile=(32, 4)), dict(tb2=24), "3d"])
def test_segment_length_changes_no_bit(ac, kw):
    """Default segment, S = 1 and S = 7 (forced through the memory limit): bit-identical Born and background traces, and
    the same final background wavefields u_nt, u_{nt-1}."""
    if kw == "3d":
        shape, nt = (36, 30, 140), 45
        v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=4)
        kw = {}
    else:
        shape, nt = (70, 150), 75
        v, h, dt, src, rec, wav, dv = case2d(*shape, nt, seed=4)
    p = plan(ac, shape, h, dt, v, src, rec, 8, **kw)
    ref, ref_tr = [t.cpu().numpy() for t in p.born(wav, dv, want_traces=True)]
    ref_u = [p.wavefield(k).cpu().numpy() for k in (0, 1)]
    assert np.abs(ref).max() > 0
    for planes in (1, 7):
        p.set_memory_limit(planes * plane_bytes(shape))
        got, got_tr = [t.cpu().numpy() for t in p.born(wav, dv, want_traces=True)]
        assert np.array_equal(got, ref), planes
        assert np.array_equal(got_tr, ref_tr), planes
        for k in (0, 1):
            assert np.array_equal(p.wavefield(k).cpu().numpy(), ref_u[k]), (planes, k)
    p.set_memory_limit(plane_bytes(shape) - 4)          # not even one snapshot plane
    with pytest.raises(ValueError):
        p.born(wav, dv)
    p.close()


def test_zero_and_scaled_perturbations(ac):
    """born(0) is exactly 0.  born(2 dv) vs 2 born(dv): the Born sweep's precursor passes through the denormal range, where
    scaling by 2 is inexact (test_fd2d_gpu's linearity check of the forward notes the same), so this is checked to 1e-6
    rel-L2 rather than bit for bit; the number of samples that differ is printed."""
    shape, nt = (70, 150), 260
    v, h, dt, src, rec, wav, dv = case2d(*shape, nt, seed=6)
    p = plan(ac, shape, h, dt, v, src, rec, 12, tile=(32, 4))
    assert float(p.born(wav, np.zeros(shape, np.float32))[0].abs().max()) == 0.0
    b1 = p.born(wav, dv)[0].cpu().numpy()
    b2 = p.born(wav, 2.0 * dv)[0].cpu().numpy()
    print("\n[born 2 dv vs 2 born(dv)] %d of %d samples differ, rel-L2 %.2e" % (int(np.sum(b2 != 2 * b1)), b1.size, rel_l2(b2, 2 * b1)))
    assert rel_l2(b2, 2 * b1) <= 1e-6
    p.close()


@pytest.mark.parametrize("kw", [dict(tile=(32, 4)), dict(tb2=24)])
def test_checkpointed_gauss_newton_matches_stored(ac, kw):
    """Same bound as test_checkpointed_gradient_matches_stored: segments pair the deferred imaging differently."""
    nz, nx, nt = 50, 160, 210
    v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=9)
    p = plan(ac, (nz, nx), h, dt, v, src, rec, 10, **kw)
    h0, d0 = p.gauss_newton(wav, dv, want_dtraces=True)
    p.set_memory_limit(70 * plane_bytes((nz, nx)))      # < nt planes -> segments of 21 steps
    h1, d1 = p.gauss_newton(wav, dv, want_dtraces=True)
    assert np.array_equal(d1.cpu().numpy(), d0.cpu().numpy())
    assert rel_l2(h1.cpu().numpy(), h0.cpu().numpy()) <= 1e-6
    p.set_memory_limit(5 * plane_bytes((nz, nx)))
    with pytest.raises(ValueError):
        p.gauss_newton(wav, dv)
    p.close()


# ------------------------------------------------------------------------------------------------ 6. no interference
@pytest.mark.parametrize("kw", [dict(tile=(32, 4)), dict(tb2=24), "3d"])
def test_born_and_gauss_newton_leave_forward_and_gradient_unchanged(ac, kw):
    if kw == "3d":
        shape, nt = (36, 30, 140), 61
        v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=8)
        kw = {}
    else:
        shape, nt = (70, 150), 121
        v, h, dt, src, rec, wav, dv = case2d(*shape, nt, seed=8)
    fresh = plan(ac, shape, h, dt, v, src, rec, 8, **kw)
    tr0 = fresh.forward(wav).cpu().numpy()
    w0 = [fresh.wavefield(i).cpu().numpy() for i in (0, 1)]
    obs = 0.8 * tr0
    J0, g0, _ = fresh.gradient(wav, obs)
    fresh.close()
    p = plan(ac, shape, h, dt, v, src, rec, 8, **kw)
    p.born(wav, dv)
    for i in (0, 1):
        assert np.array_equal(p.wavefield(i).cpu().numpy(), w0[i])       # u_nt, u_{nt-1} of the background
    p.gauss_newton(wav, dv)
    assert np.array_equal(p.forward(wav).cpu().numpy(), tr0)
    J1, g1, _ = p.gradient(wav, obs)
    assert J1 == pytest.approx(J0, rel=1e-12)
    assert np.array_equal(g1.cpu().numpy(), g0.cpu().numpy())
    p.close()


# ------------------------------------------------------------------------------------------------ 7. launches, pad columns
@pytest.mark.parametrize("kw", [dict(tile=(32, 4)), dict(tb2=24)])
def test_launch_counts(ac, kw):
    """tile: a Born shot is 2 nt step launches (background + scattered); tb2: the background pairs steps inside each segment
    of S = min(nt, 128) steps (ceil(len / 2) launches per segment) + nt scattered one-step launches.  Gauss-Newton = the
    gradient's launches - 1 (no residual kernel) + nt (the scattered sweep)."""
    shape, nt = (70, 150), 75
    v, h, dt, src, rec, wav, dv = case2d(*shape, nt, seed=1)
    p = plan(ac, shape, h, dt, v, src, rec, 8, **kw)
    obs = p.forward(wav).clone()
    n0 = p.launch_count()
    p.born(wav, dv)
    nb = p.launch_count() - n0
    if "tile" in kw:
        assert nb == 2 * nt
    else:
        segs = [min(128, nt - s) for s in range(0, nt, 128)]
        assert nb == sum((s + 1) // 2 for s in segs) + nt
    n0 = p.launch_count()
    p.gradient(wav, obs)
    ng = p.launch_count() - n0
    n0 = p.launch_count()
    p.gauss_newton(wav, dv)
    assert p.launch_count() - n0 == ng - 1 + nt
    p.close()


@pytest.mark.parametrize("case", ["tile", "tile_checkpointed", "tb2", "3d", "3d_checkpointed"])
def test_pad_columns_stay_zero_after_born_and_gauss_newton(ac, case):
    import torch
    three_d = case.startswith("3d")
    shape = (36, 40, 150) if three_d else (90, 300)
    nt = 60
    v = fo.layered_model(shape, 1500.0, 3500.0, 3).astype(np.float32)
    dt = fo.stable_dt(3500.0, 10.0, 3 if three_d else 2)
    wav = fo.ricker(nt, dt, 15.0).astype(np.float32)
    kw = {} if three_d else ({"tb2": 24} if case.startswith("tb2") else {"tile": (32, 4)})
    if three_d:
        src, rec = [(5, 20, shape[2] - 2)], [(4, 10, shape[2] - 1), (6, 30, 3)]
    else:
        src, rec = [(5, shape[1] - 2)], [(4, shape[1] - 1), (6, 3)]
    dv = blobs(shape, [tuple(n // 2 for n in shape[:-1]) + (shape[-1] - 2,)], 4.0)
    p = plan(ac, shape, 10.0, dt, v, src, rec, 10, **kw)
    if case.endswith("checkpointed"):
        p.set_memory_limit(30 * plane_bytes(shape))
    p.born(wav, dv)
    p.gauss_newton(wav, dv)
    p.born(wav, dv)
    torch.cuda.synchronize()
    nx = shape[-1]
    for idx in range(8):
        pad = p.field_view(idx)[..., nx:]
        assert pad.numel() > 0
        assert float(pad.abs().max()) == 0.0, "buffer %d has non-zero pad columns" % idx
    p.close()


# ------------------------------------------------------------------------------------------------ 8. errors
def test_argument_errors(ac):
    shape, nt = (40, 140), 30
    v, h, dt, src, rec, wav, dv = case2d(*shape, nt, seed=2)
    p = ac.Propagator2D(shape, h, dt, nabs=6)
    p.set_geometry(src, rec)
    with pytest.raises(ValueError):
        p.born(wav, dv)                                   # model not set
    with pytest.raises(ValueError):
        p.gauss_newton(wav, dv)
    p.set_model(v)
    with pytest.raises(ValueError, match=r"\(40, 140\)"):
        p.born(wav, dv[:, :-1])                           # wrong dv shape: the message names the grid shape
    with pytest.raises(ValueError):
        p.gauss_newton(wav, dv.T)
    with pytest.raises(ValueError):
        p.born(wav[:0], dv)                               # nt < 1
    with pytest.raises(ValueError):
        p.gauss_newton(wav[:0], dv)
    import torch
    with pytest.raises(ValueError):
        p.born(wav, dv, out=torch.empty((nt, len(rec) + 1), device="cuda"))
    with pytest.raises(ValueError):
        p.gauss_newton(wav, dv, hv=torch.empty(shape, dtype=torch.float64, device="cuda"))
    p.close()


def test_slab_plans_refuse_born_and_gauss_newton(ac):
    """Plans connected as peer-memory slabs (here two plans of one process) reject both calls: the slab step ids assume
    the same launch sequence on every rank."""
    from full_waveform_inversion_b200 import _lib
    lib = _lib.load()
    shape, nt = (28, 20, 140), 20
    v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=1)
    up = ac.Propagator(shape, h, dt, nabs=4, graphs=False)
    dn = ac.Propagator(shape, h, dt, nabs=4, graphs=False)
    _lib.check(lib.fwi_fd_slab_connect_local(up._h, 0, 24, None, 0, dn._h))
    _lib.check(lib.fwi_fd_slab_connect_local(dn._h, 4, 28, up._h, 24, None))
    up.set_model(v)
    up.set_geometry([(5, 10, 40)], [(4, 10, 60)])
    with pytest.raises(ValueError, match="slab"):
        up.born(wav[:, :1], dv)
    with pytest.raises(ValueError, match="slab"):
        up.gauss_newton(wav[:, :1], dv)
    up.close()
    dn.close()


# ------------------------------------------------------------------------------------------------ 9. sharded product
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _gn_problem():
    nz, nx, nt = 90, 200, 160
    v = fo.layered_model((nz, nx), 1700.0, 3000.0, 4).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(3000.0, h, 2)
    wav = fo.ricker(nt, dt, 18.0).astype(np.float32)
    shots = [([(4, int(sx))], [(4, x) for x in range(0, nx, 2)]) for sx in np.linspace(15, nx - 15, 5)]
    dv = blobs((nz, nx), [(40, 60), (60, 150)], 6.0).astype(np.float32)
    return v, h, dt, wav, shots, dv


def _gn_worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from full_waveform_inversion_b200 import acoustic as ac
        v, h, dt, wav, shots, dv = _gn_problem()
        hv = ac.gauss_newton_product(torch.from_numpy(v).cuda(), h, dt, shots, wav, dv, nabs=12)
        if rank == 0:
            np.save(out, hv.cpu().numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_sharded_gauss_newton_product_two_ranks_one_gpu(ac, tmp_path):
    """Two processes on cuda:0 over gloo (as test_distributed_gpu.py): round-robin shots + one all-reduce equals the
    single-process sum over the same shots to 1e-6 (fp32 summation order)."""
    import torch
    import torch.multiprocessing as mp
    out = str(tmp_path / "hv.npy")
    mp.spawn(_gn_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = np.load(out)
    v, h, dt, wav, shots, dv = _gn_problem()
    want = ac.gauss_newton_product(torch.from_numpy(v).cuda(), h, dt, shots, wav, dv, nabs=12).cpu().numpy()
    assert np.abs(want).max() > 0
    assert np.linalg.norm(got - want) <= 1e-6 * np.linalg.norm(want)
