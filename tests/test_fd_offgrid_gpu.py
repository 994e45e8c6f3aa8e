"""Off-grid sources and receivers on the GPU (spec B7, tests/offgrid_reference.py), on every 2-D kernel family and in 3-D,
with the free surface off and on.

  * integral float positions are the integer API bit for bit (torch.equal): forward, gradient, Born, Gauss-Newton;
  * against the float64 B7 reference: traces and Born traces rel-L2 <= 1e-5, gradients and H dv <= 1e-4, with points within
    4 cells of every edge, 0 < z < 1, and a dense receiver line at fractional x whose taps share cells;
  * the plan's contract: checkpointing and the kernel family change no bit, pad columns stay zero, launch counts, errors,
    and the survey entry points.
"""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fd_oracle as fo  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))     # the B5 - B7 references live beside the tests
import offgrid_reference as ogr  # noqa: E402


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


def f32(x):
    return np.asarray(x, np.float32).astype(np.float64)


def case2d(nt=160, seed=0):
    """48 x 140: points within 4 cells of every edge, 0 < z < 1, a receiver in every column at fractional x."""
    nz, nx = 48, 140
    rng = np.random.default_rng(seed)
    v = f32(fo.layered_model((nz, nx), 1600.0, 3200.0, 4) + 60.0 * rng.standard_normal((nz, nx)))
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 2)
    src = np.array([(0.4, 30.5), (20.25, 1.6), (45.7, 137.2)])
    rec = np.array([(0.7, x + 0.5) for x in range(nx - 1)] + [(47.0, 3.3), (30.6, 139.0), (46.2, 0.8)])
    wav = f32(np.stack([fo.ricker(nt, dt, 18.0), 0.7 * fo.ricker(nt, dt, 22.0), -0.5 * fo.ricker(nt, dt, 15.0)], 1))
    dv = f32(sum(a * np.exp(-((np.arange(nz)[:, None] - cz) ** 2 + (np.arange(nx)[None] - cx) ** 2) / 18.0)
                 for a, cz, cx in [(1.0, nz // 2, nx // 2), (-0.7, 2, nx // 4), (0.8, nz - 3, nx - 4)]))
    return v, h, dt, src, rec, wav, dv


def case3d(nt=60, seed=0):
    shape = (20, 24, 131)
    rng = np.random.default_rng(seed)
    v = f32(fo.layered_model(shape, 1700.0, 3000.0, 3) + 50.0 * rng.standard_normal(shape))
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 3)
    src = np.array([(0.6, 12.3, 60.5), (17.5, 2.2, 128.7)])
    rec = np.array([(0.8, y + 0.5, x + 0.25) for y in (0, 11, 22) for x in range(0, 130, 3)] + [(19.0, 23.0, 130.0)])
    wav = f32(np.stack([fo.ricker(nt, dt, 22.0), 0.6 * fo.ricker(nt, dt, 17.0)], 1))
    g = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    dv = f32(np.exp(-sum((gi - c) ** 2 for gi, c in zip(g, (10, 12, 65))) / 12.0)
             - 0.6 * np.exp(-sum((gi - c) ** 2 for gi, c in zip(g, (2, 3, 30))) / 12.0))
    return shape, v, h, dt, src, rec, wav, dv


def plan(ac, shape, h, dt, v, src, rec, nabs, **kw):
    p = ac.Propagator(shape, h, dt, nabs=nabs, **kw)
    p.set_model(v)
    p.set_geometry(src, rec)
    return p


PLANS_2D = [dict(), dict(tile=(32, 4)), dict(tile=(28, 4)), dict(tile=(42, 6)), dict(tile=(56, 8)), dict(tb2=24),
            dict(tb2=32), dict(tile=(32, 4), graphs=False)]
_ref = {}


def reference(ndim, fs):
    """Float64 B7 results: traces, gradient (obs = 0.8 x the reference traces), Born traces, H dv."""
    if (ndim, fs) not in _ref:
        if ndim == 2:
            v, h, dt, src, rec, wav, dv = case2d()
            nabs = 10
        else:
            _, v, h, dt, src, rec, wav, dv = case3d()
            nabs = 5
        p = ogr.Problem(v, h, dt, src, rec, nabs=nabs, free_surface=fs)
        tr = p.forward(wav)
        obs = f32(0.8 * tr)
        J, g, _ = p.misfit_and_gradient(wav, obs)
        _ref[(ndim, fs)] = dict(tr=tr, obs=obs, J=J, g=g, born=p.born(wav, dv)[0], hv=p.gauss_newton(wav, dv), nabs=nabs)
    return _ref[(ndim, fs)]


def check_vs_reference(p, wav, dv, ref, tag):
    tr = p.forward(wav).cpu().numpy()
    J, g, tr2 = p.gradient(wav, ref["obs"], want_traces=True)
    e = [rel_l2(tr, ref["tr"]), rel_l2(g.cpu().numpy(), ref["g"]), rel_l2(p.born(wav, dv)[0].cpu().numpy(), ref["born"]),
         rel_l2(p.gauss_newton(wav, dv)[0].cpu().numpy(), ref["hv"])]
    print("\n[off-grid %s] rel-L2 traces / gradient / born / gauss-newton: %.2e %.2e %.2e %.2e, misfit %.2e"
          % (tag, *e, abs(J - ref["J"]) / ref["J"]))
    assert e[0] <= 1e-5 and e[1] <= 1e-4 and e[2] <= 1e-5 and e[3] <= 1e-4
    assert abs(J - ref["J"]) <= 1e-5 * ref["J"] and np.array_equal(tr2.cpu().numpy(), tr)


# ------------------------------------------------------------------------------------------------ 1. vs the B7 reference
@pytest.mark.parametrize("fs", [False, True])
@pytest.mark.parametrize("kw", PLANS_2D)
def test_vs_reference_2d(ac, kw, fs):
    v, h, dt, src, rec, wav, dv = case2d()
    ref = reference(2, fs)
    p = plan(ac, v.shape, h, dt, v, src, rec, ref["nabs"], free_surface=fs, **kw)
    check_vs_reference(p, wav, dv, ref, "2-D %s fs=%d" % (kw, fs))
    p.close()


@pytest.mark.parametrize("fs", [False, True])
@pytest.mark.parametrize("by", ["16", "14"])
def test_vs_reference_3d(ac, by, fs, monkeypatch):
    monkeypatch.setenv("FWI_FD3D_BY", by)
    shape, v, h, dt, src, rec, wav, dv = case3d()
    ref = reference(3, fs)
    p = plan(ac, shape, h, dt, v, src, rec, ref["nabs"], free_surface=fs)
    check_vs_reference(p, wav, dv, ref, "3-D by=%s fs=%d" % (by, fs))
    p.close()


# ------------------------------------------------------------------------------------------------ 2. integral positions
def integral_case(ndim):
    if ndim == 2:
        v, h, dt, _, _, wav, dv = case2d(nt=121)
        src = [(1, 30), (20, 2), (46, 137)]
        rec = [(1, x) for x in range(0, 140, 2)] + [(47, 3), (30, 139)]
        return v.shape, v, h, dt, src, rec, wav, dv, 10
    shape, v, h, dt, _, _, wav, dv = case3d(nt=41)
    return shape, v, h, dt, [(1, 12, 60), (17, 2, 128)], [(1, y, x) for y in (0, 11, 23) for x in range(0, 131, 4)], wav, dv, 5


def run_all(p, wav, dv, obs):
    import torch
    tr = p.forward(wav).clone()
    J, g, gtr = p.gradient(wav, obs, want_traces=True)
    b, btr = p.born(wav, dv, want_traces=True)
    hv, hdtr = p.gauss_newton(wav, dv, want_dtraces=True)
    torch.cuda.synchronize()
    return J, [tr, g, gtr, b, btr, hv, hdtr]


@pytest.mark.parametrize("fs", [False, True])
@pytest.mark.parametrize("kw", [dict(), dict(tile=(32, 4)), dict(tile=(42, 6)), dict(tb2=24), dict(tb2=32), "3d"])
def test_integral_positions_are_the_integer_api(ac, kw, fs):
    """Float positions with integral values give the integer API's bits; set_geometry with ints then clears them."""
    import torch
    shape, v, h, dt, src, rec, wav, dv, nabs = integral_case(3 if kw == "3d" else 2)
    kw = {} if kw == "3d" else kw
    p = plan(ac, shape, h, dt, v, src, rec, nabs, free_surface=fs, **kw)
    obs = 0.8 * p.forward(wav).cpu().numpy()
    J0, want = run_all(p, wav, dv, obs)
    p.set_geometry(np.asarray(src, np.float64), np.asarray(rec, np.float64))
    J1, got = run_all(p, wav, dv, obs)
    assert J1 == pytest.approx(J0, rel=1e-12)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    p.set_geometry(src, rec)
    J2, again = run_all(p, wav, dv, obs)
    assert all(torch.equal(a, b) for a, b in zip(again, want))
    p.close()


# ------------------------------------------------------------------------------------------------ 3. the plan's contract
@pytest.mark.parametrize("fs", [False, True])
def test_checkpointing_and_family_change_no_bit(ac, fs):
    """nt = 200 with a 70-plane limit: segments of 20 steps, which pair the adjoint steps as the stored sweep does."""
    import torch
    v, h, dt, src, rec, wav, dv = case2d(nt=200, seed=3)
    nz, nx = v.shape
    out = {}
    for name, kw in (("tile", dict(tile=(32, 4))), ("tb2", dict(tb2=24))):
        p = plan(ac, v.shape, h, dt, v, src, rec, 10, free_surface=fs, **kw)
        obs = 0.7 * p.forward(wav).cpu().numpy()
        J0, res = run_all(p, wav, dv, obs)
        p.set_memory_limit(70 * nz * 160 * 4)
        g1 = p.gradient(wav, obs)[1]
        hv1 = p.gauss_newton(wav, dv)[0]
        assert torch.equal(g1, res[1]) and torch.equal(hv1, res[5]), name
        for i in range(8):
            assert not p.field_view(i)[:, nx:].any()
        out[name] = res
        p.close()
    assert all(torch.equal(a, b) for a, b in zip(out["tile"], out["tb2"]))


@pytest.mark.parametrize("kw", [dict(tile=(32, 4)), dict(tb2=24), "3d"])
def test_launch_counts(ac, kw):
    """Per shot on top of the integer geometry's launches: forward 2 (wavelet spread, trace gather), gradient 3 (wavelet
    spread, synthetics gather, residual spread), Born 2 (+1 for the background traces), Gauss-Newton 3."""
    if kw == "3d":
        shape, v, h, dt, src, rec, wav, dv = case3d(nt=21)
        kw, nabs = {}, 5
    else:
        v, h, dt, src, rec, wav, dv = case2d(nt=75)
        shape, nabs = v.shape, 10
    counts = []
    for pts in ((np.round(src).astype(int), np.round(rec).astype(int)), (src, rec)):
        p = plan(ac, shape, h, dt, v, pts[0], pts[1], nabs, **kw)
        obs = np.zeros((wav.shape[0], len(rec)), np.float32)
        c = []
        for call in (lambda: p.forward(wav), lambda: p.gradient(wav, obs), lambda: p.born(wav, dv),
                     lambda: p.born(wav, dv, want_traces=True), lambda: p.gauss_newton(wav, dv)):
            n0 = p.launch_count()
            call()
            c.append(p.launch_count() - n0)
        counts.append(c)
        p.close()
    assert [b - a for a, b in zip(*counts)] == [2, 3, 2, 3, 3], counts


def test_errors(ac):
    from full_waveform_inversion_b200 import _lib
    v, h, dt, src, rec, wav, _ = case2d(nt=20)
    p = plan(ac, v.shape, h, dt, v, src, rec, 10)
    for bad, what in (((np.nan, 5.0), "not finite"), ((3.0, np.inf), "not finite"), ((-0.5, 5.0), "outside"),
                      ((47.01, 5.0), "outside"), ((5.0, 139.5), "outside")):
        with pytest.raises(ValueError, match=r"receiver 1 at .*%s" % what):
            p.set_geometry(src, [(3.5, 4.5), bad])
    with pytest.raises(ValueError, match="source 0 at"):
        p.set_geometry([(2.5, -1.0)], rec)
    p.close()
    p = plan(ac, v.shape, h, dt, v, src, rec, 10, free_surface=True)
    for z in (0.0, -0.0):
        with pytest.raises(ValueError, match=r"source 2 at \(z=-?0, y=0, x=7.5\) lies on the free surface"):
            p.set_geometry([(1.5, 3.0), (0.5, 4.0), (z, 7.5)], rec)
    p.set_geometry([(0.01, 3.0)], [(0.99, 7.0)])                      # 0 < z < 1 is allowed
    p.close()
    # caller-driven single steps take the integer geometry only
    p = plan(ac, v.shape, h, dt, v, src, rec, 10)
    w = ac._dev_f32(wav, p.torch_device)
    with pytest.raises(ValueError, match="off-grid positions"):
        p.step(0, 0, w.data_ptr())
    p.set_geometry(np.round(src).astype(int), np.round(rec).astype(int))
    p.step(0, 0, w.data_ptr())
    p.close()
    # peer-memory slabs
    lib = _lib.load()
    shape = (28, 12, 140)
    up = ac.Propagator(shape, 10.0, 1e-3, nabs=3)
    dn = ac.Propagator(shape, 10.0, 1e-3, nabs=3)
    _lib.check(lib.fwi_fd_slab_connect_local(dn._h, 4, 28, up._h, 24, None))
    with pytest.raises(ValueError, match="peer-memory slab"):
        dn.set_geometry([(10.5, 5.0, 7.0)], [(12.0, 6.0, 7.25)])
    dn.set_geometry([(10, 5, 7)], [(12, 6, 7)])
    up.close()
    dn.close()


def test_survey_entry_points_accept_float_shots(ac):
    import torch
    v, h, dt, src, rec, wav, dv = case2d(nt=100, seed=5)
    shots = [(src[:1], rec), (src[1:], rec[::2])]
    p = ac.Propagator(v.shape, h, dt, nabs=10, free_surface=True)
    p.set_model(v)
    w = wav[:, 0]
    want_tr, want_born = [], []
    want_hv = torch.zeros(v.shape, device=p.torch_device)
    want_g = torch.zeros(v.shape, device=p.torch_device)
    for s, r in shots:
        p.set_geometry(s, r)
        want_tr.append(p.forward(w).clone())
        want_born.append(p.born(w, dv)[0])
        p.gauss_newton(w, dv, hv=want_hv)
    observed = [0.8 * t for t in want_tr]
    J_want = 0.0
    for (s, r), o in zip(shots, observed):
        p.set_geometry(s, r)
        J_want += p.gradient(w, o, grad=want_g)[0]
    kw = dict(nabs=10, free_surface=True)
    assert all(torch.equal(a, b) for a, b in zip(ac.forward_model(v, h, dt, shots, w, **kw), want_tr))
    assert all(torch.equal(a, b) for a, b in zip(ac.born_model(v, h, dt, shots, w, dv, **kw), want_born))
    assert torch.equal(ac.gauss_newton_product(v, h, dt, shots, w, dv, allreduce=False, **kw), want_hv)
    J, g = ac.gradient(v, h, dt, shots, w, observed, allreduce=False, **kw)
    assert J == pytest.approx(J_want, rel=1e-12) and torch.equal(g, want_g)
    _, hist = ac.fwi(v, h, dt, shots, w, observed, 1, 1400.0, 3400.0, **kw)
    assert hist[0] == pytest.approx(J_want, rel=1e-12)
    p.close()
