"""Track B (2-D) parity on the GPU: CUDA path through the C ABI vs the SELF-oracle oracle/fd_oracle.py.
The reference has no propagator (SURVEY 0) - these are not reference-parity claims.

Tolerances (north_star): traces rel-L2 <= 1e-5, gradient rel-L2 <= 1e-4, stated per test.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fd_oracle as fo  # noqa: E402


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


def _case(nz, nx, nt, seed=0, nsrc=1, f0=18.0):
    rng = np.random.default_rng(seed)
    v = fo.layered_model((nz, nx), 1600.0, 3200.0, 4) + 60.0 * rng.standard_normal((nz, nx))
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 2)
    src = [(6 + 3 * i, nx // 3 + 11 * i) for i in range(nsrc)]
    rec = [(5, x) for x in range(2, nx - 2, 3)] + [(nz - 7, nx // 2)]
    wav = np.stack([fo.ricker(nt, dt, f0 * (1 + 0.2 * i)) for i in range(nsrc)], 1)
    return v.astype(np.float32).astype(np.float64), h, dt, src, rec, wav.astype(np.float32).astype(np.float64)


# the default kernel depends on the grid size (two-steps-per-pass for small and for larger-than-L2 grids, the one-step tile
# kernel in between, which is what the bench workload runs): the parity tests pin both
KERNELS = [dict(), dict(tile=(32, 4))]


@pytest.mark.parametrize("kw", KERNELS)
@pytest.mark.parametrize("nz,nx,nt,nsrc", [(70, 150, 260, 1), (33, 129, 150, 2), (130, 64, 200, 1), (40, 300, 120, 3)])
def test_forward_traces_and_wavefield(ac, nz, nx, nt, nsrc, kw):
    v, h, dt, src, rec, wav = _case(nz, nx, nt, seed=nz, nsrc=nsrc)
    p = fo.Problem(v, h, dt, src, rec, nabs=12, alpha=0.3)
    want, _, (cur, old) = p.forward(wav, return_state=True)
    prop = ac.Propagator2D((nz, nx), h, dt, nabs=12, alpha=0.3, **kw)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    got = prop.forward(wav).cpu().numpy()
    assert got.shape == want.shape
    assert rel_l2(got, want) <= 1e-5                      # traces tolerance of the north_star
    assert rel_l2(prop.wavefield(0).cpu().numpy(), cur) <= 1e-5
    assert rel_l2(prop.wavefield(1).cpu().numpy(), old) <= 1e-5
    # source placement / receiver indexing are integer-exact: first non-zero sample appears at the same step
    nzw = np.nonzero(np.abs(want).max(1) > 0)[0][0]
    nzg = np.nonzero(np.abs(got).max(1) > 0)[0][0]
    assert nzw == nzg
    prop.close()


@pytest.mark.parametrize("kind,cfg", [("tile", (32, 4)), ("graphs", False), ("tb2", 32), ("tb2", 24),
                                      ("tile", (28, 4)), ("tile", (42, 6)), ("tile", (56, 8))])
def test_kernel_variants_agree(ac, kind, cfg):
    """Every step-kernel variant (one-tile-per-CTA shapes, two-steps-per-pass, plain launches) gives the oracle's traces and gradient."""
    v, h, dt, src, rec, wav = _case(75, 300, 150, seed=3)
    obs = fo.Problem(v * 1.03, h, dt, src, rec, nabs=10).forward(wav)
    J_want, g_want, tr_want = fo.Problem(v, h, dt, src, rec, nabs=10).misfit_and_gradient(wav, obs)
    prop = ac.Propagator2D((75, 300), h, dt, nabs=10, **{kind: cfg})
    prop.set_model(v)
    prop.set_geometry(src, rec)
    assert rel_l2(prop.forward(wav).cpu().numpy(), tr_want) <= 1e-5
    J, g, _ = prop.gradient(wav, obs)
    assert abs(J - J_want) <= 1e-4 * J_want
    assert rel_l2(g.cpu().numpy(), g_want) <= 1e-4
    prop.close()


@pytest.mark.parametrize("kw", KERNELS)
@pytest.mark.parametrize("nz,nx,nt", [(60, 140, 220), (45, 131, 160)])
def test_gradient_vs_self_oracle(ac, nz, nx, nt, kw):
    v, h, dt, src, rec, wav = _case(nz, nx, nt, seed=7)
    obs = fo.Problem(v * 1.04, h, dt, src, rec, nabs=10).forward(wav).astype(np.float32).astype(np.float64)
    J_want, g_want, tr_want = fo.Problem(v, h, dt, src, rec, nabs=10).misfit_and_gradient(wav, obs)
    prop = ac.Propagator2D((nz, nx), h, dt, nabs=10, **kw)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    J, g, tr = prop.gradient(wav, obs, want_traces=True)
    assert rel_l2(tr.cpu().numpy(), tr_want) <= 1e-5
    assert abs(J - J_want) <= 1e-4 * J_want
    assert rel_l2(g.cpu().numpy(), g_want) <= 1e-4         # gradient tolerance of the north_star
    # accumulation into an existing gradient
    J2, g2, _ = prop.gradient(wav, obs, grad=g.clone())
    assert rel_l2(g2.cpu().numpy(), 2 * g_want) <= 1e-4
    prop.close()


@pytest.mark.parametrize("kw", KERNELS)
def test_checkpointed_gradient_matches_stored(ac, kw):
    """Two-level checkpointing recomputes w_n exactly: same gradient as holding every snapshot in HBM."""
    nz, nx, nt = 50, 160, 210
    v, h, dt, src, rec, wav = _case(nz, nx, nt, seed=9)
    obs = fo.Problem(v * 0.96, h, dt, src, rec, nabs=10).forward(wav)
    prop = ac.Propagator2D((nz, nx), h, dt, nabs=10, **kw)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    J0, g0, _ = prop.gradient(wav, obs)
    plane = nz * 160 * 4
    prop.set_memory_limit(70 * plane)                      # < nt planes -> segments of ceil(sqrt(2 nt)) = 21 steps
    J1, g1, _ = prop.gradient(wav, obs)
    assert abs(J1 - J0) <= 1e-12 * J0
    # identical up to the pairing of the deferred imaging at the receiver points (segments pair steps differently)
    assert rel_l2(g1.cpu().numpy(), g0.cpu().numpy()) <= 1e-6
    # the last forward sweep was the recompute of the first segment: wavefield() returns its u_21 and u_20
    import torch
    cur, old = prop.wavefield(0), prop.wavefield(1)
    prop.forward(wav[:21])
    assert torch.equal(prop.wavefield(0), cur)
    assert torch.equal(prop.wavefield(1), old)
    prop.set_memory_limit(5 * plane)
    with pytest.raises(ValueError):
        prop.gradient(wav, obs)
    prop.close()


def test_entry_points_misfit_update_fwi(ac):
    import torch
    nz, nx, nt = 40, 90, 150
    v_true = fo.layered_model((nz, nx), 1800.0, 2600.0, 3)
    v0 = np.full_like(v_true, 2100.0)
    h = 10.0
    dt = fo.stable_dt(v_true.max(), h, 2)
    wav = fo.ricker(nt, dt, 20.0)
    shots = [([(3, sx)], [(3, x) for x in range(2, nx - 2, 2)]) for sx in (12, 45, 78)]
    obs = ac.forward_model(torch.tensor(v_true, dtype=torch.float32), h, dt, shots, wav, nabs=8)
    obs_ref = [fo.Problem(v_true, h, dt, s, r, nabs=8).forward(wav[:, None].astype(np.float64)) for s, r in shots]
    for a, b in zip(obs, obs_ref):
        assert rel_l2(a.cpu().numpy(), b) <= 1e-5
    syn = ac.forward_model(torch.tensor(v0, dtype=torch.float32), h, dt, shots, wav, nabs=8)
    J = ac.misfit(syn, obs)
    J_ref = sum(fo.misfit(s.cpu().numpy(), o.cpu().numpy()) for s, o in zip(syn, obs))
    assert abs(J - J_ref) <= 1e-6 * J_ref
    Jg, g = ac.gradient(torch.tensor(v0, dtype=torch.float32), h, dt, shots, wav, obs, nabs=8)
    assert abs(Jg - J) <= 1e-5 * J
    g_ref = sum(fo.Problem(v0, h, dt, s, r, nabs=8).misfit_and_gradient(wav[:, None].astype(np.float64), o.cpu().numpy().astype(np.float64))[1]
                for (s, r), o in zip(shots, obs))
    assert rel_l2(g.cpu().numpy(), g_ref) <= 1e-4
    vt = torch.tensor(v0, dtype=torch.float32, device="cuda")
    step = 0.01 * ac.absmax(vt) / ac.absmax(g)
    v1 = ac.model_update(vt.clone(), g, step, 1500.0, 3000.0)
    np.testing.assert_allclose(v1.cpu().numpy(), fo.model_update(v0.astype(np.float32), g.cpu().numpy(), np.float32(step), 1500.0, 3000.0), rtol=1e-6)
    v_inv, hist = ac.fwi(v0, h, dt, shots, wav, obs, 3, 1500.0, 3000.0, nabs=8)
    assert hist[-1] < hist[0]
    v_orc, hist_orc = fo.fwi(v0, h, dt, shots, wav[:, None].astype(np.float64), [o.cpu().numpy().astype(np.float64) for o in obs],
                             3, 1500.0, 3000.0, nabs=8)
    np.testing.assert_allclose(hist, hist_orc, rtol=2e-3)


def test_size_independent_properties_at_scale(ac):
    """A BASELINE-config-2-shaped grid (1000 x 3000) for a few hundred steps: linearity in the wavelet,
    reciprocity of source and receiver, and causality - none needs the CPU oracle at this size."""
    import torch
    nz, nx, nt = 1000, 3000, 600
    v = torch.tensor(fo.layered_model((nz, nx), 1500.0, 4500.0, 6), dtype=torch.float32)
    h = 10.0
    dt = fo.stable_dt(4500.0, h, 2)
    wav = fo.ricker(nt, dt, 12.0).astype(np.float32)
    a, b = (40, 700), (50, 715)
    prop = ac.Propagator2D((nz, nx), h, dt, nabs=40)
    prop.set_model(v)
    prop.set_geometry([a], [b, (500, 2500)])
    t1 = prop.forward(wav).cpu().numpy()
    t2 = prop.forward(2.0 * wav).cpu().numpy()
    # linearity. Not bit-exact even for a power of two: the numerical precursor passes through the denormal range,
    # where scaling is inexact, and from then on the two runs carry independent fp32 rounding noise.
    assert rel_l2(t2, 2.0 * t1) <= 2e-5
    t2 = prop.forward(2.5 * wav).cpu().numpy()
    assert rel_l2(t2, 2.5 * t1) <= 2e-5                                    # linearity up to fp32 rounding noise
    assert np.all(t1[:, 1] == 0.0)                                         # causality: ~19 km away, not reached in 600 steps
    prop.set_geometry([b], [a])
    t3 = prop.forward(wav).cpu().numpy()
    # reciprocity holds for u/m (the injection is scaled by m at the source): both points sit in the same layer
    assert rel_l2(t3[:, 0], t1[:, 0]) <= 1e-4
    prop.close()


@pytest.mark.parametrize("shape", [(100, 300), (33, 131), (1000, 3000), (2600, 3000), (2503, 3001)])
def test_size_dependent_default_kernel_is_bit_identical_to_the_tile_kernel(ac, shape):
    """fwi_fd2d_create picks the step kernel by grid size (small / L2-resident / larger than L2); whatever it picks
    gives the tile kernel's traces and gradient bit for bit."""
    import torch
    nz, nx = shape
    nt = 41
    v = torch.tensor(fo.layered_model(shape, 1500.0, 4500.0, 5), dtype=torch.float32)
    h = 10.0
    dt = fo.stable_dt(4500.0, h, 2)
    wav = fo.ricker(nt, dt, 40.0).astype(np.float32)
    src, rec = [(nz // 2, nx // 2)], [(nz // 2 + dz, nx // 2 + dx) for dz in (-3, 0, 6) for dx in range(-40, 41, 8)]
    out = []
    for kw in (dict(), dict(tile=(32, 4))):
        prop = ac.Propagator2D(shape, h, dt, nabs=20, **kw)
        prop.set_model(v)
        prop.set_geometry(src, rec)
        tr = prop.forward(wav)
        obs = 0.9 * tr
        J, g, _ = prop.gradient(wav, obs)
        out.append((tr.cpu().numpy(), J, g.cpu().numpy()))
        prop.close()
    assert np.abs(out[0][0]).max() > 0 and np.abs(out[0][2]).max() > 0
    assert np.array_equal(out[0][0], out[1][0])
    assert abs(out[0][1] - out[1][1]) <= 1e-12 * abs(out[1][1])
    assert np.array_equal(out[0][2], out[1][2])


def test_argument_errors(ac):
    prop = ac.Propagator2D((20, 40), 10.0, 1e-3)
    with pytest.raises(ValueError):
        prop.set_geometry([(25, 3)], [(1, 1)])
    with pytest.raises(ValueError):
        prop.set_model(np.ones((21, 40), np.float32))
    with pytest.raises(ValueError):
        prop.forward(np.zeros(10, np.float32))             # model not set
    with pytest.raises(ValueError):
        ac.Propagator2D((20, 40), 10.0, -1.0)
    for kw in (dict(tile=(64, 8)), dict(tile=(16, 2)), dict(tb2=16)):        # shapes the library does not build
        with pytest.raises(ValueError):
            ac.Propagator2D((40, 300), 10.0, 1e-3, **kw)
    prop.close()


@pytest.mark.parametrize("kw", [dict(tile=(32, 4)), dict(tb2=24)])
def test_programmatic_dependent_launch_does_not_change_results(ac, monkeypatch, kw):
    """Steps chained with programmatic dependent launch (default) vs plainly serialised launches (FWI_PDL=0, read when
    the plan is created), with and without CUDA graphs: identical traces and gradients."""
    v, h, dt, src, rec, wav = _case(90, 400, 121, seed=11)
    obs = fo.Problem(v * 1.03, h, dt, src, rec, nabs=10).forward(wav)
    out = []
    for pdl, graphs in (("1", True), ("0", True), ("1", False)):
        monkeypatch.setenv("FWI_PDL", pdl)
        prop = ac.Propagator2D((90, 400), h, dt, nabs=10, graphs=graphs, **kw)
        prop.set_model(v)
        prop.set_geometry(src, rec)
        tr = prop.forward(wav).cpu().numpy()
        J, g, _ = prop.gradient(wav, obs)
        out.append((tr, J, g.cpu().numpy()))
        prop.close()
    for tr, J, g in out[1:]:
        assert np.array_equal(tr, out[0][0])
        assert abs(J - out[0][1]) <= 1e-12 * abs(out[0][1])
        assert np.array_equal(g, out[0][2])
