"""Edge cases on the GPU (both tracks): empty / single / ragged batches, odd lengths, duplicated and boundary points."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fd_oracle as fo  # noqa: E402
from oracle import mc_oracle as orc  # noqa: E402


@pytest.fixture(scope="module")
def mods():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from full_waveform_inversion_b200 import acoustic as ac
    from full_waveform_inversion_b200 import full_waveform_inversion as fw
    return ac, fw


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


# ------------------------------------------------------------------------------------------------ Track A
@pytest.mark.parametrize("N", [1, 2, 31, 33, 129, 1000])
def test_ragged_batch_sizes(mods, N):
    """Batch sizes that do not fill a CTA / a warp: tail lanes must not leak into the results."""
    _, fw = mods
    d, G, _ = orc.synthetic_inputs(K=21, C=9, T=65, seed=1)           # odd T: the 2-samples-per-iteration loop has a tail
    Ms = np.random.default_rng(N).standard_normal((N, 9))
    prob = fw.SourceInversion(d, G)
    for metric, norm, simul in (("VR", False, False), ("PCC", True, True), ("gau", True, False)):
        got = prob.similarity(Ms, metric, norm, simul)
        want = orc.similarity_batch(d, G, Ms, metric, norm, simul)
        assert got.shape == (N,)
        np.testing.assert_allclose(got, want, rtol=0, atol=2e-6)
    prob.close()


@pytest.mark.parametrize("K", [1, 2, 13, 40, 97])
def test_trace_counts_beyond_the_warp_layout(mods, K):
    """More traces than warps per CTA (each warp then loops), prime counts, a single trace."""
    _, fw = mods
    d, G, _ = orc.synthetic_inputs(K=K, C=6, T=70, seed=K)
    Ms = np.random.default_rng(3).standard_normal((200, 6))
    prob = fw.SourceInversion(d, G)
    for metric, norm, simul in (("VR", False, True), ("CC", False, False), ("VR", True, False)):
        np.testing.assert_allclose(prob.similarity(Ms, metric, norm, simul),
                                   orc.similarity_batch(d, G, Ms, metric, norm, simul), rtol=0, atol=2e-6)
    prob.close()


def test_empty_batch_and_zero_vector(mods):
    import torch
    _, fw = mods
    d, G, _ = orc.synthetic_inputs(K=4, C=6, T=64, seed=2)
    prob = fw.SourceInversion(d, G)
    empty = torch.empty((6, 0), dtype=torch.float32, device="cuda")
    assert prob.eval_dev(empty, 0, 0).shape == (0,)                      # N = 0 is a no-op, not an error
    assert prob.forward_dev(empty).shape == (0, 4, 64)
    z = prob.similarity(np.zeros((1, 6)), "VR", False, False)             # M = 0: VR = 1 - sum d^2 / sum d^2 = 0
    assert abs(z[0]) <= 1e-6                                             # fp32 rounding of d leaves ~1e-7
    z = prob.similarity(np.zeros((1, 6)), "PCC", False, False)            # 0/0 like the reference (NaN), not a crash
    assert np.isnan(z[0])
    prob.close()


def test_monte_carlo_single_sample_and_remainders(mods):
    _, fw = mods
    d, G, _ = orc.synthetic_inputs(K=5, C=3, T=64, seed=6)
    MTs, MTp, _ = fw.perform_monte_carlo_sampled_waveform_inversion(d, G, 1, 1.0, "single_force", "VR", False, False)
    assert MTs.shape == (3, 1) and MTp.shape == (1,) and abs(MTp[0] - 1.0) < 1e-6
    # q3: a sample count that does not divide the worker count keeps every sample (no silent zeros)
    MTs, MTp, _ = fw.perform_monte_carlo_sampled_waveform_inversion(d, G, 1001, 1.0, "single_force", "VR", False, False, num_processors=8)
    assert MTs.shape == (3, 1001) and np.all(np.linalg.norm(MTs, axis=0) > 0.99) and np.all(MTp > 0)


# ------------------------------------------------------------------------------------------------ Track B
# the size-dependent default, the two-steps-per-pass kernel with 32 core rows and the one-step kernel with 28-row tiles
EDGE_KERNELS = [dict(), pytest.param(dict(tb2=32), id="tb2_32"), pytest.param(dict(tile=(28, 4)), id="tile_28x4")]


def _grid(nz=37, nx=131, seed=0):
    rng = np.random.default_rng(seed)
    v = (2000.0 + 500.0 * rng.random((nz, nx))).astype(np.float32).astype(np.float64)
    h = 10.0
    return v, h, fo.stable_dt(v.max(), h, 2)


@pytest.mark.parametrize("kw", EDGE_KERNELS)
@pytest.mark.parametrize("nt", [1, 2, 3, 37])
def test_short_and_odd_step_counts(mods, kw, nt):
    """nt = 1 and odd nt: the two-steps-per-pass kernel must hand its leftover step to the one-step kernel, the
    deferred-imaging adjoint must finish an unpaired step."""
    ac, _ = mods
    v, h, dt = _grid()
    src, rec = [(5, 40)], [(5, 40), (5, 41), (6, 40)] + [(4, x) for x in range(3, 128, 5)]
    full = fo.ricker(200, dt, 30.0)
    k0 = int(np.argmax(full)) - 1
    wav = full[k0: k0 + nt, None]                    # start at the wavelet's peak so even one step records something
    obs = fo.Problem(v * 1.05, h, dt, src, rec, nabs=6).forward(wav)
    J_want, g_want, tr_want = fo.Problem(v, h, dt, src, rec, nabs=6).misfit_and_gradient(wav, obs)
    prop = ac.Propagator2D(v.shape, h, dt, nabs=6, **kw)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    assert rel_l2(prop.forward(wav).cpu().numpy(), tr_want) <= 1e-5
    J, g, _ = prop.gradient(wav, obs)
    assert abs(J - J_want) <= 1e-4 * J_want and rel_l2(g.cpu().numpy(), g_want) <= 1e-4
    prop.close()


@pytest.mark.parametrize("kw", EDGE_KERNELS)
def test_corner_duplicate_and_colocated_points(mods, kw):
    """Sources in the grid corners, two sources on the same cell, a receiver on the source cell, duplicated
    receivers, points on tile boundaries (x = 119/120/127/128, z = 15/16/23/24/27/28/31/32)."""
    ac, _ = mods
    v, h, dt = _grid(48, 260, seed=3)
    nz, nx = v.shape
    src = [(0, 0), (nz - 1, nx - 1), (16, 128), (16, 128), (31, 119), (24, 119), (27, 128)]
    rec = [(0, 0), (16, 128), (16, 128), (15, 127), (32, 120), (nz - 1, 0), (0, nx - 1), (20, 200),
           (23, 120), (24, 119), (27, 127), (28, 128)]
    nt = 90
    wav = np.stack([fo.ricker(nt, dt, 25.0) * a for a in (1.0, -0.5, 0.8, 0.3, 0.6, -0.7, 0.4)], 1)
    obs = fo.Problem(v * 0.97, h, dt, src, rec, nabs=5).forward(wav)
    J_want, g_want, tr_want = fo.Problem(v, h, dt, src, rec, nabs=5).misfit_and_gradient(wav, obs)
    prop = ac.Propagator2D(v.shape, h, dt, nabs=5, **kw)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    got = prop.forward(wav).cpu().numpy()
    assert rel_l2(got, tr_want) <= 1e-5
    assert np.array_equal(got[:, 1], got[:, 2])                          # duplicated receivers read the same cell
    J, g, _ = prop.gradient(wav, obs)
    assert abs(J - J_want) <= 1e-4 * J_want and rel_l2(g.cpu().numpy(), g_want) <= 1e-4
    prop.close()


def test_no_receivers_no_sources_and_tiny_grids(mods):
    ac, _ = mods
    v, h, dt = _grid(9, 10, seed=5)                                      # smaller than one halo-padded tile
    src, rec = [(4, 5)], [(2, 2), (8, 9)]
    wav = fo.ricker(30, dt, 30.0)[:, None]
    want = fo.Problem(v, h, dt, src, rec, nabs=2).forward(wav)
    prop = ac.Propagator2D(v.shape, h, dt, nabs=2)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    assert rel_l2(prop.forward(wav).cpu().numpy(), want) <= 1e-5
    prop.set_geometry(src, np.zeros((0, 2), dtype=int))                   # no receivers: propagate only
    assert prop.forward(wav).shape == (30, 0)
    assert rel_l2(prop.wavefield(0).cpu().numpy(), fo.Problem(v, h, dt, src, rec, nabs=2).forward(wav, return_state=True)[2][0]) <= 1e-5
    prop.set_geometry(np.zeros((0, 2), dtype=int), rec)                   # no sources: the field stays identically zero
    assert float(prop.forward(np.zeros((30, 0), np.float32)).abs().max()) == 0.0
    with pytest.raises(ValueError):
        prop.gradient(np.zeros((30, 0), np.float32), np.zeros((30, 2), np.float32))   # a gradient needs a source
    prop.close()


# ------------------------------------------------------------------------------------------------ Track B: pad columns
@pytest.mark.parametrize("case", ["tile", "tile_checkpointed", "tb2", "tb2_checkpointed", "3d", "3d_checkpointed"])
def test_pad_columns_of_every_wavefield_buffer_stay_zero(mods, case):
    """Rows are padded to 32 floats; the step kernels compute the pad columns [nx, px) too (m = 0 there) and the slab
    protocol relies on them staying zero in all 8 wavefield buffers - also in the buffers that are only cleared when
    the plan is created (2/3/6/7: second pair of the two-steps-per-pass kernel, checkpoint restores)."""
    import torch
    ac, _ = mods
    three_d = case.startswith("3d")
    shape = (36, 40, 150) if three_d else (90, 300)                       # nx not a multiple of 32: 10 / 20 pad columns
    nt = 60
    v = fo.layered_model(shape, 1500.0, 3500.0, 3).astype(np.float32)
    dt = fo.stable_dt(3500.0, 10.0, 3 if three_d else 2)
    wav = fo.ricker(nt, dt, 15.0).astype(np.float32)
    kw = {}
    if case.startswith("tb2"):
        kw["tb2"] = 24
    elif not three_d:
        kw["tile"] = (32, 4)
    prop = (ac.Propagator3D if three_d else ac.Propagator2D)(shape, 10.0, dt, nabs=10, **kw)
    prop.set_model(torch.from_numpy(v).cuda())
    if three_d:
        prop.set_geometry([(5, 20, shape[2] - 2)], [(4, 10, shape[2] - 1), (6, 30, 3)])      # points in the last real columns
    else:
        prop.set_geometry([(5, shape[1] - 2)], [(4, shape[1] - 1), (6, 3)])
    if case.endswith("checkpointed"):
        plane = int(np.prod(shape[:-1])) * ((shape[-1] + 31) // 32 * 32) * 4
        prop.set_memory_limit(30 * plane)                                  # half the nt = 60 snapshots fit: checkpointed segments
    obs = prop.forward(wav).clone() * 0.5
    prop.gradient(wav, obs)
    prop.gradient(wav, obs)
    torch.cuda.synchronize()
    nx = shape[-1]
    for idx in range(8):
        pad = prop.field_view(idx)[..., nx:]
        assert pad.numel() > 0
        assert float(pad.abs().max()) == 0.0, "buffer %d has non-zero pad columns" % idx
    prop.close()
