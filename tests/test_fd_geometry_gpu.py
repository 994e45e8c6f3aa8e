"""A rejected fwi_fd*_set_geometry / set_positions leaves the plan with the geometry it had: every source and receiver is
checked before anything in the plan changes, so the next shot runs the previous geometry bit for bit.  The same holds one
level up for SlabPropagator's per-rank source and receiver bookkeeping."""
import os
import socket

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


NT = 121          # odd: a tb2 plan runs its last step with the one-step tile kernel, which reads the tile point lists


def case(shape):
    v = fo.layered_model(shape, 1700.0, 3000.0, 3).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(3000.0, h, len(shape))
    wav = np.stack([fo.ricker(NT, dt, 18.0), 0.7 * fo.ricker(NT, dt, 22.0), -0.5 * fo.ricker(NT, dt, 15.0)], 1)
    return v, h, dt, wav.astype(np.float32)


PLANS = [((48, 140), dict(tile=(32, 4))), ((48, 140), dict(tb2=24)), ((20, 24, 131), dict())]


@pytest.mark.parametrize("shape,kw", PLANS, ids=["tile32x4", "tb2_24", "3d"])
def test_rejected_set_geometry_keeps_the_previous_geometry(ac, shape, kw):
    import torch
    v, h, dt, wav = case(shape)
    mid = tuple(n // 2 for n in shape[1:-1])                      # (y,) in 3-D, () in 2-D
    src = [(5,) + mid + (30,), (10,) + mid + (70,), (16,) + mid + (120,)]
    rec = [(3,) + mid + (x,) for x in range(2, shape[-1] - 2, 3)]
    p = ac.Propagator(shape, h, dt, nabs=10, **kw)
    try:
        p.set_model(v)
        p.set_geometry(src, rec)
        tr = p.forward(wav).clone()
        u = p.wavefield(0)                                        # u_nt: holds the injection of the last, single step
        obs = 0.8 * tr
        J, g, gtr = p.gradient(wav, obs, want_traces=True)
        bad = rec[:-1] + [(3,) + mid + (shape[-1] + 5,)]          # the last receiver lies outside the grid
        with pytest.raises(ValueError, match="receiver"):
            p.set_geometry(src[:2], bad)
        assert p.nsrc == 3 and p.nrec == len(rec)
        assert torch.equal(p.forward(wav), tr) and torch.equal(p.wavefield(0), u)
        J2, g2, gtr2 = p.gradient(wav, obs, want_traces=True)
        # (the misfit is a sum of atomic adds: its last bit depends on their order)
        assert J2 == pytest.approx(J, rel=1e-12) and torch.equal(g2, g) and torch.equal(gtr2, gtr)
    finally:
        p.close()


def test_rejected_set_geometry_keeps_off_grid_positions(ac):
    import torch
    shape = (48, 140)
    v, h, dt, wav = case(shape)
    wav2 = np.ascontiguousarray(wav[:, :2])
    p = ac.Propagator(shape, h, dt, nabs=10, tile=(32, 4))
    try:
        p.set_model(v)
        # float positions, then an integer geometry with a bad receiver: the positions stay
        p.set_geometry(np.array([(10.5, 30.25), (25.0, 90.5)]), np.array([(3.5, x + 0.5) for x in range(2, 136, 4)]))
        tr = p.forward(wav2).clone()
        with pytest.raises(ValueError, match="receiver"):
            p.set_geometry([(5, 30)], [(3, 10), (3, 200)])
        assert torch.equal(p.forward(wav2), tr)
        # integer geometry, then positions with a NaN coordinate: the integer geometry stays
        p.set_geometry([(5, 30), (20, 70), (40, 120)], [(3, x) for x in range(2, 138, 3)])
        tr = p.forward(wav).clone()
        with pytest.raises(ValueError, match="not finite"):
            p.set_geometry(np.array([(10.5, 30.25)]), np.array([(3.5, 20.5), (np.nan, 40.0)]))
        assert torch.equal(p.forward(wav), tr)
    finally:
        p.close()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_slab_set_geometry_rejection_keeps_rank_state(ac):
    import torch
    import torch.distributed as dist
    shape = (48, 140)
    v, h, dt, wav = case(shape)
    w = np.ascontiguousarray(wav[:, 0])                           # one wavelet for every source
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % _free_port(), rank=0, world_size=1)
    try:
        slab = ac.SlabPropagator(shape, h, dt, nabs=10, use_graphs=False)
        try:
            slab.set_model(v)
            rec = [(3, x) for x in range(2, 138, 3)]
            slab.set_geometry([(5, 30), (20, 90)], rec)
            tr = slab.forward(w).clone()
            bad = rec[:-1] + [(3, 150)]                           # as many receivers as before, the last one outside the grid
            with pytest.raises(ValueError, match="receiver"):
                slab.set_geometry([(5, 30)], bad)
            assert torch.equal(slab.forward(w), tr)
            assert slab.nsrc_global == 2 and slab.nrec_global == len(rec)
        finally:
            slab.close()
    finally:
        dist.destroy_process_group()
