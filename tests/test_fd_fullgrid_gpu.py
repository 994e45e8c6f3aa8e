"""Track B checked at EVERY grid point at the benchmarked sizes, against float64 references (oracle/fd_check.py).

The parity tests of test_fd_scale_gpu.py compare one global rel-L2 per array, which the strong arrivals next to the
single source dominate; they cannot see the partial last tiles, the pad columns, the sponge strips or the far and late
parts of the record.  Here:

(a) one step of the step API from random full fields (buffers 0/1 forward with a snapshot, 4/5 adjoint with imaging) for
    every built tile shape of the one-step 2-D kernel and for the 3-D kernel, against `step64` with the bound
    |err| <= K1 eps32 S at every point, the receiver row and the image included;
(b) short sweeps with dense injection (sources every 3 cells plus every edge row and column, random wavelets, a receiver
    on every point, random observed data) through the public forward / gradient - tb2, deferred imaging (ADJ2), graphs,
    PDL, checkpointing - against the float64 C port with the bound |err| <= K2 eps32 max_9x9|ref| on every step's field,
    on the final state and on the gradient;
(c) a 2000-step sweep with sources near all four edges: rel-L2 per receiver group x time window and per gradient region,
    against the float32 port's on the same selection;
(d) the comparator run on deliberately perturbed GPU runs (one sponge value, one model point) must name the place.

Each case prints its worst err / (eps32 scale), with location and region."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fd_check as fc  # noqa: E402
from oracle import fd_oracle as fo  # noqa: E402
from oracle import fd_oracle_c as foc  # noqa: E402

# K1: one step; K2: every step's field and the final state of a sweep; K2_GRAD: the gradient of a sweep (a sum of nt
# products of two fields).  Each is at least 4x the worst ratio measured on a B200 (148 SMs, default power limit):
# 3.1 for one step, 27.1 for the fields and 50 for the gradients (see the docstrings of (a) and (b)).
K1, K2, K2_GRAD = 16.0, 128.0, 256.0
H, ALPHA = 10.0, 0.3


@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from full_waveform_inversion_b200 import acoustic
    return acoustic, torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def velocity(shape, seed):
    rng = np.random.default_rng(seed)
    v = (fo.layered_model(shape, 1500.0, 4500.0, 6) + 50.0 * rng.standard_normal(shape)).astype(np.float32)
    return v, fo.stable_dt(float(v.max()), H, len(shape))


def axis_points(n, every, tile=None):
    """Coordinates every `every` cells plus both edges and, with `tile`, both sides of every tile boundary."""
    pts = set(range(0, n, every)) | {0, n - 1}
    if tile:
        for b in range(tile, n, tile):
            pts |= {b - 1, b}
    return np.array(sorted(pts))


def lattice(shape, every, tiles=None):
    axes = [axis_points(n, every, None if tiles is None else tiles[k]) for k, n in enumerate(shape)]
    return np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, len(shape))


def all_points(shape):
    return np.stack(np.meshgrid(*[np.arange(n) for n in shape], indexing="ij"), -1).reshape(-1, len(shape))


def pads_are_zero(prop, buffers):
    import torch
    torch.cuda.synchronize()
    nx = prop.shape[-1]
    for i in buffers:
        pad = prop.field_view(i)[..., nx:]
        assert pad.numel() == 0 or float(pad.abs().max()) == 0.0, "wavefield buffer %d has non-zero pad columns" % i


def tile_sizes(d):
    """Tile length per axis of a decomposition (for the lattice of tile boundaries)."""
    return (d.zchunk, d.ty, d.tx) if d.kind == "3d" else (d.tz, d.tx)


# ------------------------------------------------------------------------------------------------ (a) one step
ONE_STEP = [((nz, nx), tile) for nz, nx in ((1000, 3000), (2503, 3001)) for tile in ((32, 4), (28, 4), (42, 6), (56, 8))]
ONE_STEP_3D = [((64, 512, 512), 14), ((64, 512, 512), 16), ((200, 150, 517), None)]


def one_step(ac, shape, nabs, decomp, seed, **kw):
    import torch
    rng = np.random.default_rng(seed)
    v, dt = velocity(shape, seed)
    tiles = tile_sizes(decomp)
    src, rec = lattice(shape, 5, tiles), lattice(shape, 4, tiles)
    prop = ac.Propagator(shape, H, dt, nabs=nabs, alpha=ALPHA, **kw)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    prop.reserve_snapshots(1)
    nx = shape[-1]

    def fill(i):
        a = rng.standard_normal(shape).astype(np.float32)
        f = prop.field_view(i)
        f.zero_()
        f[..., :nx] = torch.from_numpy(a).cuda()
        return a
    dev = lambda a: torch.from_numpy(a).cuda()
    u_n, u_o = fill(0), fill(1)
    f = rng.standard_normal(len(src)).astype(np.float32)
    r = rng.standard_normal(len(rec)).astype(np.float32)
    f_d, r_d, rec_out = dev(f), dev(r), torch.zeros(len(rec), dtype=torch.float32, device="cuda")
    prop.step(1, 0, f_d.data_ptr(), rec_out.data_ptr(), snap_index=0)      # FWD_SAVE: u_{n+1} -> buffer 1, w_n -> snapshot 0
    prop.reset(1)
    q_n, q_o = fill(4), fill(5)
    prop.step(2, 0, r_d.data_ptr(), None, snap_index=0)                    # ADJ: q -> buffer 5, image += q w_n
    torch.cuda.synchronize()
    new = prop.field_view(1)[..., :nx].cpu().numpy()
    qnew = prop.field_view(5)[..., :nx].cpu().numpy()
    img = prop.wavefield(2).cpu().numpy()
    rows = rec_out.cpu().numpy()
    pads_are_zero(prop, (0, 1, 4, 5))
    prop.close()

    m, g = fc.model(v, H, dt, nabs, ALPHA)
    si, ri = tuple(src.T), tuple(rec.T)
    new64, w64, S, aw = fc.step64(u_n, u_o, m, g, (si, f))
    q64, _, Sq, _ = fc.step64(q_n, q_o, m, g, (ri, r))
    del u_n, u_o, q_n, q_o
    label = "%s %s" % (shape, decomp)
    res = [fc.check_points("u_{n+1} " + label, new, new64, S, K1, decomp),
           fc.check_points("receiver row " + label, rows, new64[ri], S[ri], K1),
           fc.check_points("adjoint q " + label, qnew, q64, Sq, K1, decomp),
           fc.check_points("image " + label, img, q64 * w64, Sq * np.abs(w64) + np.abs(q64) * aw, K1, decomp)]
    for x in res:
        print("\n" + x.summary(), end="")
    for x in res:
        x.check()


@pytest.mark.parametrize("shape,tile", ONE_STEP, ids=["%dx%d-%dx%d" % (s + t) for s, t in ONE_STEP])
def test_one_step_2d_every_tile_shape(env, shape, tile):
    """FWD_SAVE then ADJ through the step API with every built tile of the one-step kernel: 1000 x 3000 and 2503 x 3001
    (partial last tile row and column for every height, pad columns).  Worst ratio measured on a B200 over these and the
    3-D cases: 3.1 (u_{n+1} 2.8, receiver rows 2.2, adjoint field 3.1, image 1.7)."""
    ac, sms = env
    d = fc.Decomp.for_plan(shape, sms, 40, tile=tile)
    one_step(ac, shape, 40, d, seed=sum(shape) + tile[0], tile=tile)


@pytest.mark.parametrize("shape,by", ONE_STEP_3D, ids=["%dx%dx%d-by%s" % (s + (b,)) for s, b in ONE_STEP_3D])
def test_one_step_3d(env, monkeypatch, shape, by):
    """The 3-D kernel with 14- and 16-row tiles on 512-wide planes (the slab shape) and the default at a ragged shape
    with several z chunks."""
    ac, sms = env
    if by:
        monkeypatch.setenv("FWI_FD3D_BY", str(by))
    else:
        monkeypatch.delenv("FWI_FD3D_BY", raising=False)
    d = fc.Decomp.for_plan(shape, sms, 16, by=by)
    if by is None:
        assert d.zchunk < shape[0]                       # the ragged case must have several z chunks
    one_step(ac, shape, 16, d, seed=sum(shape))


# ------------------------------------------------------------------------------------------------ (b) dense sweeps
def dense_inputs(shape, nt, seed=1):
    rng = np.random.default_rng(seed)
    v, dt = velocity(shape, seed)
    src = lattice(shape, 3)
    rec = all_points(shape)
    wav = rng.standard_normal((nt, len(src))).astype(np.float32)
    obs = rng.standard_normal((nt, len(rec))).astype(np.float32)
    return v, dt, src, rec, wav, obs


_ORACLE = {}


def dense_oracle(shape, nt, nabs):
    """float64 C port: every step's field, the final state and the gradient (cached for the 2-D cases)."""
    key = (shape, nt, nabs)
    if key in _ORACLE:
        return _ORACLE[key]
    v, dt, src, rec, wav, obs = dense_inputs(shape, nt)
    _, state = foc.forward(v, H, dt, src, rec, wav, nabs=nabs, alpha=ALPHA, dtype=np.float64, return_state=True)
    _, g64, tr64 = foc.misfit_and_gradient(v, H, dt, src, rec, wav, obs, nabs=nabs, alpha=ALPHA, dtype=np.float64)
    tr64 = tr64.reshape((nt,) + shape)
    out = dict(tr=tr64, lm=None, state=state, grad=g64)
    if shape == (1000, 3000):                             # reused by the forced-kernel and the perturbation cases
        out["lm"] = [fc.local_max(t) for t in tr64]
        _ORACLE[key] = out
    return out


def dense_gpu(ac, shape, nt, nabs, perturb=None, memory_limit=0, **kw):
    """GPU forward + gradient of the dense case -> (traces of the forward, traces of the gradient, state, gradient,
    launches of the forward, the propagator's plane size in bytes)."""
    import torch
    v, dt, src, rec, wav, obs = dense_inputs(shape, nt)
    prop = ac.Propagator(shape, H, dt, nabs=nabs, alpha=ALPHA, **kw)
    vg = v.copy()
    if perturb and "v" in perturb:
        idx, fac = perturb["v"]
        vg[idx] *= np.float32(fac)
    prop.set_model(vg)
    if perturb and "gx" in perturb:
        gx = ac.sponge_profile(shape[-1], nabs, ALPHA)
        gx[-1] *= np.float32(perturb["gx"])
        prop.set_profiles(gx=gx)
    prop.set_geometry(src, rec)
    l0 = prop.launch_count()
    trf = prop.forward(wav).cpu().numpy()
    launches = prop.launch_count() - l0
    _, g, tr = prop.gradient(wav, obs, want_traces=True)
    out = dict(trf=trf.reshape((nt,) + shape), tr=tr.cpu().numpy().reshape((nt,) + shape), grad=g.cpu().numpy(),
               state=(prop.wavefield(0).cpu().numpy(), prop.wavefield(1).cpu().numpy()), launches=launches)
    plane = int(np.prod(shape[:-1])) * ((shape[-1] + 31) // 32 * 32) * 4
    if memory_limit:
        prop.set_memory_limit(memory_limit * plane)
        _, gc, trc = prop.gradient(wav, obs, want_traces=True)
        out["grad_ckpt"] = gc.cpu().numpy()
        out["tr_ckpt"] = trc.cpu().numpy().reshape((nt,) + shape)
    pads_are_zero(prop, range(8))
    prop.close()
    return out


def dense_checks(label, got, ref, d):
    res = [fc.check_sweep("traces " + label, got["tr"], ref["tr"], K2, d, scales=ref["lm"]),
           fc.check_field("u_nt " + label, got["state"][0], ref["state"][0], K2, d),
           fc.check_field("u_nt-1 " + label, got["state"][1], ref["state"][1], K2, d),
           fc.check_field("gradient " + label, got["grad"], ref["grad"], K2_GRAD, d)]
    if "grad_ckpt" in got:
        res.append(fc.check_field("checkpointed gradient " + label, got["grad_ckpt"], ref["grad"], K2_GRAD, d))
    for x in res:
        print("\n" + x.summary(), end="")
    return res


DENSE_2D = [((1000, 3000), None), ((751, 2301), None), ((2503, 3001), None), ((1000, 3000), ("tb2", 24)),
            ((1000, 3000), ("tile", (28, 4)))]


@pytest.mark.parametrize("nt", [8, 13])
@pytest.mark.parametrize("shape,force", DENSE_2D, ids=["%dx%d-%s" % (s + ((f[0] if f else "default"),)) for s, f in DENSE_2D])
def test_dense_sweep_2d(env, shape, force, nt):
    """Dense sweeps through forward / gradient: the default plan at 1000 x 3000 (one-step kernel, 56-row tiles on 148
    SMs, deferred imaging), 751 x 2301 (tb2, 24 core rows: 7-row last tile row, 21-column last core column) and
    2503 x 3001 (tb2, 32 core rows), and tb2 / 28-row tiles forced at 1000 x 3000.  nt = 8 pairs every step; nt = 13 leaves
    a single forward step behind the two-step passes and an unpaired adjoint step, and is repeated with the memory limit
    at 12 snapshot planes, i.e. checkpointed segments of 6 + 6 + 1 steps.  Worst ratios measured on a B200 over these
    and the 3-D cases: fields 27.1 (2503 x 3001, nt = 13), gradients 50 (the same case, checkpointed); the float32 C port
    reaches 5.9 and 11.1 on the CPU test grid of test_fd_check.py."""
    ac, sms = env
    kw = {} if force is None else {force[0]: force[1]}
    d = fc.Decomp.for_plan(shape, sms, 40, **kw)
    got = dense_gpu(ac, shape, nt, 40, memory_limit=12 if nt == 13 else 0, **kw)
    assert got["launches"] == (nt // 2 + nt % 2 if d.kind == "tb2" else nt), (d, got["launches"])
    assert np.array_equal(got["trf"], got["tr"])           # forward and the gradient's forward: the same numbers
    ref = dense_oracle(shape, nt, 40)
    res = dense_checks("%s %s nt=%d" % (shape, d, nt), got, ref, d)
    if "grad_ckpt" in got:
        assert np.array_equal(got["tr_ckpt"], got["tr"])
        assert fc.rel_l2(got["grad_ckpt"], got["grad"]) <= 1e-6
    for x in res:
        x.check()


@pytest.mark.parametrize("by", [14, 16])
def test_dense_sweep_3d(env, monkeypatch, by):
    """64 x 512 x 512 with 14- and 16-row tiles, nt = 9 (one unpaired deferred-imaging step)."""
    ac, sms = env
    monkeypatch.setenv("FWI_FD3D_BY", str(by))
    shape, nt = (64, 512, 512), 9
    d = fc.Decomp.for_plan(shape, sms, 16, by=by)
    got = dense_gpu(ac, shape, nt, 16)
    assert got["launches"] == nt
    assert np.array_equal(got["trf"], got["tr"])
    del got["trf"]
    ref = dense_oracle(shape, nt, 16)
    for x in dense_checks("%s %s nt=%d" % (shape, d, nt), got, ref, d):
        x.check()


# ------------------------------------------------------------------------------------------------ (c) late, far, deep
def test_long_sweep_regions_and_windows(env):
    """1000 x 3000, nt = 2000, two sources near the surface and one near each of the left, right and bottom edges,
    each firing a Ricker pulse every 500 steps (so that every window holds fresh arrivals, not only the sponge-damped
    tail of the first); receivers on the surface and bottom rows and the first and last columns, each edge in two
    halves; observed data zero.  Per receiver group x 500-step window and per gradient region (sponge strips, last tile
    row / column, interior): GPU rel-L2 <= max(4 x the float32 port's, 1e-6), at most 1e-4, and every selection
    carries at least 1e-6 of the float64 norm."""
    import torch
    ac, sms = env
    nz, nx, nt, nabs = 1000, 3000, 2000, 40
    v = fo.layered_model((nz, nx), 1500.0, 4500.0, 6).astype(np.float32)
    dt = fo.stable_dt(4500.0, H, 2)
    src = [(4, 1000), (4, 2500), (500, 2985), (985, 1500), (500, 15)]
    wav = np.stack([sum(fo.ricker(nt, dt, 10.0, t0=0.12 + 0.05 * k + 500 * j * dt) for j in range(4)) * (1.0 - 0.15 * k)
                    for k in range(len(src))], 1).astype(np.float32)
    groups = {}
    for name, start, n in (("surface", 0, nx), ("bottom", nx, nx), ("left", 2 * nx, nz), ("right", 2 * nx + nz, nz)):
        groups[name + " 1st half"] = start + np.arange(n // 2)             # each half of an edge, so that the
        groups[name + " 2nd half"] = start + np.arange(n // 2, n)          # receivers far from a source count too
    rec = [(0, x) for x in range(nx)] + [(nz - 1, x) for x in range(nx)] + [(z, 0) for z in range(nz)] + [(z, nx - 1) for z in range(nz)]
    obs = np.zeros((nt, len(rec)), np.float32)
    prop = ac.Propagator((nz, nx), H, dt, nabs=nabs, alpha=ALPHA)
    prop.set_model(torch.from_numpy(v))
    prop.set_geometry(src, rec)
    _, g, tr = prop.gradient(wav, obs, want_traces=True)
    g, tr = g.cpu().numpy(), tr.cpu().numpy()
    prop.close()
    _, g64, tr64 = foc.misfit_and_gradient(v, H, dt, src, rec, wav, obs, nabs, ALPHA, dtype=np.float64, seg=50)
    _, g32, tr32 = foc.misfit_and_gradient(v, H, dt, src, rec, wav, obs, nabs, ALPHA, dtype=np.float32, seg=50)
    d = fc.Decomp.for_plan((nz, nx), sms, nabs)
    rows = fc.region_table(tr, tr32, tr64, fc.trace_selections(groups, nt, [(k, k + 500) for k in range(0, nt, 500)]))
    rows += fc.region_table(g, g32, g64, {"gradient " + k: m for k, m in d.masks().items()})
    print("\n" + fc.format_table("1000x3000 nt=2000, %s" % d, rows))
    for name, e_gpu, e_32, share in rows:
        assert share >= 1e-6, "%s carries no signal (%.2e of the norm)" % (name, share)
        assert e_gpu <= min(max(4.0 * e_32, 1e-6), 1e-4), "%s: GPU rel-L2 %.3e vs float32 port %.3e" % (name, e_gpu, e_32)


# ------------------------------------------------------------------------------------------------ (d) teeth
def test_comparator_catches_a_sponge_value_on_the_gpu(env):
    """gx[nx-1] scaled by 1 + 1e-3 in the GPU plan only: the sweep check fails and names column nx-1."""
    ac, sms = env
    shape, nt = (1000, 3000), 8
    d = fc.Decomp.for_plan(shape, sms, 40)
    got = dense_gpu(ac, shape, nt, 40, perturb={"gx": 1.0 + 1e-3})
    res = fc.check_sweep("traces, perturbed sponge", got["tr"], dense_oracle(shape, nt, 40)["tr"], K2, d,
                         scales=dense_oracle(shape, nt, 40)["lm"])
    print("\n" + res.report())
    assert not res.ok and res.where[1][1] == shape[1] - 1


def test_comparator_catches_a_model_point_in_the_last_tile_row_on_the_gpu(env):
    """v at (955, 1501), inside the last partial row of 56-row tiles (z >= 952), scaled by 1 + 1e-2 in the GPU plan only:
    the sweep check fails and names that point (the step after the first that reaches it: ratio ~2e3)."""
    ac, sms = env
    shape, nt, pt = (1000, 3000), 8, (955, 1501)
    d = fc.Decomp.for_plan(shape, sms, 40)
    assert "last-tile-row" in d.label(pt)
    got = dense_gpu(ac, shape, nt, 40, perturb={"v": (pt, 1.0 + 1e-2)})
    ref = dense_oracle(shape, nt, 40)
    res = fc.check_sweep("traces, perturbed model", got["tr"], ref["tr"], K2, d, scales=ref["lm"])
    print("\n" + res.report())
    assert not res.ok and tuple(int(i) for i in res.where[1]) == pt
