"""Track B (3-D) parity on the GPU vs the SELF-oracle oracle/fd_oracle.py (no reference counterpart, SURVEY 0).
Tolerances: traces rel-L2 <= 1e-5, gradient rel-L2 <= 1e-4."""
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


def _case(shape, nt, seed=0):
    rng = np.random.default_rng(seed)
    nz, ny, nx = shape
    v = fo.layered_model(shape, 1700.0, 3000.0, 3) + 50.0 * rng.standard_normal(shape)
    v = v.astype(np.float32).astype(np.float64)
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 3)
    src = [(5, ny // 2, nx // 3), (7, ny // 3, nx // 2)]
    rec = [(4, y, x) for y in range(2, ny - 2, 5) for x in range(2, nx - 2, 7)] + [(nz - 6, ny // 2, nx // 2)]
    wav = np.stack([fo.ricker(nt, dt, 22.0), 0.6 * fo.ricker(nt, dt, 17.0)], 1).astype(np.float32).astype(np.float64)
    return v, h, dt, src, rec, wav


@pytest.mark.parametrize("shape,nt", [((40, 37, 150), 90), ((70, 20, 64), 80), ((18, 50, 131), 60)])
def test_forward_3d(ac, shape, nt):
    v, h, dt, src, rec, wav = _case(shape, nt, seed=shape[0])
    want, _, (cur, old) = fo.Problem(v, h, dt, src, rec, nabs=8).forward(wav, return_state=True)
    prop = ac.Propagator(shape, h, dt, nabs=8)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    got = prop.forward(wav).cpu().numpy()
    assert rel_l2(got, want) <= 1e-5
    assert rel_l2(prop.wavefield(0).cpu().numpy(), cur) <= 1e-5
    assert rel_l2(prop.wavefield(1).cpu().numpy(), old) <= 1e-5
    prop.close()


def test_gradient_3d_and_checkpointing(ac):
    shape, nt = (36, 30, 140), 70
    v, h, dt, src, rec, wav = _case(shape, nt, seed=5)
    obs = fo.Problem(v * 1.03, h, dt, src, rec, nabs=8).forward(wav)
    J_want, g_want, tr_want = fo.Problem(v, h, dt, src, rec, nabs=8).misfit_and_gradient(wav, obs)
    prop = ac.Propagator(shape, h, dt, nabs=8)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    J, g, tr = prop.gradient(wav, obs, want_traces=True)
    assert rel_l2(tr.cpu().numpy(), tr_want) <= 1e-5
    assert abs(J - J_want) <= 1e-4 * J_want
    assert rel_l2(g.cpu().numpy(), g_want) <= 1e-4
    plane = shape[0] * shape[1] * 160 * 4
    prop.set_memory_limit(40 * plane)          # 70 snapshots do not fit -> checkpointed recompute
    J2, g2, _ = prop.gradient(wav, obs)
    assert abs(J2 - J) <= 1e-12 * J
    assert rel_l2(g2.cpu().numpy(), g.cpu().numpy()) <= 1e-6     # deferred-imaging pairs differ between segmentations
    prop.close()


def test_slab_owned_range_logic_on_one_gpu(ac):
    """The slab decomposition's per-rank logic, emulated on ONE GPU: two plans own the upper / lower half of the grid
    (4 ghost planes each), compute only their owned planes (`fwi_fd_slab_connect` without peers) and the ghost planes
    are refreshed by device copies standing in for the NVLink push.  Owned planes must equal a single-grid run
    bit for bit.  (The peer-memory push itself needs two GPUs: tools/slab_check.py.)"""
    import ctypes
    import torch
    from full_waveform_inversion_b200 import _lib
    shape, nt = (48, 20, 140), 50
    v, h, dt, src, rec, wav = _case(shape, nt, seed=11)
    src = [(6, 10, 40), (40, 8, 100)]
    rec = [(5, y, x) for y in (3, 9, 15) for x in range(4, 136, 12)] + [(44, 10, 70)]
    wav = wav[:, :2]
    full = ac.Propagator(shape, h, dt, nabs=6)
    full.set_model(v)
    full.set_geometry(src, rec)
    want = full.forward(wav).cpu().numpy()
    want_field = full.wavefield(0).cpu().numpy()
    full.close()

    H, half = 4, shape[0] // 2
    lib = _lib.load()
    gz = ac.sponge_profile(shape[0], 6, 0.3)
    plans, metas = [], []
    for r in range(2):
        z0, up, down = r * half, (H if r else 0), (0 if r else H)
        lo, hi = z0 - up, z0 + half + down
        p = ac.Propagator((hi - lo,) + shape[1:], h, dt, nabs=6, graphs=False)
        p.set_profiles(gz=gz[lo:hi])
        _lib.check(lib.fwi_fd_slab_connect(p._h, up, up + half, None, None, 0, None, None))
        p.set_model(v[lo:hi])
        s_loc = [(z - lo, y, x) for z, y, x in src if z0 <= z < z0 + half]
        r_ids = [i for i, (z, y, x) in enumerate(rec) if z0 <= z < z0 + half]
        r_loc = [(rec[i][0] - lo, rec[i][1], rec[i][2]) for i in r_ids]
        s_ids = [i for i, (z, y, x) in enumerate(src) if z0 <= z < z0 + half]
        p.set_geometry(s_loc if s_loc else np.zeros((0, 3), int), r_loc)
        plans.append(p)
        metas.append((lo, up, s_ids, r_ids))
    got = np.zeros_like(want)
    fields = [[p.field_view(i) for i in range(2)] for p in plans]
    wav_d = [torch.tensor(np.ascontiguousarray(wav[:, m[2]]) if m[2] else np.zeros((nt, 1)), dtype=torch.float32, device="cuda") for m in metas]
    out_d = [torch.zeros((nt, max(1, len(m[3]))), dtype=torch.float32, device="cuda") for m in metas]
    for p in plans:
        p.reset(0)
    cur = 0
    for n in range(nt):
        for r, p in enumerate(plans):
            p.step(0, cur, wav_d[r].data_ptr() + n * wav_d[r].shape[1] * 4, out_d[r].data_ptr() + n * out_d[r].shape[1] * 4)
        cur ^= 1
        a, b = fields[0][cur], fields[1][cur]              # upper slab: [own 24 | ghost 4]; lower slab: [ghost 4 | own 24]
        a[half:half + H].copy_(b[H:2 * H])                 # lower slab's first owned planes -> upper slab's bottom ghost
        b[0:H].copy_(a[half - H:half])                     # upper slab's last owned planes -> lower slab's top ghost
    for r, m in enumerate(metas):
        got[:, m[3]] = out_d[r][:, : len(m[3])].cpu().numpy()
    assert np.array_equal(got, want)
    px = fields[0][cur].shape[-1]
    upper = fields[0][cur][:half, :, : shape[2]].cpu().numpy()
    lower = fields[1][cur][H:, :, : shape[2]].cpu().numpy()
    assert np.array_equal(np.concatenate([upper, lower]), want_field)
    for p in plans:
        p.close()


def test_slab_rejects_points_in_ghost_planes(ac):
    """A slab computes only its owned planes and its neighbours overwrite the ghost planes, so a source or receiver there
    would be injected into a plane that is overwritten, or binned past the last z chunk.  The two plans of
    test_slab_owned_range_logic_on_one_gpu: set_geometry accepts points in the first and last owned planes and raises
    ValueError, naming the owned range, for a source or a receiver in either ghost zone."""
    from full_waveform_inversion_b200 import _lib
    shape = (48, 20, 140)
    H, half = 4, shape[0] // 2
    lib = _lib.load()
    for r in range(2):
        up, down = (H if r else 0), (0 if r else H)
        p = ac.Propagator((half + up + down,) + shape[1:], 10.0, 1e-3, nabs=6, graphs=False)
        _lib.check(lib.fwi_fd_slab_connect(p._h, up, up + half, None, None, 0, None, None))
        owned = [(up, 10, 40), (up + half - 1, 3, 139)]
        p.set_geometry(owned, owned)
        ghosts = range(half, half + H) if down else range(0, H)
        for z in (ghosts[0], ghosts[-1]):
            bad = [(z, 10, 40)]
            with pytest.raises(ValueError, match=r"\[%d, %d\)" % (up, up + half)):
                p.set_geometry(bad, owned)
            with pytest.raises(ValueError, match=r"\[%d, %d\)" % (up, up + half)):
                p.set_geometry(owned, owned + bad)
        p.close()


def _local_slabs(ac, shape, h, dt, nabs, nslab, v, src, rec, **kw):
    """What SlabPropagator builds per rank, for `nslab` plans living on ONE GPU and connected with
    fwi_fd_slab_connect_local (the peer-memory protocol without IPC)."""
    from full_waveform_inversion_b200 import _lib
    lib = _lib.load()
    H, nz = 4, shape[0]
    base, rem = divmod(nz, nslab)
    counts = [base + (1 if r < rem else 0) for r in range(nslab)]
    gz = ac.sponge_profile(nz, nabs, 0.3)
    slabs = []
    for r in range(nslab):
        z0 = sum(counts[:r])
        up, down = (H if r else 0), (H if r < nslab - 1 else 0)
        lo, hi = z0 - up, z0 + counts[r] + down
        p = ac.Propagator((hi - lo,) + shape[1:], h, dt, nabs=nabs, **kw)
        p.set_profiles(gz=gz[lo:hi])
        slabs.append(dict(p=p, z0=z0, n=counts[r], up=up, lo=lo, hi=hi))
    for r, s in enumerate(slabs):
        upp = slabs[r - 1] if r else None
        dnp = slabs[r + 1] if r < nslab - 1 else None
        _lib.check(lib.fwi_fd_slab_connect_local(s["p"]._h, s["up"], s["up"] + s["n"], upp["p"]._h if upp else None,
                                                 (upp["hi"] - upp["lo"] - H) if upp else 0, dnp["p"]._h if dnp else None))
    for s in slabs:
        s["p"].set_model(v[s["lo"]:s["hi"]])
        s["src_ids"] = [i for i, q in enumerate(src) if s["z0"] <= q[0] < s["z0"] + s["n"]]
        s["rec_ids"] = [i for i, q in enumerate(rec) if s["z0"] <= q[0] < s["z0"] + s["n"]]
        loc = lambda ids, pts: np.array([(pts[i][0] - s["lo"], pts[i][1], pts[i][2]) for i in ids], dtype=np.int64).reshape(-1, 3)
        s["p"].set_geometry(loc(s["src_ids"], src), loc(s["rec_ids"], rec))
    return slabs


def _run_ranks(slabs, fn):
    """One host thread and one CUDA stream per emulated rank (the kernels of neighbouring slabs wait for each other).
    `fn` must not allocate device memory: in ONE process cudaMalloc (also torch's caching allocator growing a pool)
    can wait for the device, i.e. for a neighbour's kernel that is itself waiting for this thread's launch.  Ranks of a
    real run are separate processes on separate GPUs."""
    import threading
    import torch
    err = []

    def work(r):
        try:
            with torch.cuda.stream(slabs[r]["stream"]):
                fn(r, slabs[r])
                slabs[r]["stream"].synchronize()
        except Exception as exc:                                  # noqa: BLE001
            err.append(exc)
    th = [threading.Thread(target=work, args=(r,)) for r in range(len(slabs))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if err:
        raise err[0]


@pytest.mark.parametrize("nslab,graphs,limit_planes,edge_rec", [(2, True, 0, True), (3, True, 0, True), (3, False, 0, True), (3, True, 34, True),
                                                                 (2, True, 30, True), (3, True, 0, False), (3, True, 34, False)])
def test_peer_memory_slab_protocol_on_one_gpu(ac, nslab, graphs, limit_planes, edge_rec):
    """The fused compute + halo-push protocol (device-resident step ids, early boundary pushes with the last chunk marching
    downwards, fence kernel before memsets / checkpoint restores, CUDA-graph replay, per-slab checkpointing, slabs without
    sources) between plans of one process on one GPU.  Traces and owned gradient planes equal a single-plan run bit for bit
    when every w_n is held; with checkpointing the deferred-imaging pairs differ (as on a single plan): <= 1e-6."""
    import ctypes
    import torch
    from full_waveform_inversion_b200 import _lib
    shape, nt = (72, 20, 140), 60
    v, h, dt, _, _, wav = _case(shape, nt, seed=21)
    src = [(6, 10, 40), (40, 8, 100), (23, 5, 17)]                # (23, ..) and (24, ..) straddle the 3-slab boundary at z = 24
    rec = [(5, y, x) for y in (3, 9, 15) for x in range(4, 136, 12)] + [(44, 10, 70)]
    if edge_rec:                                                  # receivers in boundary planes; without them the last of 3 slabs has
        rec += [(24, 5, 17), (47, 19, 139), (48, 0, 0), (71, 10, 10)]     # neither sources nor receivers
    wav = np.stack([wav[:, 0], wav[:, 1], 0.5 * wav[:, 0]], 1)
    full = ac.Propagator(shape, h, dt, nabs=6)
    full.set_model(v * 1.03)
    full.set_geometry(src, rec)
    obs = full.forward(wav).clone()
    full.set_model(v)
    want_tr = full.forward(wav).cpu().numpy()
    J_want, g_want, _ = full.gradient(wav, obs)
    g_want = g_want.cpu().numpy()
    full.close()

    slabs = _local_slabs(ac, shape, h, dt, 6, nslab, v, src, rec, graphs=graphs)
    plane = shape[1] * 160 * 4
    if limit_planes:
        for s in slabs:
            s["p"].set_memory_limit(limit_planes * (s["hi"] - s["lo"]) * plane)      # 60 snapshots do not fit -> segments of 11
    for s in slabs:                   # allocations and graph instantiation up front: in ONE process they can wait for the device,
        s["p"].reserve(nt, gradient=False)     # i.e. for a neighbour's kernel that is itself waiting for this plan's launch
        s["p"].reserve(nt, gradient=True)      # (ranks of a real run are separate processes on separate GPUs)
    wav_t, obs_t = torch.tensor(wav, dtype=torch.float32, device="cuda"), obs
    for s in slabs:                   # every buffer the ranks touch exists before they start (see _run_ranks)
        s["stream"] = torch.cuda.Stream()
        s["w"] = wav_t[:, s["src_ids"]].contiguous()
        s["obs"] = obs_t[:, s["rec_ids"]].contiguous()
        s["tr"] = torch.zeros((nt, len(s["rec_ids"])), dtype=torch.float32, device="cuda")
        s["g"] = torch.zeros(s["p"].shape, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()

    def fwd(r, s):
        s["p"].forward(s["w"], out=s["tr"])

    def grad(r, s):
        s["g"].zero_()
        s["p"].gradient(s["w"], s["obs"], grad=s["g"], traces_out=s["tr"], want_misfit=False)

    lib = _lib.load()

    def no_timeouts():
        for s in slabs:
            e = ctypes.c_int(0)
            _lib.check(lib.fwi_fd_slab_error(s["p"]._h, ctypes.byref(e)))
            assert e.value == 0, "a step kernel timed out waiting for its neighbour"

    for rep in range(2):                                           # second pass replays the cached graphs
        got = np.zeros_like(want_tr)
        _run_ranks(slabs, fwd)
        no_timeouts()
        for s in slabs:
            got[:, s["rec_ids"]] = s["tr"].cpu().numpy()
        assert np.array_equal(got, want_tr)
        _run_ranks(slabs, grad)
        no_timeouts()
        got = np.zeros_like(want_tr)
        g_got = np.concatenate([s["g"][s["up"]: s["up"] + s["n"]].cpu().numpy() for s in slabs])
        for s in slabs:
            got[:, s["rec_ids"]] = s["tr"].cpu().numpy()
        assert np.array_equal(got, want_tr)
        if limit_planes:
            assert rel_l2(g_got, g_want) <= 1e-6
        else:
            assert np.array_equal(g_got, g_want)
    torch.cuda.synchronize()
    for s in slabs:
        s["p"].close()


def test_peer_memory_slab_timeout_is_reported_not_hung(ac):
    """A slab whose neighbour never launches: the step kernels give up after the (shortened) timeout, every later launch
    returns at once, and the error flag is raised instead of computing on stale ghost planes."""
    import ctypes
    import time
    import torch
    from full_waveform_inversion_b200 import _lib
    shape, nt = (48, 20, 140), 40
    v, h, dt, _, _, wav = _case(shape, nt, seed=3)
    slabs = _local_slabs(ac, shape, h, dt, 6, 2, v, [(6, 10, 40)], [(5, 9, 30), (40, 9, 30)])
    lib = _lib.load()
    p = slabs[0]["p"]
    _lib.check(lib.fwi_fd_slab_set_timeout(p._h, 50.0))
    t0 = time.perf_counter()
    p.forward(torch.tensor(wav[:, :1], dtype=torch.float32, device="cuda"))       # rank 1 never runs
    torch.cuda.synchronize()
    assert time.perf_counter() - t0 < 5.0                          # one timeout, not one per step
    e = ctypes.c_int(0)
    _lib.check(lib.fwi_fd_slab_error(p._h, ctypes.byref(e)))
    assert e.value == 1
    _lib.check(lib.fwi_fd_slab_clear_error(p._h))
    _lib.check(lib.fwi_fd_slab_error(p._h, ctypes.byref(e)))
    assert e.value == 0
    for s in slabs:
        s["p"].close()


@pytest.mark.parametrize("by", ["14", "16"])
def test_tile_height_variants_agree_with_the_oracle(ac, monkeypatch, by):
    """The 3-D kernel's tile height (16 rows / 8 consumer warps, or 14 rows / 7 warps - chosen per plan, FWI_FD3D_BY forces it):
    same traces and gradient, against the oracle and bit-identical to each other."""
    shape, nt = (30, 45, 150), 60
    v, h, dt, src, rec, wav = _case(shape, nt, seed=8)
    obs = fo.Problem(v * 1.03, h, dt, src, rec, nabs=8).forward(wav)
    J_want, g_want, tr_want = fo.Problem(v, h, dt, src, rec, nabs=8).misfit_and_gradient(wav, obs)
    monkeypatch.setenv("FWI_FD3D_BY", by)
    prop = ac.Propagator(shape, h, dt, nabs=8)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    J, g, tr = prop.gradient(wav, obs, want_traces=True)
    prop.close()
    assert rel_l2(tr.cpu().numpy(), tr_want) <= 1e-5 and rel_l2(g.cpu().numpy(), g_want) <= 1e-4 and abs(J - J_want) <= 1e-4 * J_want
    monkeypatch.setenv("FWI_FD3D_BY", "16")
    ref = ac.Propagator(shape, h, dt, nabs=8)
    ref.set_model(v)
    ref.set_geometry(src, rec)
    J2, g2, tr2 = ref.gradient(wav, obs, want_traces=True)
    ref.close()
    assert np.array_equal(tr.cpu().numpy(), tr2.cpu().numpy()) and np.array_equal(g.cpu().numpy(), g2.cpu().numpy())
