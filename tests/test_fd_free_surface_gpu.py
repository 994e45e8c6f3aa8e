"""The free-surface top boundary on the GPU (spec B6, tests/free_surface_reference.py).

Three kinds of check:
  * against the float64 FS oracle: traces and wavefields rel-L2 <= 1e-5, gradients <= 1e-4, Born <= 1e-5, Gauss-Newton
    <= 1e-4 (the north_star tolerances), on every 2-D kernel family with partial last tiles and in 3-D at both tile heights;
  * bit for bit (torch.equal) against the plain propagator on the grid doubled about row 0 with image sources and image
    receivers (B6's anchor), which needs no oracle and so also runs at 1000 x 3000;
  * the plan's contract: zero surface row and pad columns, launch counts, errors, peer-memory slabs.
"""
import ctypes
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fd_oracle as fo  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))     # the B5 / B6 references live beside the tests
import born_reference as br  # noqa: E402
import free_surface_reference as fsr  # noqa: E402


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


def case2d(nz, nx, nt, seed=0):
    """Sources at z = 1, 2 and 4 (inside the mirrored halo), receivers at z = 1 and one deep."""
    rng = np.random.default_rng(seed)
    v = f32(fo.layered_model((nz, nx), 1600.0, 3200.0, 4) + 60.0 * rng.standard_normal((nz, nx)))
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 2)
    src = [(1, nx // 3), (2, nx // 2 + 7), (4, 2 * nx // 3)]
    rec = [(1, x) for x in range(2, nx - 2, 3)] + [(nz - 7, nx // 2)]
    wav = f32(np.stack([fo.ricker(nt, dt, 18.0), 0.7 * fo.ricker(nt, dt, 22.0), -0.5 * fo.ricker(nt, dt, 15.0)], 1))
    dv = f32(sum(a * np.exp(-((np.arange(nz)[:, None] - cz) ** 2 + (np.arange(nx)[None] - cx) ** 2) / 18.0)
                 for a, cz, cx in [(1.0, nz // 2, nx // 2), (-0.7, 2, nx // 4), (0.8, nz - 3, nx - 4)]))
    return v, h, dt, src, rec, wav, dv


def case3d(shape, nt, seed=0):
    rng = np.random.default_rng(seed)
    nz, ny, nx = shape
    v = f32(fo.layered_model(shape, 1700.0, 3000.0, 3) + 50.0 * rng.standard_normal(shape))
    h = 10.0
    dt = fo.stable_dt(v.max(), h, 3)
    src = [(1, ny // 2, nx // 3), (4, ny // 3, nx // 2)]
    rec = [(1, y, x) for y in range(2, ny - 2, 5) for x in range(2, nx - 2, 7)] + [(nz - 6, ny // 2, nx // 2)]
    wav = f32(np.stack([fo.ricker(nt, dt, 22.0), 0.6 * fo.ricker(nt, dt, 17.0)], 1))
    g = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    dv = f32(np.exp(-sum((gi - c) ** 2 for gi, c in zip(g, (nz // 2, ny // 2, nx // 2))) / 12.0)
             - 0.6 * np.exp(-sum((gi - c) ** 2 for gi, c in zip(g, (2, 3, nx // 4))) / 12.0))
    return v, h, dt, src, rec, wav, dv


def plan(ac, shape, h, dt, v, src, rec, nabs, **kw):
    p = ac.Propagator(shape, h, dt, nabs=nabs, **kw)
    p.set_model(v)
    p.set_geometry(src, rec)
    return p


def obs_for(ac, shape, h, dt, v, src, rec, nabs, wav, **kw):
    """Observed data from a 3 % faster model, same boundary."""
    p = plan(ac, shape, h, dt, v * 1.03, src, rec, nabs, free_surface=True, **kw)
    out = p.forward(wav).cpu().numpy().astype(np.float64)
    p.close()
    return out


PLANS_2D = [dict(tile=(32, 4)), dict(tile=(28, 4)), dict(tile=(42, 6)), dict(tile=(56, 8)), dict(tb2=24), dict(tb2=32),
            dict(), dict(graphs=False)]
_oracle = {}


def oracle2d(nz, nx, nt, nabs=12):
    key = (nz, nx, nt)
    if key not in _oracle:
        v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=nz)
        p = fsr.Problem(v, h, dt, src, rec, nabs=nabs)
        tr, _, (cur, old) = p.forward(wav, return_state=True)
        _oracle[key] = tr, cur, old
    return _oracle[key]


# ------------------------------------------------------------------------------------------------ 1. vs float64 oracle
@pytest.mark.parametrize("kw", PLANS_2D)
@pytest.mark.parametrize("nt", [200, 201])
def test_forward_vs_oracle_2d(ac, kw, nt):
    """Every 2-D kernel family (tb2 at even and odd nt), 70 x 150: partial last tiles in z and x."""
    nz, nx = 70, 150
    v, h, dt, src, rec, wav, _ = case2d(nz, nx, nt, seed=nz)
    tr, cur, old = oracle2d(nz, nx, nt)
    p = plan(ac, (nz, nx), h, dt, v, src, rec, 12, free_surface=True, **kw)
    got = p.forward(wav).cpu().numpy()
    e = [rel_l2(got, tr), rel_l2(p.wavefield(0).cpu().numpy(), cur), rel_l2(p.wavefield(1).cpu().numpy(), old)]
    print("\n[fs forward 2-D %s nt=%d] rel-L2 traces / u_n / u_n-1: %.2e %.2e %.2e" % (kw, nt, *e))
    assert max(e) <= 1e-5
    p.close()


@pytest.mark.parametrize("by", ["16", "14"])
def test_forward_vs_oracle_3d(ac, by, monkeypatch):
    monkeypatch.setenv("FWI_FD3D_BY", by)
    shape, nt = (30, 37, 150), 90
    v, h, dt, src, rec, wav, _ = case3d(shape, nt, seed=3)
    tr, _, (cur, old) = fsr.Problem(v, h, dt, src, rec, nabs=8).forward(wav, return_state=True)
    p = plan(ac, shape, h, dt, v, src, rec, 8, free_surface=True)
    got = p.forward(wav).cpu().numpy()
    e = [rel_l2(got, tr), rel_l2(p.wavefield(0).cpu().numpy(), cur), rel_l2(p.wavefield(1).cpu().numpy(), old)]
    print("\n[fs forward 3-D by=%s] rel-L2 traces / u_n / u_n-1: %.2e %.2e %.2e" % (by, *e))
    assert max(e) <= 1e-5
    p.close()


@pytest.mark.parametrize("kw,limit", [(dict(), 0), (dict(), 60), (dict(tb2=24), 0), (dict(tb2=32), 60), (dict(tile=(32, 4)), 60)])
def test_gradient_vs_oracle_2d(ac, kw, limit):
    """Stored (limit 0) and checkpointed (60 planes for 260 steps) gradients, rel-L2 <= 1e-4; misfit to 1e-5."""
    nz, nx, nt = 70, 150, 260
    v, h, dt, src, rec, wav, _ = case2d(nz, nx, nt, seed=1)
    obs = obs_for(ac, (nz, nx), h, dt, v, src, rec, 12, wav)
    J, g, _ = fsr.Problem(v, h, dt, src, rec, nabs=12).misfit_and_gradient(wav, obs)
    p = plan(ac, (nz, nx), h, dt, v, src, rec, 12, free_surface=True, memory_limit=limit * nz * 160 * 4, **kw)
    Jg, gg, _ = p.gradient(wav, obs)
    e = rel_l2(gg.cpu().numpy(), g)
    print("\n[fs gradient 2-D %s limit=%d] rel-L2 %.2e, misfit %.2e" % (kw, limit, e, abs(Jg - J) / J))
    assert e <= 1e-4 and abs(Jg - J) <= 1e-5 * J
    assert not gg[0].any()
    p.close()


def test_gradient_born_gauss_newton_vs_oracle_3d(ac):
    shape, nt = (24, 30, 131), 70
    v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=4)
    obs = obs_for(ac, shape, h, dt, v, src, rec, 6, wav)
    prob = fsr.Problem(v, h, dt, src, rec, nabs=6)
    _, g, _ = prob.misfit_and_gradient(wav, obs)
    p = plan(ac, shape, h, dt, v, src, rec, 6, free_surface=True)
    e = [rel_l2(p.gradient(wav, obs)[1].cpu().numpy(), g), rel_l2(p.born(wav, dv)[0].cpu().numpy(), br.born(prob, wav, dv)[0]),
         rel_l2(p.gauss_newton(wav, dv)[0].cpu().numpy(), br.gauss_newton(prob, wav, dv))]
    print("\n[fs 3-D] rel-L2 gradient / born / gauss-newton: %.2e %.2e %.2e" % tuple(e))
    assert e[0] <= 1e-4 and e[1] <= 1e-5 and e[2] <= 1e-4
    p.close()


@pytest.mark.parametrize("kw", [dict(), dict(tile=(32, 4)), dict(tb2=24)])
def test_born_and_gauss_newton_vs_oracle_2d(ac, kw):
    nz, nx, nt = 70, 150, 200
    v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=2)
    prob = fsr.Problem(v, h, dt, src, rec, nabs=12)
    p = plan(ac, (nz, nx), h, dt, v, src, rec, 12, free_surface=True, **kw)
    eb = rel_l2(p.born(wav, dv)[0].cpu().numpy(), br.born(prob, wav, dv)[0])
    eg = rel_l2(p.gauss_newton(wav, dv)[0].cpu().numpy(), br.gauss_newton(prob, wav, dv))
    print("\n[fs 2-D %s] rel-L2 born %.2e, gauss-newton %.2e" % (kw, eb, eg))
    assert eb <= 1e-5 and eg <= 1e-4
    p.close()


# ------------------------------------------------------------------------------------------------ 2. the doubled-grid anchor
def anchor_pair(ac, shape, h, dt, v, src, rec, nabs, kw_fs, kw_plain=None):
    v2, s2, r2 = fsr.doubled(v, src, rec, image_receivers=True)
    fs = plan(ac, shape, h, dt, v, src, rec, nabs, free_surface=True, **kw_fs)
    pl = plan(ac, v2.shape, h, dt, v2, s2, r2, nabs, **(kw_fs if kw_plain is None else kw_plain))
    return fs, pl, v2


def check_anchor(ac, shape, h, dt, v, src, rec, wav, dv, nabs, kw, linear=True):
    import torch
    nz, nrec = shape[0], len(rec)
    fs, pl, v2 = anchor_pair(ac, shape, h, dt, v, src, rec, nabs, kw)
    w2 = np.concatenate([wav, -wav], 1)
    tr, tr2 = fs.forward(wav), pl.forward(w2)
    assert torch.equal(tr, tr2[:, :nrec]) and torch.equal(-tr, tr2[:, nrec:])
    for k in (0, 1):
        assert torch.equal(fs.wavefield(k), pl.wavefield(k)[nz - 1:])
    obs = (0.9 * tr).cpu().numpy()
    J, g, _ = fs.gradient(wav, obs)
    J2, g2, _ = pl.gradient(w2, np.concatenate([obs, -obs], 1))
    assert torch.equal(g, g2[nz - 1:]) and J2 == pytest.approx(2.0 * J, rel=1e-12)
    if linear:
        dv2 = np.concatenate([dv[:0:-1], dv], 0)
        b, b2 = fs.born(wav, dv)[0], pl.born(w2, dv2)[0]
        assert torch.equal(b, b2[:, :nrec])
        hv, hv2 = fs.gauss_newton(wav, dv)[0], pl.gauss_newton(w2, dv2)[0]
        assert torch.equal(hv, hv2[nz - 1:])
    fs.close()
    pl.close()


@pytest.mark.parametrize("kw", PLANS_2D[:6])
@pytest.mark.parametrize("nt", [120, 121])
def test_doubled_grid_bit_identical_2d(ac, kw, nt):
    nz, nx = 61, 150
    v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=7)
    check_anchor(ac, (nz, nx), h, dt, v, src, rec, wav, dv, 12, kw)


def test_doubled_grid_bit_identical_3d(ac):
    shape, nt = (20, 30, 131), 50
    v, h, dt, src, rec, wav, dv = case3d(shape, nt, seed=8)
    check_anchor(ac, shape, h, dt, v, src, rec, wav, dv, 6, {})


def test_doubled_grid_bit_identical_at_scale(ac):
    """1000 x 3000 (bench.py's size, its default kernel) against 1999 x 3000, nt = 1000: forward and gradient."""
    nz, nx, nt = 1000, 3000, 1000
    rng = np.random.default_rng(0)
    v = f32(fo.layered_model((nz, nx), 1500.0, 4500.0, 8) + 20.0 * rng.standard_normal((nz, nx)))
    h = 10.0
    dt = fo.stable_dt(4600.0, h, 2)
    src = [(2, nx // 2)]
    rec = [(1, x) for x in range(10, nx - 10, 10)] + [(500, 17), (998, 2999)]
    wav = f32(fo.ricker(nt, dt, 12.0))[:, None]
    check_anchor(ac, (nz, nx), h, dt, v, src, rec, wav, None, 20, {}, linear=False)


# ------------------------------------------------------------------------------------------------ 3. the plan's contract
@pytest.mark.parametrize("kw", [dict(), dict(tb2=24), dict(tile=(42, 6))])
def test_surface_row_pad_columns_and_launch_counts(ac, kw):
    nz, nx, nt = 70, 150, 101
    v, h, dt, src, rec, wav, _ = case2d(nz, nx, nt, seed=9)
    fs = plan(ac, (nz, nx), h, dt, v, src, rec, 12, free_surface=True, **kw)
    off = plan(ac, (nz, nx), h, dt, v, src, rec, 12, **kw)
    for p in (fs, off):
        p.forward(wav)
        p.gradient(wav, np.zeros((nt, len(rec)), np.float32))
    assert fs.launch_count() == off.launch_count()
    fs.forward(wav)
    for k in (0, 1):
        u = fs.wavefield(k)
        assert not u[0].any() and u[1:].abs().max() > 0
    for i in range(8):
        assert not fs.field_view(i)[:, nx:].any()
    fs.close()
    off.close()


def test_points_on_the_surface_are_rejected(ac):
    nz, nx = 40, 140
    v, h, dt, src, rec, wav, _ = case2d(nz, nx, 10)
    for kw in (dict(), dict(tb2=24)):
        p = plan(ac, (nz, nx), h, dt, v, src, rec, 8, free_surface=True, **kw)
        with pytest.raises(ValueError, match=r"source 1 at \(z=0, y=0, x=9\) lies on the free surface"):
            p.set_geometry([(3, 3), (0, 9)], rec)
        with pytest.raises(ValueError, match=r"receiver 0 at \(z=0, y=0, x=2\)"):
            p.set_geometry(src, [(0, 2)])
        p.close()
    p = plan(ac, (nz, nx), h, dt, v, [(0, 9)], [(0, 2)], 8)          # allowed without the surface
    p.close()
    p = plan(ac, (12, 10, 140), h, dt, np.full((12, 10, 140), 2000.0), [(1, 2, 3)], [(5, 5, 5)], 3, free_surface=True)
    with pytest.raises(ValueError, match="free surface"):
        p.set_geometry([(0, 2, 3)], [(5, 5, 5)])
    p.close()


def test_set_free_surface_clears_geometry_and_rebuilds_the_sponge(ac):
    from full_waveform_inversion_b200 import _lib
    nz, nx, nt = 40, 140, 30
    v, h, dt, src, rec, wav, _ = case2d(nz, nx, nt, seed=10)
    obs = np.zeros((nt, len(rec)), np.float32)
    p = plan(ac, (nz, nx), h, dt, v, src, rec, 8)
    want_off = p.forward(wav).clone()
    for enable in (1, 0):
        _lib.check(p._lib.fwi_fd2d_set_free_surface(p._h, enable))
        with pytest.raises(ValueError, match="at least one source and one receiver"):
            p.gradient(wav, obs)
        p.set_geometry(src, rec)
    import torch
    assert torch.equal(p.forward(wav), want_off)                      # off again: the plain sponge is back
    p.close()


def test_slab_with_upper_neighbour_rejects_the_surface(ac):
    from full_waveform_inversion_b200 import _lib
    lib = _lib.load()
    shape = (28, 12, 140)
    up = ac.Propagator((28,) + shape[1:], 10.0, 1e-3, nabs=3)
    dn = ac.Propagator((28,) + shape[1:], 10.0, 1e-3, nabs=3, free_surface=True)
    with pytest.raises(ValueError, match="upper neighbour"):
        _lib.check(lib.fwi_fd_slab_connect_local(dn._h, 4, 28, up._h, 24, None))
    _lib.check(lib.fwi_fd2d_set_free_surface(dn._h, 0))
    _lib.check(lib.fwi_fd_slab_connect_local(dn._h, 4, 28, up._h, 24, None))
    with pytest.raises(ValueError, match="upper neighbour"):
        _lib.check(lib.fwi_fd2d_set_free_surface(dn._h, 1))
    _lib.check(lib.fwi_fd2d_set_free_surface(up._h, 1))              # the top slab may have the surface
    up.close()
    dn.close()


@pytest.mark.parametrize("nslab,graphs,limit_planes", [(2, True, 0), (3, True, 0), (3, False, 0), (3, True, 34), (2, False, 30)])
def test_peer_memory_slabs_with_free_surface(ac, nslab, graphs, limit_planes):
    """The fused slab protocol between plans of one process on one GPU, the top plan with the surface: traces and the
    owned gradient planes equal the single FS plan bit for bit (with every w_n held; checkpointed runs pair deferred
    imaging steps differently, as on a single plan: <= 1e-6)."""
    import threading
    import torch
    from full_waveform_inversion_b200 import _lib
    lib = _lib.load()
    shape, nt, nabs, H = (72, 20, 140), 60, 6, 4
    v, h, dt, _, _, wav, _ = case3d(shape, nt, seed=21)
    src = [(1, 10, 40), (40, 8, 100), (23, 5, 17)]
    rec = [(1, y, x) for y in (3, 9, 15) for x in range(4, 136, 12)] + [(44, 10, 70), (24, 5, 17), (71, 10, 10)]
    wav = np.stack([wav[:, 0], wav[:, 1], 0.5 * wav[:, 0]], 1)
    full = plan(ac, shape, h, dt, v * 1.03, src, rec, nabs, free_surface=True)
    obs = full.forward(wav).clone()
    full.set_model(v)
    want_tr = full.forward(wav).cpu().numpy()
    _, g_want, _ = full.gradient(wav, obs)
    g_want = g_want.cpu().numpy()
    full.close()

    nz = shape[0]
    base, rem = divmod(nz, nslab)
    counts = [base + (1 if r < rem else 0) for r in range(nslab)]
    gz = ac.sponge_profile(nz, nabs, 0.3, free_surface=True)
    slabs = []
    for r in range(nslab):
        z0 = sum(counts[:r])
        up, down = (H if r else 0), (H if r < nslab - 1 else 0)
        lo, hi = z0 - up, z0 + counts[r] + down
        p = ac.Propagator((hi - lo,) + shape[1:], h, dt, nabs=nabs, graphs=graphs, free_surface=(r == 0))
        p.set_profiles(gz=gz[lo:hi])
        slabs.append(dict(p=p, z0=z0, n=counts[r], up=up, lo=lo, hi=hi))
    for r, s in enumerate(slabs):
        upp = slabs[r - 1] if r else None
        dnp = slabs[r + 1] if r < nslab - 1 else None
        _lib.check(lib.fwi_fd_slab_connect_local(s["p"]._h, s["up"], s["up"] + s["n"], upp["p"]._h if upp else None,
                                                 (upp["hi"] - upp["lo"] - H) if upp else 0, dnp["p"]._h if dnp else None))
    plane = shape[1] * 160 * 4
    wav_t = torch.tensor(wav, dtype=torch.float32, device="cuda")
    for s in slabs:
        s["p"].set_model(v[s["lo"]:s["hi"]])
        s["src_ids"] = [i for i, q in enumerate(src) if s["z0"] <= q[0] < s["z0"] + s["n"]]
        s["rec_ids"] = [i for i, q in enumerate(rec) if s["z0"] <= q[0] < s["z0"] + s["n"]]
        loc = lambda ids, pts: np.array([(pts[i][0] - s["lo"], pts[i][1], pts[i][2]) for i in ids], dtype=np.int64).reshape(-1, 3)
        s["p"].set_geometry(loc(s["src_ids"], src), loc(s["rec_ids"], rec))
        if limit_planes:
            s["p"].set_memory_limit(limit_planes * (s["hi"] - s["lo"]) * plane)
        s["p"].reserve(nt, gradient=False)      # allocations up front: in ONE process they can wait for a neighbour's kernel
        s["p"].reserve(nt, gradient=True)
        s["stream"] = torch.cuda.Stream()
        s["w"] = wav_t[:, s["src_ids"]].contiguous()
        s["obs"] = obs[:, s["rec_ids"]].contiguous()
        s["tr"] = torch.zeros((nt, len(s["rec_ids"])), dtype=torch.float32, device="cuda")
        s["g"] = torch.zeros(s["p"].shape, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()

    def run(fn):
        err = []

        def work(s):
            try:
                with torch.cuda.stream(s["stream"]):
                    fn(s)
                    s["stream"].synchronize()
            except Exception as exc:                              # noqa: BLE001
                err.append(exc)
        th = [threading.Thread(target=work, args=(s,)) for s in slabs]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if err:
            raise err[0]
        for s in slabs:
            e = ctypes.c_int(0)
            _lib.check(lib.fwi_fd_slab_error(s["p"]._h, ctypes.byref(e)))
            assert e.value == 0, "a step kernel timed out waiting for its neighbour"

    def grad(s):
        s["g"].zero_()
        s["p"].gradient(s["w"], s["obs"], grad=s["g"], traces_out=s["tr"], want_misfit=False)

    for rep in range(2):                                           # the second pass replays the cached graphs
        run(lambda s: s["p"].forward(s["w"], out=s["tr"]))
        got = np.zeros_like(want_tr)
        for s in slabs:
            got[:, s["rec_ids"]] = s["tr"].cpu().numpy()
        assert np.array_equal(got, want_tr)
        run(grad)
        g = np.zeros_like(g_want)
        for s in slabs:
            g[s["z0"]:s["z0"] + s["n"]] = s["g"][s["up"]:s["up"] + s["n"]].cpu().numpy()
        if limit_planes:
            assert rel_l2(g, g_want) <= 1e-6
        else:
            assert np.array_equal(g, g_want)
        assert not g[0].any()
    for s in slabs:
        s["p"].close()


# ------------------------------------------------------------------------------------------------ 4. entry points
def test_entry_points_with_free_surface(ac):
    import torch
    nz, nx, nt = 50, 140, 120
    v, h, dt, src, rec, wav, dv = case2d(nz, nx, nt, seed=11)
    shots = [(src[:1], rec), (src[1:], rec[::2])]
    p = ac.Propagator((nz, nx), h, dt, nabs=10, free_surface=True)
    p.set_model(v)
    want_tr, want_born, want_hv, want_g, J_want = [], [], torch.zeros((nz, nx), device=p.torch_device), \
        torch.zeros((nz, nx), device=p.torch_device), 0.0
    w = wav[:, 0]
    for s, r in shots:
        p.set_geometry(s, r)
        want_tr.append(p.forward(w).clone())
        want_born.append(p.born(w, dv)[0])
        p.gauss_newton(w, dv, hv=want_hv)
    observed = [0.8 * t for t in want_tr]
    for (s, r), o in zip(shots, observed):
        p.set_geometry(s, r)
        J_want += p.gradient(w, o, grad=want_g)[0]
    kw = dict(nabs=10, free_surface=True)
    assert all(torch.equal(a, b) for a, b in zip(ac.forward_model(v, h, dt, shots, w, **kw), want_tr))
    assert all(torch.equal(a, b) for a, b in zip(ac.born_model(v, h, dt, shots, w, dv, **kw), want_born))
    assert torch.equal(ac.gauss_newton_product(v, h, dt, shots, w, dv, allreduce=False, **kw), want_hv)
    J, g = ac.gradient(v, h, dt, shots, w, observed, allreduce=False, **kw)
    assert J == pytest.approx(J_want, rel=1e-12) and torch.equal(g, want_g)
    # without the flag the entry points model the plain boundary
    assert not torch.equal(ac.forward_model(v, h, dt, shots, w, nabs=10)[0], want_tr[0])
    # a caller's propagator keeps its own setting
    assert torch.equal(ac.forward_model(v, h, dt, shots, w, nabs=10, propagator=p)[0], want_tr[0])
    _, hist = ac.fwi(v, h, dt, shots, w, observed, 1, 1400.0, 3400.0, **kw)
    assert hist[0] == pytest.approx(J_want, rel=1e-12)
    p.close()
