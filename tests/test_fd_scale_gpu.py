"""Track B parity AT THE BENCHMARKED SIZES: the default CUDA path (tile kernel + programmatic dependent launch + CUDA
graphs, or whatever fwi_fd2d_create picks for the size) against the float64 build of the self-oracle's C port
(oracle/fd_oracle_c.c with -DFDC_DOUBLE, equal to oracle/fd_oracle.py to 1e-12 and anchored to analytic Green's
functions by tests/test_fd_analytic.py).  "vs self-oracle": the reference has no propagator (SURVEY 0).

Every test prints the measured rel-L2 errors; the float32 build of the same C code is run beside the GPU so the
inherent fp32 noise of the specification at that size is on record next to the GPU's.

What these check: one global rel-L2 per array in bench.py's geometry (one source at depth 4, a receiver in every surface
column).  That norm is carried by the few hundred cells next to the source - at 1000 x 3000, nt = 1000 the gradient is
exactly zero outside 6.5 % of the grid and far receivers record zeros - so the last tiles, the sponge strips, the pad
columns and late or distant signal are checked pointwise in test_fd_fullgrid_gpu.py instead."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fd_oracle as fo  # noqa: E402
from oracle import fd_oracle_c as foc  # noqa: E402

TOL_TRACES, TOL_GRAD = 1e-5, 1e-4          # north_star tolerances


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


def bench_case(nz, nx, nt, f0=10.0, sx=None):
    """bench.py's workload shape: layered 1500 -> 4500 m/s, source and a receiver in every column at depth index 4."""
    v = fo.layered_model((nz, nx), 1500.0, 4500.0, 6).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(4500.0, h, 2)
    wav = fo.ricker(nt, dt, f0).astype(np.float32)
    src = [(4, nx // 3 if sx is None else sx)]
    rec = [(4, x) for x in range(nx)]
    return v, h, dt, wav, src, rec


def gpu_gradient(ac, v, h, dt, wav, src, rec, nabs, obs=None, **kw):
    import torch
    prop = ac.Propagator(v.shape, h, dt, nabs=nabs, **kw)
    if obs is None:
        prop.set_model(torch.from_numpy(v) * 1.02)
        prop.set_geometry(src, rec)
        obs = prop.forward(wav).clone()
    prop.set_model(v)
    prop.set_geometry(src, rec)
    J, g, tr = prop.gradient(wav, obs, want_traces=True)
    out = (J, g.cpu().numpy(), tr.cpu().numpy(), obs.cpu().numpy() if hasattr(obs, "cpu") else obs)
    prop.close()
    return out


def check_against_float64(label, v, h, dt, wav, src, rec, nabs, got, seg):
    J, g, tr, obs = got
    J64, g64, tr64 = foc.misfit_and_gradient(v, h, dt, src, rec, wav, obs, nabs=nabs, dtype=np.float64, seg=seg)
    J32, g32, tr32 = foc.misfit_and_gradient(v, h, dt, src, rec, wav, obs, nabs=nabs, dtype=np.float32, seg=seg)
    e_tr, e_g, e_J = rel_l2(tr, tr64), rel_l2(g, g64), abs(J - J64) / J64
    print("\n[%s] GPU vs float64 oracle: traces rel-L2 %.3e, gradient rel-L2 %.3e, misfit rel %.3e   |   float32 CPU port vs float64: traces %.3e, gradient %.3e"
          % (label, e_tr, e_g, e_J, rel_l2(tr32, tr64), rel_l2(g32, g64)))
    # source placement / receiver indexing are integer-exact: the 9-point-per-axis star reaches 4 cells per step and the
    # source value enters u_1, so a receiver at offset d sees its first non-zero sample at step sum_axes ceil(|d_axis| / 4)
    # (checked where the precursor has not yet underflowed fp32: up to 5 hops)
    s0 = np.asarray(src[0])
    hops = np.array([int(sum(-(-abs(int(a) - int(b)) // 4) for a, b in zip(r, s0))) for r in rec])
    near = np.nonzero(hops <= 5)[0]
    assert len(near) >= 3
    first = (np.abs(tr[:, near]) > 0).argmax(0)
    assert np.array_equal(first, hops[near]), (first, hops[near])
    assert np.array_equal((np.abs(tr64[:, near]) > 0).argmax(0), hops[near])
    return e_tr, e_g, e_J


def test_bench_grid_1000x3000_nt1000_vs_float64_oracle(ac):
    """(a) of VERDICT r1: 1000 x 3000, the bench geometry (3000 receivers), nt = 1000, default kernel path."""
    v, h, dt, wav, src, rec = bench_case(1000, 3000, 1000)
    got = gpu_gradient(ac, v, h, dt, wav, src, rec, 40)
    e_tr, e_g, e_J = check_against_float64("2-D 1000x3000 nt=1000", v, h, dt, wav, src, rec, 40, got, seg=50)
    assert e_tr <= TOL_TRACES and e_g <= TOL_GRAD and e_J <= 1e-4


def test_marmousi_sized_751x2301_nt1000_vs_float64_oracle(ac):
    """(c): BASELINE config 3's grid (2301 x 751 cells: nz = 751, nx = 2301)."""
    v, h, dt, wav, src, rec = bench_case(751, 2301, 1000, f0=12.0)
    got = gpu_gradient(ac, v, h, dt, wav, src, rec, 40)
    e_tr, e_g, e_J = check_against_float64("2-D 751x2301 nt=1000", v, h, dt, wav, src, rec, 40, got, seg=50)
    assert e_tr <= TOL_TRACES and e_g <= TOL_GRAD and e_J <= 1e-4


def test_3d_192cubed_nt300_vs_float64_oracle(ac):
    """(d): 3-D 192^3 x 300 steps, gradient with every w_n held in HBM (8.5 GB)."""
    n, nt = 192, 300
    shape = (n, n, n)
    v = (fo.layered_model(shape, 1700.0, 3400.0, 5) + 30.0 * np.random.default_rng(0).standard_normal(shape)).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(float(v.max()), h, 3)
    wav = fo.ricker(nt, dt, 14.0).astype(np.float32)
    src = [(6, n // 2, n // 3)]
    rec = [(5, y, x) for y in range(4, n - 4, 6) for x in range(4, n - 4, 6)]
    got = gpu_gradient(ac, v, h, dt, wav, src, rec, 16)
    e_tr, e_g, e_J = check_against_float64("3-D 192^3 nt=300", v, h, dt, wav, src, rec, 16, got, seg=20)
    assert e_tr <= TOL_TRACES and e_g <= TOL_GRAD and e_J <= 1e-4


def test_full_size_pdl_and_graphs_do_not_change_a_bit(ac, monkeypatch):
    """PDL's early prefetch of u_{n-1} / m (fd2d.cu) at a size where it can race: 1000 x 3000 is 24 x 32 = 768 CTAs,
    more than one wave, 1000 steps.  Default (PDL + graphs) vs FWI_PDL=0 vs graphs off, three repeats of the default:
    bit-identical traces and gradients."""
    v, h, dt, wav, src, rec = bench_case(1000, 3000, 1000)
    ref = gpu_gradient(ac, v, h, dt, wav, src, rec, 40)
    obs = ref[3]
    runs = []
    for pdl, graphs in (("1", True), ("1", True), ("0", True), ("1", False)):
        monkeypatch.setenv("FWI_PDL", pdl)
        runs.append(gpu_gradient(ac, v, h, dt, wav, src, rec, 40, obs=obs, graphs=graphs))
    monkeypatch.delenv("FWI_PDL")
    for J, g, tr, _ in runs:
        assert np.array_equal(tr, ref[2])
        assert np.array_equal(g, ref[1])
        assert abs(J - ref[0]) <= 1e-12 * ref[0]          # float64 atomics in the misfit reduction: order not fixed


def test_adjoint_dot_product_through_the_cuda_kernels(ac):
    """<L w, d> = <w, L^T d> at 500 x 1500 with L = forward modelling (wavelets at the sources -> traces at the receivers).
    With the oracle's change of variable q = m g lambda the adjoint recursion IS the forward step (fd_oracle B3), so
    L^T d is the same CUDA step kernel run on the time-reversed d injected at the receivers and sampled at the sources,
    reversed in time again - the operator the gradient's back-propagation applies.  fp32: relative mismatch <= 1e-4."""
    import torch
    nz, nx, nt = 500, 1500, 700
    rng = np.random.default_rng(5)
    v = (fo.layered_model((nz, nx), 1600.0, 3800.0, 5) + 40.0 * rng.standard_normal((nz, nx))).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(float(v.max()), h, 2)
    src = [(5, 300), (40, 700), (250, 1200)]
    rec = [(4, x) for x in range(10, nx - 10, 7)] + [(300, 600), (499, 1499), (0, 0)]
    w = np.stack([fo.ricker(nt, dt, 12.0 + 3 * i) for i in range(len(src))], 1).astype(np.float32)
    w *= rng.standard_normal(w.shape).astype(np.float32) * 0.3 + 1.0
    d = rng.standard_normal((nt, len(rec))).astype(np.float32)
    d *= np.hanning(nt)[:, None].astype(np.float32)
    prop = ac.Propagator2D((nz, nx), h, dt, nabs=30)
    prop.set_model(v)
    prop.set_geometry(src, rec)
    Lw = prop.forward(w).cpu().numpy().astype(np.float64)
    prop.set_geometry(rec, src)
    LTd = prop.forward(np.ascontiguousarray(d[::-1])).cpu().numpy()[::-1].astype(np.float64)
    prop.close()
    lhs, rhs = float(np.sum(Lw * d.astype(np.float64))), float(np.sum(w.astype(np.float64) * LTd))
    print("\n[adjoint dot product 500x1500 nt=700] <Lw,d> = %.9e  <w,L^T d> = %.9e  rel diff %.2e" % (lhs, rhs, abs(lhs - rhs) / abs(lhs)))
    assert abs(lhs - rhs) <= 1e-4 * abs(lhs)


def test_gradient_is_the_derivative_of_the_misfit_at_500x1500(ac):
    """Directional derivative through the CUDA path at 500 x 1500: (J(v + e dv) - J(v - e dv)) / 2e vs <gradient, dv> with
    dv = the box-smoothed gradient scaled to 1 m/s (a direction the misfit is sensitive to) and e = 2 m/s.  The same
    experiment with the float64 oracle agrees to 6e-6 and with the float32 CPU port to 2e-6; tolerance 1e-3."""
    from scipy.ndimage import uniform_filter
    nz, nx, nt = 500, 1500, 600
    v = fo.layered_model((nz, nx), 1600.0, 3800.0, 5).astype(np.float32)
    h = 10.0
    dt = fo.stable_dt(3900.0, h, 2)
    wav = fo.ricker(nt, dt, 12.0).astype(np.float32)
    src, rec = [(4, 500)], [(4, x) for x in range(0, nx, 2)]
    prop = ac.Propagator2D((nz, nx), h, dt, nabs=30)
    prop.set_geometry(src, rec)
    prop.set_model(v * np.float32(1.03))
    obs = prop.forward(wav).clone()
    prop.set_model(v)
    J, g, _ = prop.gradient(wav, obs)
    g = g.cpu().numpy().astype(np.float64)
    dv = uniform_filter(g, 9)
    dv = (dv / np.abs(dv).max()).astype(np.float32)
    eps = 2.0
    Js = []
    for s in (+1.0, -1.0):
        prop.set_model(v + np.float32(s * eps) * dv)
        Js.append(ac.misfit(prop.forward(wav), obs))
    prop.close()
    fd = (Js[0] - Js[1]) / (2 * eps)
    an = float(np.sum(g * dv))
    print("\n[directional derivative 500x1500 nt=600] J %.6e  finite difference %.6e  <grad,dv> %.6e  rel diff %.2e" % (J, fd, an, abs(fd - an) / abs(fd)))
    assert abs(fd - an) <= 1e-3 * abs(fd)
