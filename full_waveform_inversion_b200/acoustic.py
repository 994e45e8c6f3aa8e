"""Track B host layer: acoustic finite-difference forward model, misfit, gradient and model update.

The reference has no such code (SURVEY 0); BASELINE.json's north_star asks for these entry points
("forward model to synthetic traces, misfit, gradient, model update").  The numerical specification
is frozen in ``oracle/fd_oracle.py`` (B1-B4) and every function here cites it.  All arithmetic runs in
the sm_100a kernels of ``csrc/fd2d.cu`` / ``csrc/fd3d.cu`` through the C ABI; torch tensors only carry
device buffers, and ``torch.distributed`` (NCCL) carries the one collective: the gradient all-reduce
over shots.

Conventions: velocity grids are (nz, nx) [2-D] or (nz, ny, nx) [3-D] float32, x contiguous;
a shot is ``(src, rec)`` with integer index arrays of shape (n, ndim) in (z[, y], x) order, or float positions in cell
units (spec B7, tests/offgrid_reference.py: a point between cells is a short list of weighted cells);
wavelets are (nt,) or (nt, nsrc); traces are (nt, nrec), time-major; a velocity perturbation dv is grid-shaped.
`free_surface=True` makes grid row (plane) z = 0 a pressure-free surface (spec B6, tests/free_surface_reference.py):
the field is mirrored oddly above it, the sponge leaves that face undamped, and sources and receivers need z >= 1.
"""
from __future__ import annotations

import contextlib
import ctypes
import math
from ctypes import POINTER, c_double, c_float, c_int, c_int64, c_uint64, c_void_p

import numpy as np
import torch

from . import _lib
from ._lib import check, current_stream, ptr

_lib.register({
    "fwi_fd2d_create": (c_int, [c_int, c_int, c_int, c_float, c_float, c_int, c_float, POINTER(c_void_p)]),
    "fwi_fd2d_destroy": (c_int, [c_void_p]),
    "fwi_fd2d_set_tile": (c_int, [c_void_p, c_int, c_int]),
    "fwi_fd2d_set_graphs": (c_int, [c_void_p, c_int]),
    "fwi_fd2d_set_tb2": (c_int, [c_void_p, c_int]),
    "fwi_fd2d_set_free_surface": (c_int, [c_void_p, c_int]),
    "fwi_fd2d_set_memory_limit": (c_int, [c_void_p, c_uint64]),
    "fwi_fd2d_set_model": (c_int, [c_void_p, c_void_p, c_void_p]),
    "fwi_fd2d_set_geometry": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "fwi_fd2d_forward": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "fwi_fd2d_wavefield": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "fwi_fd2d_gradient": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, POINTER(c_double), c_void_p]),
    "fwi_fd2d_born": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "fwi_fd2d_gauss_newton": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "fwi_fd2d_launch_count": (c_int64, [c_void_p]),
    "fwi_fd3d_create": (c_int, [c_int, c_int, c_int, c_int, c_float, c_float, c_int, c_float, POINTER(c_void_p)]),
    "fwi_fd3d_set_geometry": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "fwi_fd2d_set_positions": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "fwi_fd3d_set_positions": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "fwi_fd_set_profiles": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "fwi_fd_field_ptr": (c_void_p, [c_void_p, c_int]),
    "fwi_fd_pitch": (c_int, [c_void_p]),
    "fwi_fd_reserve_snapshots": (c_int, [c_void_p, c_int]),
    "fwi_fd_reserve": (c_int, [c_void_p, c_int, c_int]),
    "fwi_fd_reset": (c_int, [c_void_p, c_int, c_void_p]),
    "fwi_fd_step": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "fwi_fd_finalize_gradient": (c_int, [c_void_p, c_void_p, c_void_p]),
    "fwi_fd_slab_info": (c_int, [c_void_p, c_void_p, c_void_p]),
    "fwi_fd_slab_connect": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "fwi_fd_slab_error": (c_int, [c_void_p, POINTER(c_int)]),
    "fwi_fd_slab_set_timeout": (c_int, [c_void_p, c_double]),
    "fwi_fd_slab_clear_error": (c_int, [c_void_p]),
    "fwi_fd_slab_connect_local": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "fwi_fd_misfit": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_double), c_void_p]),
    "fwi_fd_model_update": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_void_p]),
    "fwi_fd_absmax": (c_int, [c_void_p, c_int64, POINTER(c_float), c_void_p]),
})

COEF = (-205.0 / 72.0, 8.0 / 5.0, -1.0 / 5.0, 8.0 / 315.0, -1.0 / 560.0)


def ricker(nt, dt, f0, t0=None):
    """Ricker wavelet (fd_oracle.ricker): (1 - 2a) exp(-a), a = (pi f0 (t - t0))^2, t0 = 1.2/f0."""
    t0 = 1.2 / f0 if t0 is None else t0
    a = (math.pi * f0 * (np.arange(nt) * dt - t0)) ** 2
    return ((1.0 - 2.0 * a) * np.exp(-a)).astype(np.float32)


def stable_dt(vmax, h, ndim, cfl=0.6):
    """Time step inside the leapfrog stability limit of the 8th-order stencil (fd_oracle.stable_dt)."""
    rho = ndim * (abs(COEF[0]) + 2.0 * sum(abs(c) for c in COEF[1:]))
    return cfl * 2.0 * h / (vmax * math.sqrt(rho))


def _dev_f32(x, device):
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.float32).contiguous()
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).to(device)


def _points(pts, ndim, dtype=np.int32):
    a = np.ascontiguousarray(np.asarray(pts, dtype=dtype).reshape(-1, ndim))
    return [np.ascontiguousarray(a[:, k]) for k in range(ndim)]


def _off_grid(*point_sets):
    """True if any of the point sets is a non-empty array of a floating dtype: positions in cell units (spec B7)."""
    for pts in point_sets:
        a = pts.cpu().numpy() if isinstance(pts, torch.Tensor) else np.asarray(pts)
        if a.size and a.dtype.kind == "f":
            return True
    return False


class Propagator:
    """One GPU's propagator plan (wraps ``fwi_fd2d``; 2-D or 3-D by the length of `shape`): model, sponge,
    wavefields, TMA descriptors, cached CUDA graphs.  `free_surface`: z = 0 is a free surface (spec B6)."""

    def __init__(self, shape, h, dt, nabs=20, alpha=0.3, device=None, tile=None, memory_limit=0, graphs=True, tb2=None,
                 free_surface=False):
        self._lib = _lib.require_gpu()
        self.shape = tuple(int(n) for n in shape)
        self.ndim = len(self.shape)
        if self.ndim not in (2, 3):
            raise ValueError("grid must be 2-D (nz, nx) or 3-D (nz, ny, nx)")
        self.nz, self.nx = self.shape[0], self.shape[-1]
        self.h, self.dt = float(h), float(dt)
        self.device = torch.cuda.current_device() if device is None else int(device)
        self._h = c_void_p()
        if self.ndim == 2:
            check(self._lib.fwi_fd2d_create(self.device, self.nz, self.nx, self.h, self.dt, int(nabs), float(alpha),
                                            ctypes.byref(self._h)))
        else:
            check(self._lib.fwi_fd3d_create(self.device, self.nz, self.shape[1], self.nx, self.h, self.dt, int(nabs),
                                            float(alpha), ctypes.byref(self._h)))
        if tile is not None:
            check(self._lib.fwi_fd2d_set_tile(self._h, int(tile[0]), int(tile[1])))
        if tb2 is not None:
            check(self._lib.fwi_fd2d_set_tb2(self._h, int(tb2)))
        if memory_limit:
            check(self._lib.fwi_fd2d_set_memory_limit(self._h, int(memory_limit)))
        if not graphs:
            check(self._lib.fwi_fd2d_set_graphs(self._h, 0))
        self.free_surface = bool(free_surface)
        if self.free_surface:
            check(self._lib.fwi_fd2d_set_free_surface(self._h, 1))
        self.nsrc = self.nrec = 0

    @property
    def torch_device(self):
        return torch.device("cuda", self.device)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.fwi_fd2d_destroy(self._h)
            self._h = None

    __del__ = close

    def set_memory_limit(self, nbytes):
        check(self._lib.fwi_fd2d_set_memory_limit(self._h, int(nbytes)))

    def set_model(self, v):
        v = _dev_f32(v, self.torch_device)
        if tuple(v.shape) != self.shape:
            raise ValueError("velocity grid %s does not match the plan %s" % (tuple(v.shape), self.shape))
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd2d_set_model(self._h, ptr(v), current_stream()))
        self._v = v

    def set_geometry(self, src, rec):
        """Sources and receivers as (n, ndim) arrays in (z[, y], x) order.  Integer arrays (or lists of ints) are grid indices
        (B2).  If either is a floating array, both are positions in cell units (spec B7): each coordinate in [0, n - 1],
        z > 0 with a free surface; a point between cells injects into / samples a weighted list of cells."""
        if _off_grid(src, rec):
            s_ = _points(src, self.ndim, np.float64)
            r_ = _points(rec, self.ndim, np.float64)
            fn = self._lib.fwi_fd2d_set_positions if self.ndim == 2 else self._lib.fwi_fd3d_set_positions
        else:
            s_ = _points(src, self.ndim)
            r_ = _points(rec, self.ndim)
            fn = self._lib.fwi_fd2d_set_geometry if self.ndim == 2 else self._lib.fwi_fd3d_set_geometry
        check(fn(self._h, len(s_[0]), *[a.ctypes.data_as(c_void_p) for a in s_],
                 len(r_[0]), *[a.ctypes.data_as(c_void_p) for a in r_]))
        self.nsrc, self.nrec = len(s_[0]), len(r_[0])

    def _wavelet(self, wavelet):
        w = _dev_f32(wavelet, self.torch_device)
        if w.ndim == 1:
            w = w[:, None].expand(-1, self.nsrc).contiguous()
        if w.shape[1] != self.nsrc:
            raise ValueError("wavelet has %d columns but the shot has %d sources" % (w.shape[1], self.nsrc))
        return w if w.is_contiguous() else w.contiguous()

    def forward(self, wavelet, out=None):
        """nt leapfrog steps from rest -> traces (nt, nrec) device tensor (fd_oracle.Problem.forward)."""
        w = self._wavelet(wavelet)
        nt = w.shape[0]
        traces = out if out is not None else torch.empty((nt, self.nrec), dtype=torch.float32, device=self.torch_device)
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd2d_forward(self._h, ptr(w), nt, ptr(traces), current_stream()))
        return traces

    def wavefield(self, which=0):
        out = torch.empty(self.shape, dtype=torch.float32, device=self.torch_device)
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd2d_wavefield(self._h, which, ptr(out), current_stream()))
        return out

    def gradient(self, wavelet, observed, grad=None, want_traces=False, want_misfit=True, traces_out=None):
        """One shot: (J, grad (nz,nx) accumulated into `grad`, traces|None)  (fd_oracle.Problem.misfit_and_gradient).
        `traces_out`: caller-owned (nt, nrec) float32 buffer for the synthetics (no allocation inside the call)."""
        w = self._wavelet(wavelet)
        nt = w.shape[0]
        obs = _dev_f32(observed, self.torch_device)
        if tuple(obs.shape) != (nt, self.nrec):
            raise ValueError("observed traces %s do not match (nt=%d, nrec=%d)" % (tuple(obs.shape), nt, self.nrec))
        if grad is None:
            grad = torch.zeros(self.shape, dtype=torch.float32, device=self.torch_device)
        traces = traces_out if traces_out is not None else \
            (torch.empty((nt, self.nrec), dtype=torch.float32, device=self.torch_device) if want_traces else None)
        J = c_double(0.0)
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd2d_gradient(self._h, ptr(w), ptr(obs), nt, ptr(grad), ptr(traces),
                                              ctypes.byref(J) if want_misfit else None, current_stream()))
        return (J.value if want_misfit else None), grad, traces

    def _grid_arg(self, x, name):
        t = _dev_f32(x, self.torch_device)
        if tuple(t.shape) != self.shape:
            raise ValueError("%s has shape %s, expected the grid shape %s" % (name, tuple(t.shape), self.shape))
        return t

    def _out_arg(self, t, shape, name):
        if not (isinstance(t, torch.Tensor) and tuple(t.shape) == tuple(shape) and t.dtype == torch.float32
                and t.is_contiguous() and t.device == self.torch_device):
            raise ValueError("%s must be a contiguous float32 tensor of shape %s on %s" % (name, tuple(shape), self.torch_device))
        return t

    def born(self, wavelet, dv, out=None, want_traces=False):
        """Born (linearised) traces J dv for the velocity perturbation `dv` (grid-shaped) -> (dtraces (nt, nrec), background
        traces | None)  (spec B5, tests/born_reference.py born).  `out`: caller-owned (nt, nrec) float32 buffer for J dv."""
        w = self._wavelet(wavelet)
        nt = w.shape[0]
        dv = self._grid_arg(dv, "dv")
        dtr = torch.empty((nt, self.nrec), dtype=torch.float32, device=self.torch_device) if out is None else \
            self._out_arg(out, (nt, self.nrec), "out")
        traces = torch.empty((nt, self.nrec), dtype=torch.float32, device=self.torch_device) if want_traces else None
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd2d_born(self._h, ptr(w), ptr(dv), nt, ptr(dtr), ptr(traces), current_stream()))
        return dtr, traces

    def gauss_newton(self, wavelet, dv, hv=None, want_dtraces=False):
        """Gauss-Newton Hessian-vector product: hv (grid-shaped, accumulated into `hv`) += J^T J dv -> (hv, J dv | None)
        (spec B5, tests/born_reference.py gauss_newton).  Snapshots are stored or checkpointed as in `gradient`."""
        w = self._wavelet(wavelet)
        nt = w.shape[0]
        dv = self._grid_arg(dv, "dv")
        hv = torch.zeros(self.shape, dtype=torch.float32, device=self.torch_device) if hv is None else \
            self._out_arg(hv, self.shape, "hv")
        dtr = torch.empty((nt, self.nrec), dtype=torch.float32, device=self.torch_device) if want_dtraces else None
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd2d_gauss_newton(self._h, ptr(w), ptr(dv), nt, ptr(hv), ptr(dtr), current_stream()))
        return hv, dtr

    # ---- low-level stepping (the caller drives the time loop; used by SlabPropagator) --------------------------
    def set_profiles(self, gz=None, gy=None, gx=None):
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float32) for a in (gz, gy, gx)]
        check(self._lib.fwi_fd_set_profiles(self._h, *[None if a is None else a.ctypes.data_as(c_void_p) for a in arrs]))

    def field_view(self, idx):
        """Zero-copy torch view (rows..., pitch) of wavefield buffer idx (0/1 forward pair, 4/5 adjoint pair)."""
        px = int(self._lib.fwi_fd_pitch(self._h))
        shape = self.shape[:-1] + (px,)

        class _Raw:
            pass
        raw = _Raw()
        raw.__cuda_array_interface__ = {"shape": shape, "typestr": "<f4", "version": 3,
                                        "data": (int(self._lib.fwi_fd_field_ptr(self._h, idx)), False)}
        with torch.cuda.device(self.device):
            return torch.as_tensor(raw, device=self.torch_device)

    def reserve(self, nt, gradient=True):
        """Allocate the buffers of a forward / gradient over nt steps now (allocations synchronise the device)."""
        check(self._lib.fwi_fd_reserve(self._h, int(nt), 1 if gradient else 0))

    def reserve_snapshots(self, nsteps):
        check(self._lib.fwi_fd_reserve_snapshots(self._h, int(nsteps)))

    def reset(self, pair):
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd_reset(self._h, int(pair), current_stream()))

    def step(self, mode, cur, inj_row_ptr, rec_row_ptr=None, snap_index=-1):
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd_step(self._h, int(mode), int(cur), c_void_p(inj_row_ptr),
                                        None if rec_row_ptr is None else c_void_p(rec_row_ptr), int(snap_index), current_stream()))

    def finalize_gradient(self, grad):
        with torch.cuda.device(self.device):
            check(self._lib.fwi_fd_finalize_gradient(self._h, ptr(grad), current_stream()))

    def launch_count(self):
        return int(self._lib.fwi_fd2d_launch_count(self._h))


Propagator2D = Propagator
Propagator3D = Propagator


def sponge_profile(n, nabs, alpha, free_surface=False):
    """1-D Cerjan profile (fd_oracle.sponge_profile); `free_surface` leaves index 0's face undamped (spec B6)."""
    prof = np.ones(n, dtype=np.float64)
    for i in range(min(nabs, n)):
        val = math.exp(-((alpha * (nabs - i) / nabs) ** 2))
        if not free_surface:
            prof[i] = min(prof[i], val)
        prof[n - 1 - i] = min(prof[n - 1 - i], val)
    return prof.astype(np.float32)


class SlabPropagator:
    """Large grids split into z slabs over the ranks of the default process group (BASELINE config 4).

    Every rank owns a contiguous range of z planes plus a 4-plane ghost zone towards each neighbour.
    3-D (default, `p2p`): compute and halo exchange are ONE kernel.  The neighbours' wavefield arenas are mapped with
    CUDA IPC; the step kernel computes the owned planes and stores its 4 boundary planes straight into the neighbours'
    ghost planes over NVLink.  Both boundaries are computed in the first iterations of their CTAs (the last z chunk
    marches downwards), so the transfer and the neighbours' wait hide behind the interior planes.  Step ids live in
    device memory, so the whole forward / gradient time loop of a rank is one CUDA-graph replay of the plan's ordinary
    `forward` / `gradient` (same checkpointing when the snapshots do not fit, per rank); no collective per step.
    Fallback / 2-D (`p2p=False`): the ordinary step kernel runs on the local grid and the boundary planes are exchanged
    with NCCL send/recv, the loop captured as a CUDA graph (every w_n held in HBM).
    Either way the owned planes are bit-identical to a single-GPU run.  With `free_surface`, global z = 0 is a free
    surface (spec B6): every rank slices the global profile, and only rank 0's plan mirrors the field above z = 0."""

    HALO = 4

    def __init__(self, shape, h, dt, nabs=20, alpha=0.3, device=None, use_graphs=True, p2p=None, memory_limit=0,
                 free_surface=False):
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("SlabPropagator needs an initialised torch.distributed process group")
        self.dist = dist
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.shape = tuple(int(n) for n in shape)
        nz = self.shape[0]
        if nz < self.world * 2 * self.HALO:
            raise ValueError("grid has too few z planes (%d) for %d slabs" % (nz, self.world))
        base, rem = divmod(nz, self.world)
        counts = [base + (1 if r < rem else 0) for r in range(self.world)]
        self.z0 = sum(counts[: self.rank])
        self.n_own = counts[self.rank]
        self.up = self.HALO if self.rank > 0 else 0
        self.down = self.HALO if self.rank < self.world - 1 else 0
        self.local_shape = (self.n_own + self.up + self.down,) + self.shape[1:]
        device = torch.cuda.current_device() if device is None else device
        # 3-D slabs default to the fused mode (boundary planes pushed over NVLink peer memory by the step kernel
        # itself); p2p=False forces the NCCL send/recv exchange, which is also the fallback if IPC mapping fails.
        self.p2p = (p2p is None or bool(p2p)) and len(self.shape) == 3 and self.world > 1
        self.prop = Propagator(self.local_shape, h, dt, nabs, alpha, device, graphs=bool(use_graphs and self.p2p),
                               memory_limit=memory_limit, free_surface=bool(free_surface) and self.rank == 0)
        gz = sponge_profile(nz, nabs, alpha, free_surface)[self.z0 - self.up: self.z0 + self.n_own + self.down]
        self.prop.set_profiles(gz=gz)
        self.fields = [self.prop.field_view(i) for i in range(8)]
        self.nsrc = self.nrec = 0
        self.use_graphs = use_graphs
        self._graphs = {}
        if self.p2p:
            ok = torch.ones(1, device=self.prop.torch_device)
            try:
                self._connect_peers()
            except Exception:
                if p2p:
                    raise
                ok.zero_()
            self.dist.all_reduce(ok, op=self.dist.ReduceOp.MIN)
            if ok.item() == 0:
                raise RuntimeError("peer-memory slab mode could not be set up on every rank; pass p2p=False to use NCCL")

    @property
    def local_range(self):
        """(lo, hi): the global z planes this rank keeps (owned + ghosts) - what `set_model(..., local=True)` expects."""
        return self.z0 - self.up, self.z0 + self.n_own + self.down

    def _connect_peers(self):
        """Fused mode: map the neighbours' wavefield arenas (CUDA IPC over NVLink) so that the step kernel itself stores
        its boundary planes into their ghost planes; no collective call per step."""
        lib = self.prop._lib
        handle = (ctypes.c_ubyte * 64)()
        offs = (ctypes.c_uint64 * 9)()
        check(lib.fwi_fd_slab_info(self.prop._h, ctypes.cast(handle, c_void_p), ctypes.cast(offs, c_void_p)))
        mine = (bytes(handle), list(offs), self.local_shape[0])
        infos = [None] * self.world
        self.dist.all_gather_object(infos, mine)

        def pack(info):
            if info is None:
                return None, None
            hb = (ctypes.c_ubyte * 64).from_buffer_copy(info[0])
            ob = (ctypes.c_uint64 * 9)(*info[1])
            return hb, ob
        up = infos[self.rank - 1] if self.up else None
        dn = infos[self.rank + 1] if self.down else None
        uh, uo = pack(up)
        dh, do = pack(dn)
        self._peer_keepalive = (uh, uo, dh, do)
        up_ghost_z = (up[2] - self.HALO) if up else 0
        check(lib.fwi_fd_slab_connect(self.prop._h, self.up, self.up + self.n_own,
                                      None if uh is None else ctypes.cast(uh, c_void_p), None if uo is None else ctypes.cast(uo, c_void_p),
                                      up_ghost_z,
                                      None if dh is None else ctypes.cast(dh, c_void_p), None if do is None else ctypes.cast(do, c_void_p)))
        self.dist.barrier()

    def set_timeout(self, milliseconds):
        """Bound on a step kernel's wait for its neighbour (fused mode; default 2 s)."""
        check(self.prop._lib.fwi_fd_slab_set_timeout(self.prop._h, float(milliseconds)))

    def check_peers(self):
        """Fused mode: raise ON EVERY RANK if any rank's launch timed out waiting for a neighbour (the kernels then
        returned without computing, so results are invalid); the flag is cleared so the propagator can be reused."""
        if not self.p2p:
            return
        e = c_int(0)
        check(self.prop._lib.fwi_fd_slab_error(self.prop._h, ctypes.byref(e)))
        flag = torch.tensor([float(e.value)], device=self.prop.torch_device)
        self.dist.all_reduce(flag, op=self.dist.ReduceOp.MAX)
        if flag.item():
            check(self.prop._lib.fwi_fd_slab_clear_error(self.prop._h))
            self.dist.barrier()
            raise RuntimeError("slab halo exchange: a step kernel timed out waiting for its neighbour (rank %d saw it: %s); "
                               "the results of this call are invalid" % (self.rank, bool(e.value)))

    def close(self):
        # captured graphs hold NCCL work: drop them (and drain the device) BEFORE the process group goes away,
        # otherwise communicator teardown can hang
        torch.cuda.synchronize()
        self._graphs = {}
        torch.cuda.synchronize()
        if self.p2p:
            self.dist.barrier()          # nobody unmaps an arena a neighbour's kernel may still be writing into
        self.prop.close()

    @property
    def own(self):
        return slice(self.up, self.up + self.n_own)

    def set_model(self, v, local=False):
        """v: the GLOBAL velocity grid (host or device), of which every rank keeps its slab (+ ghosts); or, with
        `local=True`, just this rank's planes `local_range` - grids that need slabs do not fit one GPU or one host array."""
        if local:
            if tuple(v.shape) != self.local_shape:
                raise ValueError("local model %s does not match this rank's slab %s" % (tuple(v.shape), self.local_shape))
            self.prop.set_model(v)
        else:
            lo, hi = self.local_range
            self.prop.set_model(v[lo:hi])

    def set_geometry(self, src, rec):
        if _off_grid(src, rec):
            # a point's taps may straddle two slabs, and a rank's residual would miss the part another rank samples
            raise ValueError("SlabPropagator takes integer grid indices only; off-grid positions need a single-GPU Propagator")
        ndim = len(self.shape)
        src = np.asarray(src, dtype=np.int64).reshape(-1, ndim)
        rec = np.asarray(rec, dtype=np.int64).reshape(-1, ndim)

        def mine(p):
            keep = np.nonzero((p[:, 0] >= self.z0) & (p[:, 0] < self.z0 + self.n_own))[0]
            loc = p[keep].copy()
            loc[:, 0] += self.up - self.z0
            return keep, loc
        src_ids, s_loc = mine(src)
        rec_ids, r_loc = mine(rec)
        self.prop.set_geometry(s_loc, r_loc)            # a rejected geometry raises here and leaves the rank's state as it was
        self.src_ids, self.rec_ids = src_ids, rec_ids
        self.nsrc_global, self.nrec_global = len(src), len(rec)
        self._graphs = {}                               # captured loops hold the old list sizes

    def _exchange(self, idx):
        """NCCL mode: refresh the ghost planes of wavefield buffer idx from the neighbours' boundary planes."""
        f, H, ops = self.fields[idx], self.HALO, []
        n = f.shape[0]
        P2P = self.dist.P2POp
        if self.up:
            ops += [P2P(self.dist.isend, f[H:2 * H], self.rank - 1), P2P(self.dist.irecv, f[0:H], self.rank - 1)]
        if self.down:
            ops += [P2P(self.dist.isend, f[n - 2 * H: n - H], self.rank + 1), P2P(self.dist.irecv, f[n - H: n], self.rank + 1)]
        if ops:
            for req in self.dist.batch_isend_irecv(ops):
                req.wait()

    def _wavelet_local(self, wavelet):
        w = _dev_f32(wavelet, self.prop.torch_device)
        if w.ndim == 1:
            w = w[:, None].expand(-1, self.nsrc_global)
        if self.p2p:
            return w[:, torch.as_tensor(self.src_ids, device=w.device)].contiguous()          # (nt, 0) on a rank without sources
        return w[:, torch.as_tensor(self.src_ids, device=w.device)].contiguous() if len(self.src_ids) else \
            torch.zeros((w.shape[0], 1), dtype=torch.float32, device=w.device)

    def _loop(self, nt, mode, pair, inj, out, snap_offset, reverse):
        self.prop.reset(pair)
        cur = 0
        for k in range(nt):
            n = nt - 1 - k if reverse else k
            self.prop.step(mode, cur, inj.data_ptr() + n * inj.shape[1] * 4,
                           None if out is None or out.shape[1] == 0 else out.data_ptr() + n * out.shape[1] * 4,
                           snap_index=n + snap_offset if mode else -1)
            cur ^= 1
            self._exchange(4 * pair + cur)

    def _run(self, nt, mode, pair, inj, out, snap_offset=0, reverse=False):
        """NCCL mode: nt steps + halo exchanges.  The whole loop (step kernels and NCCL send/recv) is captured once per
        (nt, mode) into a CUDA graph over persistent staging buffers and replayed, which removes the ~0.4 ms of
        host + NCCL launch latency per step; falls back to eager stepping if capture is not possible."""
        if not self.use_graphs:
            return self._loop(nt, mode, pair, inj, out, snap_offset, reverse)
        key = (nt, mode, pair, inj.shape[1], -1 if out is None else out.shape[1], snap_offset, reverse)
        ent = self._graphs.get(key)
        if ent is None:
            try:
                inj_s = torch.empty_like(inj)
                out_s = None if out is None else torch.empty_like(out)
                self._exchange(4 * pair)                       # NCCL communicators / P2P channels must exist before capture
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._loop(nt, mode, pair, inj_s, out_s, snap_offset, reverse)
                ent = (g, inj_s, out_s)
                self._graphs[key] = ent
            except Exception:
                self.use_graphs = False
                torch.cuda.synchronize()
                return self._loop(nt, mode, pair, inj, out, snap_offset, reverse)
        g, inj_s, out_s = ent
        inj_s.copy_(inj)
        g.replay()
        if out is not None:
            out.copy_(out_s)

    def _gather_traces(self, local, nt):
        full = torch.zeros((nt, self.nrec_global), dtype=torch.float32, device=local.device)
        if len(self.rec_ids):
            full[:, torch.as_tensor(self.rec_ids, device=local.device)] = local
        self.dist.all_reduce(full)
        return full

    def forward(self, wavelet, gather=True):
        """Traces (nt, nrec) of the whole survey on every rank (`gather=False`: this rank's receivers only)."""
        w = self._wavelet_local(wavelet)
        nt = w.shape[0]
        if self.p2p:
            local = self.prop.forward(w)
            self.check_peers()
        else:
            local = torch.zeros((nt, len(self.rec_ids)), dtype=torch.float32, device=w.device)
            self._run(nt, 0, 0, w, local)
        return self._gather_traces(local, nt) if gather else local

    def gradient(self, wavelet, observed, gather=True):
        """(J, gradient of this rank's own planes (n_own, ...), traces).  Fused mode: the plan's ordinary gradient on the
        slab - w_n held in HBM, or checkpointed per rank when `memory_limit` / free memory says so."""
        w = self._wavelet_local(wavelet)
        nt = w.shape[0]
        dev = w.device
        obs = _dev_f32(observed, dev)
        mine = obs[:, torch.as_tensor(self.rec_ids, device=dev)].contiguous()       # gather = data movement only
        if self.p2p:
            Jl, grad, local = self.prop.gradient(w, mine, want_traces=True)
            self.check_peers()
            J = torch.tensor([Jl], dtype=torch.float64, device=dev)
            self.dist.all_reduce(J)
            return float(J.item()), grad[self.own], (self._gather_traces(local, nt) if gather else local)
        self.prop.reserve_snapshots(nt)
        local = torch.zeros((nt, max(1, len(self.rec_ids))), dtype=torch.float32, device=dev)[:, : len(self.rec_ids)].contiguous()
        self._run(nt, 1, 0, w, local)
        if len(self.rec_ids):
            res = torch.empty_like(local)
            Jl = c_double(0.0)
            with torch.cuda.device(dev):
                check(self.prop._lib.fwi_fd_misfit(ptr(local), ptr(mine), local.numel(), ptr(res), ctypes.byref(Jl), current_stream()))
            J = torch.tensor([Jl.value], dtype=torch.float64, device=dev)
        else:
            res = torch.zeros((nt, 1), dtype=torch.float32, device=dev)
            J = torch.zeros(1, dtype=torch.float64, device=dev)
        self.dist.all_reduce(J)
        self._run(nt, 2, 1, res, None, reverse=True)
        grad = torch.zeros(self.local_shape, dtype=torch.float32, device=dev)
        self.prop.finalize_gradient(grad)
        return float(J.item()), grad[self.own], (self._gather_traces(local, nt) if gather else local)


# ------------------------------------------------------------------------------------------------ entry points
def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


def shard_shots(n_shots, world, rank):
    """Shots owned by `rank`: round-robin (shot i -> rank i % world), so every rank gets work when n >= world."""
    return list(range(rank, n_shots, world))


def _shard(n_shots, allreduce, shot_ids):
    """(process group to sum over or None, indices of the shots this rank runs).  With `shot_ids` the caller passed
    just this rank's shots, so it runs all of them."""
    dist = _dist() if allreduce else None
    if shot_ids is not None or not dist:
        return dist, range(n_shots)
    return dist, shard_shots(n_shots, dist.get_world_size(), dist.get_rank())


@contextlib.contextmanager
def _plan(v, h, dt, nabs, alpha, device, propagator, free_surface):
    """The caller's `propagator`, or a new plan that is closed on exit; either way with the model v set."""
    prop = propagator or Propagator(tuple(v.shape), h, dt, nabs, alpha, device, free_surface=free_surface)
    try:
        prop.set_model(v)
        yield prop
    finally:
        if propagator is None:
            prop.close()


def forward_model(v, h, dt, shots, wavelet, nabs=20, alpha=0.3, device=None, propagator=None, free_surface=False):
    """Forward model every shot -> list of (nt, nrec) device tensors (fd_oracle.Problem.forward per shot)."""
    with _plan(v, h, dt, nabs, alpha, device, propagator, free_surface) as prop:
        out = []
        for src, rec in shots:
            prop.set_geometry(src, rec)
            out.append(prop.forward(wavelet))
        return out


def born_model(v, h, dt, shots, wavelet, dv, nabs=20, alpha=0.3, device=None, propagator=None, free_surface=False):
    """Born traces J dv of every shot -> list of (nt, nrec) device tensors (spec B5 per shot, tests/born_reference.py)."""
    with _plan(v, h, dt, nabs, alpha, device, propagator, free_surface) as prop:
        out = []
        for src, rec in shots:
            prop.set_geometry(src, rec)
            out.append(prop.born(wavelet, dv)[0])
        return out


def gauss_newton_product(v, h, dt, shots, wavelet, dv, nabs=20, alpha=0.3, device=None, propagator=None, allreduce=True,
                         shot_ids=None, free_surface=False):
    """Gauss-Newton Hessian-vector product summed over shots, sum_s J_s^T J_s dv -> grid-shaped device tensor.

    Under torch.distributed the shots are sharded round-robin over the ranks and the product is summed with ONE
    all-reduce, as in `gradient`; with `shot_ids`, `shots` holds just this rank's shots."""
    dist, ids = _shard(len(shots), allreduce, shot_ids)
    with _plan(v, h, dt, nabs, alpha, device, propagator, free_surface) as prop:
        hv = torch.zeros(tuple(v.shape), dtype=torch.float32, device=prop.torch_device)
        for i in ids:
            prop.set_geometry(*shots[i])
            prop.gauss_newton(wavelet, dv, hv=hv)
        if dist:
            dist.all_reduce(hv)
        return hv


def misfit(traces, observed):
    """J = 1/2 sum (traces - observed)^2 over all shots (fd_oracle.misfit)."""
    lib = _lib.require_gpu()
    if isinstance(traces, torch.Tensor):
        traces, observed = [traces], [observed]
    total = 0.0
    for t, o in zip(traces, observed):
        t = _dev_f32(t, t.device if isinstance(t, torch.Tensor) and t.is_cuda else torch.device("cuda"))
        o = _dev_f32(o, t.device)
        res = torch.empty_like(t)
        J = c_double(0.0)
        with torch.cuda.device(t.device):
            check(lib.fwi_fd_misfit(ptr(t), ptr(o), t.numel(), ptr(res), ctypes.byref(J), current_stream()))
        total += J.value
    return total


def gradient(v, h, dt, shots, wavelet, observed, nabs=20, alpha=0.3, device=None, propagator=None, allreduce=True,
             shot_ids=None, free_surface=False):
    """Misfit and dJ/dv summed over shots -> (J, grad (grid-shaped device tensor)).

    Under torch.distributed the shots are sharded round-robin over the ranks (one GPU each) and the gradient and
    the misfit are summed with ONE all-reduce over NCCL (BASELINE config 3); `shots`/`observed` hold all shots on
    every rank, or - with `shot_ids` - just this rank's."""
    dist, ids = _shard(len(shots), allreduce, shot_ids)
    with _plan(v, h, dt, nabs, alpha, device, propagator, free_surface) as prop:
        grad = torch.zeros(tuple(v.shape), dtype=torch.float32, device=prop.torch_device)
        J = 0.0
        for i in ids:
            prop.set_geometry(*shots[i])
            j, _, _ = prop.gradient(wavelet, observed[i], grad=grad)
            J += j
        if dist:
            dist.all_reduce(grad)                       # the one collective of an FWI gradient: fp32, in place over NCCL
            Jt = torch.tensor([J], dtype=torch.float64, device=grad.device)
            dist.all_reduce(Jt)                         # + the misfit (one float64 scalar)
            J = float(Jt.item())
        return J, grad


def model_update(v, grad, step, vmin, vmax):
    """v <- clip(v - step * grad, vmin, vmax), in place on the device tensor (fd_oracle.model_update)."""
    lib = _lib.require_gpu()
    if not (isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == torch.float32 and v.is_contiguous()):
        raise ValueError("v must be a contiguous float32 CUDA tensor (it is updated in place)")
    g = _dev_f32(grad, v.device)
    with torch.cuda.device(v.device):
        check(lib.fwi_fd_model_update(ptr(v), ptr(g), v.numel(), float(step), float(vmin), float(vmax), current_stream()))
    return v


def absmax(x):
    lib = _lib.require_gpu()
    out = c_float(0.0)
    with torch.cuda.device(x.device):
        check(lib.fwi_fd_absmax(ptr(x), x.numel(), ctypes.byref(out), current_stream()))
    return out.value


def fwi(v0, h, dt, shots, wavelet, observed, niter, vmin, vmax, step_frac=0.02, max_backtrack=4, nabs=20, alpha=0.3,
        device=None, callback=None, free_surface=False):
    """Steepest-descent full-waveform inversion (fd_oracle.fwi, B4) -> (v, misfit history).

    Each iteration: gradient over all shots (sharded + all-reduced when distributed), step = step_frac * max|v| /
    max|grad|, halved up to `max_backtrack` times while the misfit does not decrease."""
    device = torch.cuda.current_device() if device is None else device
    dev = torch.device("cuda", device)
    v = _dev_f32(v0, dev).clone()
    dist, ids = _shard(len(shots), True, None)
    my_shots = [shots[i] for i in ids]
    my_obs = [_dev_f32(observed[i], dev) for i in ids]

    def total_misfit(vv):
        prop.set_model(vv)
        J = 0.0
        for (src, rec), obs in zip(my_shots, my_obs):
            prop.set_geometry(src, rec)
            J += misfit(prop.forward(wavelet), obs)
        if dist:
            t = torch.tensor([J], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            J = float(t.item())
        return J

    history = []
    with _plan(v, h, dt, nabs, alpha, device, None, free_surface) as prop:
        for it in range(niter):
            J, g = gradient(v, h, dt, my_shots, wavelet, my_obs, propagator=prop, shot_ids=ids)
            history.append(J)
            gmax = absmax(g)
            if gmax == 0.0:
                break
            step = step_frac * absmax(v) / gmax
            for _ in range(max_backtrack + 1):
                trial = model_update(v.clone(), g, step, vmin, vmax)
                Jt = total_misfit(trial)
                if Jt < J:
                    v = trial
                    break
                step *= 0.5
            if callback:
                callback(it, J, v)
        history.append(total_misfit(v))
        return v, history
