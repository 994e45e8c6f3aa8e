"""Float64 reference of Born modelling and the Gauss-Newton Hessian ("spec B5"), built on oracle/fd_oracle.py's
Problem (B1-B3): its `step`, `forward(save=True)` and `adjoint`, no second stencil.  Test infrastructure only.

B5  Born / Gauss-Newton   J = d traces / d v, the exact derivative of the discrete forward B1/B2 (sponge and source
    scaling included), so the identities below hold to rounding, not to discretisation error.
    background   w_n = lap(u_n) + f_n,   u_{n+1} = g (2 u_n - g u_{n-1} + m w_n)          (B1, w_n saved)
    Born         du_{n+1} = g (2 du_n - g du_{n-1} + m lap(du_n) + dm w_n),   du_0 = du_{-1} = 0
                 dtrace[n, r] = du_{n+1}[rec_r]   (= J dv)
                 dm = (2 m / v) dv   (the velocity parameterisation of dJ/dv = (2 / v) I, B3)
    Hessian      H dv = J^T J dv = (2 / v) * adjoint(J dv, ws): the B3 adjoint run on the Born traces as its residual.
"""
from __future__ import annotations

import numpy as np


def _born(p, wavelet, dv):
    traces, ws = p.forward(wavelet, save=True)
    dm = 2.0 * p.m * np.asarray(dv, dtype=p.dtype) / p.v
    cur = np.zeros_like(p.v)     # du_n
    old = np.zeros_like(p.v)     # du_{n-1}
    dtraces = np.zeros_like(traces)
    for n in range(len(ws)):
        new, _ = p.step(cur, old)
        new = new + p.g * dm * ws[n]
        dtraces[n] = new[p.rec]
        old, cur = cur, new
    return dtraces, traces, ws


def born(p, wavelet, dv):
    """Born traces J dv (nt, nrec) and the background traces of the fd_oracle.Problem `p`, for a grid-shaped dv."""
    dtraces, traces, _ = _born(p, wavelet, dv)
    return dtraces, traces


def gauss_newton(p, wavelet, dv):
    """Gauss-Newton Hessian-vector product H dv = J^T J dv (grid-shaped) of the fd_oracle.Problem `p`."""
    dtraces, _, ws = _born(p, wavelet, dv)
    return (2.0 / p.v) * p.adjoint(dtraces, ws)
