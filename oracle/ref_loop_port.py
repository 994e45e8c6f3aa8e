"""Timing port of the reference's per-sample Monte-Carlo loop in its DEFAULT configuration (FWI:46-71):
type `single_force_crack_no_coupling`, metric VR, un-normalised, per-trace-then-mean.

TEST INFRASTRUCTURE ONLY - used by bench.py's Track A CPU lines and by tests/.  The reference itself is a Python-2
script that cannot be imported, and /root/reference does not exist on the GPU box, so the reference arm of Track A
times THIS restatement there.  Unlike oracle/mc_oracle.py (vectorised, ~3x faster than the reference) this file keeps
the reference's OPERATION STRUCTURE, because that structure is what its speed is made of:
  * the sampler makes the same scalar NumPy / `random` calls in the same order (FWI:448-510, 320-331, 226-232, 206-208),
    so with the same seeds it produces the reference's samples bit for bit (tests/test_ref_loop_port.py replays the
    draws stored with the reference's results in tests/golden/track_a_reference.npz);
  * the forward model is the K x C double loop of slice multiply-adds (FWI:260-263);
  * the misfit is one VR call per trace, three NumPy reductions each, then np.average (FWI:664-668, 682, 512-520);
  * likelihood and Bayes normalisation as FWI:774, 811, 847-848; worker fan-out as FWI:822-830 (one OS process per
    worker), with distinct seeds per worker instead of the inherited RNG state of quirk q4.
tools/ref_port_fidelity.py measured it next to the live reference in the build container (numbers in BASELINE.md).
"""
from __future__ import annotations

import multiprocessing as mp
import random
import time

import numpy as np


def rotation_y_then_z(theta, phi):                                        # FWI:226-232, the two matrices
    ry = np.vstack(([np.cos(theta), 0., np.sin(theta)], [0., 1., 0.], [-1. * np.sin(theta), 0., np.cos(theta)]))
    rz = np.vstack(([np.cos(phi), -1. * np.sin(phi), 0.], [np.sin(phi), np.cos(phi), 0.], [0., 0., 1.]))
    return ry, rz


def rotate_tensor(full, theta, phi):                                      # FWI:226-232
    ry, rz = rotation_y_then_z(theta, phi)
    first = np.dot(ry, np.dot(full, np.transpose(ry)))
    return np.dot(rz, np.dot(first, np.transpose(rz)))


def six_from_full(full):                                                  # FWI:206-208
    return np.array([full[0, 0], full[1, 1], full[2, 2], np.sqrt(2.) * full[0, 1], np.sqrt(2.) * full[0, 2], np.sqrt(2.) * full[1, 2]])


def unit_three_vector():                                                  # FWI:320-331 / 490-493: three scalar normals
    a = np.array([np.random.normal(loc=0.0, scale=1.0), np.random.normal(loc=0.0, scale=1.0),
                  np.random.normal(loc=0.0, scale=1.0)], dtype=float)
    a = a / (np.sum(a ** 2) ** -0.5)
    return a / ((np.sum(a ** 2)) ** 0.5)


def sample_single_force_crack_uncoupled():                                # FWI:448-510
    force = np.reshape(unit_three_vector(), (3, 1))
    theta_l = np.random.uniform(-1., 1.) * np.pi / 2.
    r = random.random()
    phi_l = 0. if r <= 0.5 else np.pi / 3
    with np.errstate(divide="ignore", invalid="ignore"):
        ang = np.arctan(np.sin(phi_l) / np.sin(theta_l))
    r = random.random()
    if r > 0.25 and r <= 0.5:
        ang = ang + np.pi
    if r > 0.5 and r <= 0.75:
        ang = ang + np.pi / 2
    if r > 0.75 and r <= 1.0:
        ang = ang + 3 * np.pi / 2
    lead = (((4 * (np.sin(ang) ** 2)) + (np.cos(ang) ** 2)) ** -0.5) / np.sqrt(3.)
    crack = lead * np.vstack(([np.cos(ang) - (np.sqrt(2) * np.sin(ang)), 0., 0.],
                              [0., np.cos(ang) - (np.sqrt(2) * np.sin(ang)), 0.],
                              [0., 0., np.cos(ang) + (2. * np.sqrt(2) * np.sin(ang))]))
    a = unit_three_vector()
    theta = np.arccos(a[2])
    phi = np.arccos(a[0] / np.sin(theta))
    six = np.reshape(six_from_full(rotate_tensor(crack, theta, phi)), (6, 1))
    frac = random.random()
    return np.vstack((six * (1. - frac), force * frac)), frac


def forward_model(G, M):                                                  # FWI:253-264
    out = np.zeros(np.shape(G[:, 0, :]), dtype=float)
    for i in range(len(G[:, 0, 0])):
        for j in range(len(M)):
            out[i, :] += G[i, j, :] * M[j]
    return out


def variance_reduction(data, synth):                                      # FWI:512-520
    vr = 1. - (np.sum(np.square(data - synth)) / np.sum(np.square(data)))
    if vr < 0.:
        vr = 0.
    return vr


def similarity_per_trace_vr(d, synth):                                    # FWI:662-668, 682
    per = np.zeros(len(d[:, 0]), dtype=float)
    for k in range(len(per)):
        per[k] = variance_reduction(d[k, :], synth[k, :])
    return np.average(per)


def worker(d, G, n, amplitude, seed):
    """FWI:686-784 for the default configuration -> (MTs (9, n), L (n,), amp_frac (n,))."""
    np.random.seed(seed)
    random.seed(seed)
    MTs = np.zeros((len(G[0, :, 0]), n), dtype=float)
    sim = np.zeros(n, dtype=float)
    frac = np.zeros(n, dtype=float)
    for i in range(n):
        M, f = sample_single_force_crack_uncoupled()
        M = M * amplitude
        synth = forward_model(G, M)
        s = similarity_per_trace_vr(d, synth)
        MTs[:, i] = M[:, 0]
        sim[i] = s
        frac[i] = f
    return MTs, np.exp(-(1. - sim) / 2.), frac


def _proc(args):
    d, G, n, amplitude, seed = args
    t0 = time.perf_counter()
    out = worker(d, G, n, amplitude, seed)
    return out, time.perf_counter() - t0


def monte_carlo(d, G, num_samples, amplitude, num_processors=1, seed=0):
    """FWI:786-870 for the default configuration -> (MTs (10, N), MTp (N,), seconds of the slowest worker)."""
    per = int(num_samples / num_processors)                               # FWI:822 (the remainder is dropped there; kept)
    jobs = [(d, G, per, amplitude, seed + 1000 * p) for p in range(num_processors)]
    if num_processors == 1:
        res = [_proc(jobs[0])]
    else:
        with mp.get_context("fork").Pool(num_processors) as pool:         # one OS process per worker (FWI:824-830)
            res = pool.map(_proc, jobs)
    MTs = np.concatenate([r[0][0] for r in res], axis=1)
    L = np.concatenate([r[0][1] for r in res])
    frac = np.concatenate([r[0][2] for r in res])
    p_model = 1. / len(L)                                                 # FWI:811
    MTp = L * p_model / np.sum(p_model * L)                               # FWI:847-848
    return np.vstack((MTs, frac)), MTp, max(r[1] for r in res)           # FWI:851-852


def samples_per_second(d, G, amplitude, n_per_process, num_processors):
    """Rate of the loop itself (slowest worker's in-loop time; process start-up is excluded, as it amortises over the
    reference's 10^4 .. 10^6 samples)."""
    _, _, sec = monte_carlo(d, G, n_per_process * num_processors, amplitude, num_processors)
    return n_per_process * num_processors / sec
