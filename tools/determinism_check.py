"""Debug helper: is the 2-D forward bitwise reproducible, and exactly linear under a power-of-two scaling?"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from full_waveform_inversion_b200 import acoustic as ac
from oracle import fd_oracle as fo

nz, nx, nt = 1000, 3000, 600
v = torch.tensor(fo.layered_model((nz, nx), 1500.0, 4500.0, 6), dtype=torch.float32)
dt = fo.stable_dt(4500.0, 10.0, 2)
wav = fo.ricker(nt, dt, 12.0).astype(np.float32)
for kw in (dict(tile=(28, 4)), dict(tile=(28, 4), graphs=False), dict(tile=(32, 4))):
    prop = ac.Propagator2D((nz, nx), 10.0, dt, nabs=40, **kw)
    prop.set_model(v)
    prop.set_geometry([(40, 700)], [(50, 715), (45, 705), (300, 900)])
    a = prop.forward(wav).cpu().numpy()
    b = prop.forward(wav).cpu().numpy()
    c = prop.forward(2.0 * wav).cpu().numpy()
    wa = prop.wavefield(0).cpu().numpy()
    print(kw, "repeat max diff", np.abs(a - b).max(), " x2 max diff", np.abs(c.astype(np.float64) - 2.0 * a).max(),
          "max|a|", np.abs(a).max(), "first bad rows", np.nonzero(np.abs(c.astype(np.float64) - 2.0 * a).max(1) > 0)[0][:5])
    d = np.abs(c.astype(np.float64) - 2.0 * a)
    i = np.unravel_index(np.argmax(d), d.shape)
    print("    worst at", i, a[i], c[i])
    prop.close()
