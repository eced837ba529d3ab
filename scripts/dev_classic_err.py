"""Dev helper: error statistics of the fast classic kernel against the oracle on the parity-test ensembles, beside
the oracle's own solver-to-solver difference (tridiagonal vs the reference's dense LU) on the same inputs.

    python scripts/dev_classic_err.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import ebm_b200 as ebm
from helpers import oracle_classic, rel_err, warm_init, cold_init
from test_classic_gpu import _ensemble, _par


def report(name, st, forcings, pars, inits, stride):
    nmem = len(pars)
    o = oracle_classic(st, forcings, pars, inits, lastonly=True, raw=True, seasonal=True)
    o2 = oracle_classic(st, forcings, pars, inits, lastonly=True, raw=True, seasonal=True, solver=1)
    r = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=stride)
    sel = np.arange(0, nmem, stride)
    err = rel_err(r.raw, o["raw"][sel])
    err2 = rel_err(o2["raw"][sel], o["raw"][sel])
    k, ti, v, j = np.unravel_index(err.argmax(), err.shape)
    print(f"{name}: GPU vs oracle max {err.max():.3e} (member {sel[k]}, step {ti}, var {v}, cell {j}); "
          f">1e-9: {(err > 1e-9).sum()}  >1e-10: {(err > 1e-10).sum()}  >1e-11: {(err > 1e-11).sum()} of {err.size}; "
          f"final E {rel_err(r.final['E'], o['E']).max():.2e} Tg {rel_err(r.final['Tg'], o['Tg']).max():.2e}")
    k2, t2, v2, j2 = np.unravel_index(err2.argmax(), err2.shape)
    print(f"{name}: oracle dense-LU vs oracle tridiagonal max {err2.max():.3e} (member {sel[k2]}, step {t2}, var {v2}, cell {j2}); "
          f">1e-9: {(err2 > 1e-9).sum()}  >1e-10: {(err2 > 1e-10).sum()}  >1e-11: {(err2 > 1e-11).sum()}")
    Eref = o["raw"][sel][:, :, 0, :]
    big = np.argwhere(err > 5e-10)
    if len(big):
        print("   |E_ref| at the cells with err > 5e-10:", sorted({round(float(abs(Eref[a, b, d])), 4) for a, b, c, d in big})[:12])


for nmem, nx, nt in [(70, 100, 2000), (33, 60, 1000), (5, 37, 500)]:
    st = ebm.SpaceTime(nx, nt, 3)
    f, p, i = _ensemble(nmem, nx)
    report(f"ensemble {nmem}x{nx}x{nt}", st, f, p, i, 3)
nmem, nx = 70, 100
st = ebm.SpaceTime(nx, 2000, 3)
forcings = [ebm.Forcing(-6.0 + 12.0 * (m % 9) / 8.0) for m in range(nmem)]
pars = [_par(B=1.9 + 0.05 * (m % 6), A=190.0 + (m % 4), ai=0.38 + 0.01 * (m % 5), k=1.8 + 0.1 * (m % 3)) for m in range(nmem)]
inits = [warm_init(nx) if m % 2 == 0 else cold_init(nx) for m in range(nmem)]
report("sweep of non-matrix parameters", st, forcings, pars, inits, 5)
st = ebm.SpaceTime(100, 2000, 30)
report("default member 30 y", st, [ebm.Forcing(0.0)], [_par()], [warm_init(100)], 1)
