"""ctypes wrapper around the C oracle (oracle/ebm_oracle.c).

TEST INFRASTRUCTURE ONLY -- importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs, never from the product package.  PARITY UNPINNED (see
ebm_oracle.h): Julia is not installed and the reference's only golden fixture is absent.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libebm_oracle.so")

CLASSIC_NPAR, MIZ_NPAR, NF = 15, 22, 10
CLASSIC_NVAR, MIZ_NVAR = 3, 10
SOLVE_TRIDIAG, SOLVE_DENSE_LU = 0, 1

_dp = ctypes.POINTER(ctypes.c_double)
_llp = ctypes.POINTER(ctypes.c_longlong)


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (gcc, -ffp-contract=off).  In a read-only tree an out-of-date
    library is compiled into a temporary directory instead."""
    src = os.path.join(_HERE, "ebm_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        out_dir = os.path.dirname(_SO)
        writable = os.access(out_dir if os.path.isdir(out_dir) else _HERE, os.W_OK)
        out = _SO if writable else os.path.join(tempfile.mkdtemp(prefix="ebm_oracle_"), os.path.basename(_SO))
        subprocess.run(["make", "-C", _HERE, "CC=gcc", f"OUT={out}"], check=True, capture_output=True)
        return out
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.ebm_oracle_classic_run.restype = ctypes.c_int
        _lib.ebm_oracle_miz_run.restype = ctypes.c_int
        _lib.ebm_oracle_hemispheric_mean.restype = ctypes.c_double
        _lib.ebm_oracle_forcing.restype = ctypes.c_double
        _lib.ebm_oracle_max_threads.restype = ctypes.c_int
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _c(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        assert a.shape == tuple(shape), (a.shape, shape)
    return a


def max_threads() -> int:
    return lib().ebm_oracle_max_threads()


def forcing(frow, T: float) -> float:
    frow = _c(frow, (NF,))
    return lib().ebm_oracle_forcing(_p(frow), ctypes.c_double(T))


def hemispheric_mean(v, x) -> float:
    v, x = _c(v), _c(x)
    return lib().ebm_oracle_hemispheric_mean(_p(v), _p(x), len(x))


def diag(T, E, phi, x):
    T, E, x = _c(T), _c(E), _c(x)
    phi = None if phi is None else _c(phi)
    out = np.empty(4)
    lib().ebm_oracle_diag(_p(T), _p(E), _p(phi), _p(x), len(x), _p(out))
    return out


DEBUG_MENU = {"alpha": 1, "C": 2, "T0": 3, "S": 4, "mask": 5}


def classic_step(x, t, par15, i1, f, E, Tg, debug=None):
    """One step!(Val(:Classic), ...) (src/classic.jl:37-71).  Returns dict(E, Tg, T, h[, debug]); inputs untouched."""
    x, t = _c(x), _c(t)
    nx = len(x)
    E, Tg = _c(E, (nx,)).copy(), _c(Tg, (nx,)).copy()
    T, h = np.empty(nx), np.empty(nx)
    dbg = np.empty(nx) if debug is not None else None
    fn = lib().ebm_oracle_classic_step
    fn.restype = ctypes.c_int
    rc = fn(nx, len(t), _p(x), _p(t), _p(_c(par15, (CLASSIC_NPAR,))), int(i1), ctypes.c_double(f), _p(E), _p(Tg), _p(T), _p(h),
            DEBUG_MENU[debug] if debug is not None else 0, _p(dbg))
    if rc != 0:
        raise RuntimeError(f"oracle classic_step failed: {rc}")
    out = dict(E=E, Tg=Tg, T=T, h=h)
    if debug is not None:
        out["debug"] = dbg
    return out


def classic_run(x, t, dur, winter_inx, summer_inx, par, forc, E0, Tg0, *, solver=SOLVE_TRIDIAG,
                lastonly=True, want_raw=False, want_seasonal=False, nthreads=0, stencil=0):
    """Returns dict(E, Tg[, raw[nmem,nraw,3,nx]][, seasonal[nmem,dur,3,3,nx]]); inputs untouched.
    ``stencil=1``: kappa from the generic flux-form stencil (infrastructure.jl:510-524) instead of get_diffop(nx) --
    the extension for classic on non-uniform grids (the reference uses get_diffop whatever the grid, classic.jl:21)."""
    x, t = _c(x), _c(t)
    nx, nt = len(x), len(t)
    par = _c(par).reshape(-1, CLASSIC_NPAR)
    nmem = par.shape[0]
    forc = _c(forc, (nmem, NF))
    E = _c(E0, (nmem, nx)).copy()
    Tg = _c(Tg0, (nmem, nx)).copy()
    nraw = nt if lastonly else nt * dur
    raw = np.empty((nmem, nraw, CLASSIC_NVAR, nx)) if want_raw else None
    seas = np.empty((nmem, dur, 3, CLASSIC_NVAR, nx)) if want_seasonal else None
    rc = lib().ebm_oracle_classic_run(nx, nt, dur, _p(x), _p(t), winter_inx, summer_inx, nmem, _p(par), _p(forc),
                                      _p(E), _p(Tg), int(solver) | (int(bool(stencil)) << 8), int(lastonly), _p(raw), _p(seas), nthreads)
    if rc != 0:
        raise RuntimeError(f"oracle classic_run failed: {rc}")
    return dict(E=E, Tg=Tg, raw=raw, seasonal=seas)


def miz_run(x, t, dur, winter_inx, summer_inx, grid_kind, par, forc, Ei, Ew, h, D, phi, T0=None, *,
            newton_tol=1e-8, lastonly=True, want_raw=False, want_seasonal=False, nthreads=0):
    x, t = _c(x), _c(t)
    nx, nt = len(x), len(t)
    par = _c(par).reshape(-1, MIZ_NPAR)
    nmem = par.shape[0]
    forc = _c(forc, (nmem, NF))
    st = [_c(a, (nmem, nx)).copy() for a in (Ei, Ew, h, D, phi)]
    T0 = np.zeros((nmem, nx)) if T0 is None else _c(T0, (nmem, nx)).copy()
    nraw = nt if lastonly else nt * dur
    raw = np.empty((nmem, nraw, MIZ_NVAR, nx)) if want_raw else None
    seas = np.empty((nmem, dur, 3, MIZ_NVAR, nx)) if want_seasonal else None
    iters = np.zeros(nmem, dtype=np.int64)
    fails = np.zeros(nmem, dtype=np.int64)
    rc = lib().ebm_oracle_miz_run(nx, nt, dur, _p(x), _p(t), winter_inx, summer_inx, grid_kind, nmem, _p(par), _p(forc),
                                  _p(st[0]), _p(st[1]), _p(st[2]), _p(st[3]), _p(st[4]), _p(T0),
                                  ctypes.c_double(newton_tol), int(lastonly), _p(raw), _p(seas),
                                  iters.ctypes.data_as(_llp), fails.ctypes.data_as(_llp), nthreads)
    if rc != 0:
        raise RuntimeError(f"oracle miz_run failed: {rc}")
    return dict(Ei=st[0], Ew=st[1], h=st[2], D=st[3], phi=st[4], T0=T0, raw=raw, seasonal=seas,
                newton_iters=iters, nonconv=fails)
