"""Host-side mirror of ``Infrastructure.integrate`` / ``step!`` on top of the C ABI.

``integrate`` keeps the reference's signature (src/infrastructure.jl:615-618) and returns a
``Solutions``; ``integrate_ensemble`` is the form the package extension adds -- vectors of
``Forcing`` / parameter ``Collection`` / initial conditions, one entry per member.  Every
numerical operation happens in libebm_cuda.so; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from collections import namedtuple
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from .types import (CLASSIC_PAR_ORDER, CLASSIC_VARS, MIZ_PAR_ORDER, MIZ_VARS, Collection, Forcing, Solutions,
                    SpaceTime)

__all__ = ["integrate", "integrate_ensemble", "integrate_arrays", "integrate_grids", "GroupedResult", "step", "EnsembleResult",
           "fp64_peak", "model_name"]

_MIZ_STATE = ("Ei", "Ew", "h", "D", "phi")


# What the host entry points of a model take and return (include/ebm_cuda.h): parameter order, stored variables, initial
# state in argument order, whether the closure warm start T0 follows it (optional on input; always returned), the
# int64 per-member counters, the outputs struct and the single- and multi-GPU entry points.
_Model = namedtuple("_Model", "par_order variables state T0 counters outputs run run_multi")
_MODELS = {
    "Classic": _Model(CLASSIC_PAR_ORDER, CLASSIC_VARS, ("E", "Tg"), False, (), _lib.ClassicOutputs,
                      "ebm_classic_run", "ebm_classic_run_multi"),
    "MIZ": _Model(MIZ_PAR_ORDER, MIZ_VARS, _MIZ_STATE, True, ("newton_iters", "nonconv"), _lib.MizOutputs,
                  "ebm_miz_run", "ebm_miz_run_multi"),
}


def model_name(model) -> str:
    """``:MIZ`` / ``:Classic``.  The reference dispatches on Val{:Classic}; ``:classic`` is a MethodError there."""
    name = str(model).lstrip(":")
    if name not in ("MIZ", "Classic"):
        raise ValueError(f"no method matching step!(::Val{{:{name}}}, ...): model must be :MIZ or :Classic")
    return name


@dataclass
class EnsembleResult:
    """What one ensemble call returns (all NumPy, host memory)."""
    model: str
    spacetime: SpaceTime
    nmem: int
    field_stride: int
    variables: tuple
    diag: np.ndarray | None = None       # [nmem, dur, 3, 4]  (season: winter, summer, avg; mean T, mean E, ice area, ice edge)
    seasonal: np.ndarray | None = None   # [nsel, dur, 3, nvar, nx]
    raw: np.ndarray | None = None        # [nsel, nraw, nvar, nx]
    final: dict = field(default_factory=dict)   # state arrays [nmem, nx]
    flags: np.ndarray | None = None
    newton_iters: np.ndarray | None = None
    nonconv: np.ndarray | None = None

    def solutions(self, k: int, forcing: Forcing, par: Collection, init: Collection, lastonly: bool) -> Solutions:
        """Rebuild the reference's ``Solutions`` for the k-th member that has field output."""
        sols = Solutions(self.spacetime, forcing, par, init, self.variables, lastonly)
        for vi, v in enumerate(self.variables):
            if self.raw is not None:
                sols.raw[v][:] = self.raw[k, :, vi, :]
            if self.seasonal is not None:
                sols.seasonal.winter[v][:] = self.seasonal[k, :, 0, vi, :]
                sols.seasonal.summer[v][:] = self.seasonal[k, :, 1, vi, :]
                sols.seasonal.avg[v][:] = self.seasonal[k, :, 2, vi, :]
        return sols


def _rows(pars, order) -> np.ndarray:
    out = np.empty((len(pars), len(order)))
    for m, p in enumerate(pars):
        try:
            out[m] = [p[k] for k in order]
        except KeyError as exc:   # Julia: KeyError from the Collection's Dict
            raise KeyError(f"parameter {exc.args[0]!r} missing for member {m}") from exc
    return out


def _stack(inits, key, nx) -> np.ndarray:
    a = np.ascontiguousarray(np.stack([np.asarray(i[key], dtype=np.float64) for i in inits]))
    if a.shape != (len(inits), nx):
        raise ValueError(f"init.{key} must have length nx={nx}")
    return a


def integrate_ensemble(model, st: SpaceTime, forcings, pars, inits, *, T0guess=None, debug=None, **kw) -> EnsembleResult:
    """Integrate ``len(pars)`` independent members on one GPU: one ``Forcing`` / parameter ``Collection`` / initial
    condition ``Collection`` per member (the ensemble form of the reference's ``integrate`` arguments).

    ``field_stride`` > 0 selects the members (``m % field_stride == 0``) whose seasonal (L1) and raw (L2)
    fields are returned; L0 diagnostics and final states are returned for every member.  Keyword arguments as
    ``integrate_arrays``.
    """
    name = model_name(model)
    if debug is not None:
        raise ValueError("`debug::Expr` cannot be evaluated on the device (EBM_ERR_UNSUPPORTED)")
    nmem = len(pars)
    if not (len(forcings) == nmem == len(inits)) or nmem == 0:
        raise ValueError("forcings, pars and inits must be non-empty and of equal length")
    forc = np.stack([f.row() for f in forcings])
    m = _MODELS[name]
    par = _rows(pars, m.par_order)
    state = {k: _stack(inits, k, st.nx) for k in m.state}
    if m.T0 and T0guess is not None:
        state["T0"] = np.asarray(T0guess, dtype=np.float64).reshape(nmem, st.nx)
    return integrate_arrays(name, st, forc, par, state, **kw)


@dataclass
class GroupedResult:
    """Result of ``integrate_grids``: one ``EnsembleResult`` per distinct SpaceTime, plus where each member went."""
    groups: list            # [(SpaceTime, member indices in the caller's order, EnsembleResult)]
    where: list             # member m -> (group index, row inside the group)

    def member(self, m: int) -> dict:
        """diag [dur, 3, 4], final state {name: [nx]}, flags of member m (caller's numbering)."""
        g, r = self.where[m]
        st, _, res = self.groups[g]
        out = {"spacetime": st, "diag": None if res.diag is None else res.diag[r],
               "final": {k: v[r] for k, v in res.final.items()}, "flags": None if res.flags is None else int(res.flags[r])}
        if res.newton_iters is not None:
            out["newton_iters"] = int(res.newton_iters[r])
        return out


def integrate_grids(model, sts, forcings, pars, inits, **kw) -> GroupedResult:
    """Ensemble whose members do not share one grid (SURVEY 8f-4: per-member nx / nt / duration / grid kind): ``sts[m]`` is
    member m's SpaceTime.  Members are grouped by SpaceTime -- a kernel launch integrates one grid: the latitude
    tables, the band partition and the time loop are per launch -- each group is one ``integrate_ensemble`` call, and
    the results are addressed by the caller's member index.  A member's result depends only on its own inputs, so it is
    bit-identical to integrating that member alone."""
    nmem = len(sts)
    if not (len(forcings) == nmem == len(pars) == len(inits)) or nmem == 0:
        raise ValueError("sts, forcings, pars and inits must be non-empty and of equal length")
    if kw.get("field_stride", 0) not in (0, 1):
        raise ValueError("integrate_grids: field_stride must be 0 or 1 (field output is selected per group)")
    keys, order = {}, []
    for m, st in enumerate(sts):
        key = (st.nx, st.nt, st.dur, st.grid_kind)
        if key not in keys:
            keys[key] = len(order)
            order.append((st, []))
        order[keys[key]][1].append(m)
    groups, where = [], [None] * nmem
    for g, (st, idx) in enumerate(order):
        T0 = kw.get("T0guess")
        kwg = dict(kw)
        if T0 is not None:
            kwg["T0guess"] = np.stack([np.asarray(T0[m], dtype=np.float64) for m in idx])
        res = integrate_ensemble(model, st, [forcings[m] for m in idx], [pars[m] for m in idx], [inits[m] for m in idx], **kwg)
        groups.append((st, idx, res))
        for r, m in enumerate(idx):
            where[m] = (g, r)
    return GroupedResult(groups, where)


def integrate_arrays(model, st: SpaceTime, forc, par, state, *, lastonly: bool = True, field_stride: int = 0,
                     want_diag: bool = True, want_seasonal: bool | None = None, want_raw: bool | None = None,
                     device: int = -1, strict: bool = False, years_per_launch: int = 0,
                     newton_tol: float = 0.0, newton_maxit: int = 0, step_limit: int = 0,
                     start_year: int = 0, devices=None, packet: int = 0, classic_stencil: int = 0) -> EnsembleResult:
    """Array form for large ensembles (no per-member Python objects): ``forc[nmem, 10]`` (``Forcing.row()`` layout),
    ``par[nmem, 15 | 22]`` in ``CLASSIC_PAR_ORDER`` / ``MIZ_PAR_ORDER``, ``state`` a dict of ``[nmem, nx]`` arrays
    (classic ``E, Tg``; MIZ ``Ei, Ew, h, D, phi`` and optionally the closure warm start ``T0``) -- exactly the buffers
    of ``ebm_classic_run`` / ``ebm_miz_run`` (include/ebm_cuda.h).

    ``devices``: a list of CUDA ordinals (or an int n = the first n devices, 0 = all) runs the ensemble on several
    GPUs through ``ebm_classic_run_multi`` / ``ebm_miz_run_multi``: one host thread + stream per GPU inside the
    library, members dealt in ``packet``-member packets (default 32) after a sort by cost; no field outputs.

    ``classic_stencil=1`` (classic only, an extension -- SURVEY 8f-4): kappa from the generic flux-form stencil
    (src/infrastructure.jl:500-527) instead of ``get_diffop(nx)``, i.e. the classic model on non-uniform grids; the
    default 0 reproduces the reference, which uses ``get_diffop`` whatever the grid (src/classic.jl:21)."""
    name = model_name(model)
    m = _MODELS[name]
    lib = _lib.load()
    nx, nt, dur = st.nx, st.nt, st.dur
    npar = len(m.par_order)
    par = np.ascontiguousarray(par, dtype=np.float64)
    forc = np.ascontiguousarray(forc, dtype=np.float64)
    if par.ndim != 2 or par.shape[1] != npar or par.shape[0] == 0:
        raise ValueError(f"par must be [nmem, {npar}]")
    nmem = par.shape[0]
    if forc.shape != (nmem, _lib.NFORCING):
        raise ValueError(f"forc must be [nmem, {_lib.NFORCING}] (Forcing.row() layout)")
    arrs = {}
    for k in m.state + (("T0",) if (m.T0 and "T0" in state) else ()):
        if k not in state:
            raise KeyError(f"initial state lacks {k!r}")
        a = np.ascontiguousarray(state[k], dtype=np.float64)
        if a.shape != (nmem, nx):
            raise ValueError(f"init.{k} must have length nx={nx}")
        arrs[k] = a
    grid = _lib.make_grid(st)
    opt = _lib.make_options(device, lastonly, field_stride, strict, years_per_launch, newton_maxit, newton_tol,
                            step_limit, start_year, classic_stencil)
    multi = None
    if devices is not None:
        multi = _lib.make_multi(devices=list(devices), packet=packet) if not isinstance(devices, int) else _lib.make_multi(ndevices=devices, packet=packet)
    nsel = (nmem + field_stride - 1) // field_stride if field_stride > 0 else 0
    nraw = nt if lastonly else nt * dur
    if want_seasonal is None:
        want_seasonal = nsel > 0
    if want_raw is None:
        want_raw = nsel > 0
    nvar = len(m.variables)
    res = EnsembleResult(name, st, nmem, field_stride, m.variables)
    res.diag = np.empty((nmem, dur, 3, 4)) if want_diag else None
    res.seasonal = np.empty((nsel, dur, 3, nvar, nx)) if (want_seasonal and nsel) else None
    res.raw = np.empty((nsel, nraw, nvar, nx)) if (want_raw and nsel) else None
    res.flags = np.zeros(nmem, dtype=np.int32)
    finals = m.state + (("T0",) if m.T0 else ())
    res.final = {k: np.empty((nmem, nx)) for k in finals}
    for c in m.counters:
        setattr(res, c, np.zeros(nmem, dtype=np.int64))
    out = m.outputs(_lib.dptr(res.diag), _lib.dptr(res.seasonal), _lib.dptr(res.raw), *[_lib.dptr(res.final[k]) for k in finals],
                    *[getattr(res, c).ctypes.data_as(C.POINTER(C.c_int64)) for c in m.counters],
                    res.flags.ctypes.data_as(C.POINTER(C.c_int32)))
    args = [C.byref(grid), nmem, _lib.dptr(par), _lib.dptr(forc), *[_lib.dptr(arrs.get(k)) for k in finals], C.byref(opt)]
    if multi is not None:
        _lib.check(getattr(lib, m.run_multi)(*args, C.byref(multi), C.byref(out)))
    else:
        _lib.check(getattr(lib, m.run)(*args, C.byref(out)))
    return res


def integrate(model, st: SpaceTime, forcing: Forcing, par: Collection, init: Collection, *, lastonly: bool = True,
              debug=None, verbose: bool = False, device: int = -1, strict: bool = False) -> Solutions:
    """``integrate(model, st, forcing, par, init; lastonly, debug, verbose) -> Solutions`` (one member).

    Same arguments as src/infrastructure.jl:615-618.  ``verbose`` prints the closure's non-convergence count
    (the reference @warns per step, src/miz.jl:61-63).
    """
    res = integrate_ensemble(model, st, [forcing], [par], [init], debug=debug, lastonly=lastonly, field_stride=1,
                             want_diag=False, device=device, strict=strict)
    if verbose and res.nonconv is not None and res.nonconv[0] > 0:
        print(f"Warning: solving for T0 failed at {int(res.nonconv[0])} time steps.")
    sols = res.solutions(0, forcing, par, init, lastonly)
    sols.final = {k: v[0] for k, v in res.final.items()}
    return sols


DEBUG_MENU = {"alpha": 1, "C": 2, "T0": 3, "S": 4, "mask": 5}   # include/ebm_cuda.h EBM_DEBUG_*


def step(model, t: float, f: float, vars: Collection, st: SpaceTime, par: Collection, *, debug=None) -> Collection:
    """``step!(Val(model), t, f, vars, st, par; debug)``: one time step of one member, in place, on the GPU.

    For ``:MIZ`` the closure's warm start (the reference's persistent ``T0``, src/miz.jl:47) is carried
    in ``vars.T0`` (zeros if absent).  ``debug`` (``:Classic``): the reference evaluates an arbitrary expression in
    the scope of step! and stores it as ``vars.debug`` (src/classic.jl:67-69); here it is the name of one of the
    per-cell locals of that scope -- ``"alpha"``, ``"C"``, ``"T0"``, ``"S"`` (= stat.S[:, i]), ``"mask"`` -- anything
    else is an error (an expression cannot run on the device).
    """
    name = model_name(model)
    if debug is not None and (name != "Classic" or debug not in DEBUG_MENU):
        raise ValueError(f"debug must be one of {sorted(DEBUG_MENU)} for :Classic (a `debug::Expr` cannot be evaluated "
                         "on the device: EBM_ERR_UNSUPPORTED)")
    lib = _lib.load()
    grid = _lib.make_grid(st)
    # time index exactly as src/classic.jl:45
    v = (t + st.dt / 2.0) * st.nt
    r = v % st.nt
    ti = int(round(st.nt if r == 0 else r))
    nx = st.nx
    if name == "Classic":
        p = _rows([par], CLASSIC_PAR_ORDER)[0]
        E = np.array(vars["E"], dtype=np.float64)
        Tg = np.array(vars["Tg"], dtype=np.float64)
        T, h = np.empty(nx), np.empty(nx)
        dbg = np.empty(nx) if debug is not None else None
        _lib.check(lib.ebm_classic_step_debug(C.byref(grid), _lib.dptr(p), ti, float(f), _lib.dptr(E), _lib.dptr(Tg),
                                              _lib.dptr(T), _lib.dptr(h), DEBUG_MENU.get(debug, 0),
                                              _lib.dptr(dbg) if dbg is not None else None))
        vars["E"], vars["Tg"], vars["T"], vars["h"] = E, Tg, T, h
        if dbg is not None:
            vars["debug"] = dbg
    else:
        # the reference's MIZ step! uses t itself (cos(2 pi t), src/miz.jl:11), not a table index: the device entry
        # point takes the index of t in st.t, so a t off the grid would silently get its neighbour's insolation
        if not (1 <= ti <= st.nt) or abs(float(st.t[ti - 1]) - float(t)) > 1e-12:
            raise ValueError(f"MIZ step: t = {t!r} is not one of st.t (nearest: st.t[{ti - 1}] = {float(st.t[max(min(ti, st.nt), 1) - 1])!r})")
        p = _rows([par], MIZ_PAR_ORDER)[0]
        stt = [np.array(vars[k], dtype=np.float64) for k in _MIZ_STATE]
        T0 = np.array(vars["T0"], dtype=np.float64) if "T0" in vars else np.zeros(nx)
        out = np.empty((len(MIZ_VARS), nx))
        iters = C.c_int32(0)
        _lib.check(lib.ebm_miz_step(C.byref(grid), _lib.dptr(p), ti, float(f), *[_lib.dptr(a) for a in stt],
                                    _lib.dptr(T0), _lib.dptr(out), C.byref(iters)))
        for vi, k in enumerate(MIZ_VARS):
            vars[k] = out[vi].copy()
        vars["T0"] = T0
        vars["newton_iters"] = iters.value
    return vars


def fp64_peak(device: int = -1):
    """Measured DFMA throughput (TFLOP/s, FMA = 2) and the SM clock estimate of the device."""
    lib = _lib.load()
    tf, mhz = C.c_double(0.0), C.c_double(0.0)
    _lib.check(lib.ebm_fp64_peak(device, C.byref(tf), C.byref(mhz)))
    return tf.value, mhz.value
