"""GPU parity tests for the MIZ path: libebm_cuda (through the C ABI / host mirror) vs the CPU oracle.

The MIZ model amplifies rounding-level differences: perturbing the reference algorithm's initial state by 1e-13
changes every variable by O(0.1) within 200 steps of the spin-up and the year-30 climate by ~2e-3 (measured
with the oracle, DESIGN.md "MIZ sensitivity").  Long-run pointwise parity is therefore undefined even between
two runs of the reference on different libm/BLAS builds -- which is why the reference's own test compares step
10 only (test/runtests.jl:37-47).  Parity is established in layers:

  1. the strict kernel (literal operation order, -fmad=false, serial Thomas) and the one-step entry point are
     BIT-IDENTICAL to the oracle over whole trajectories (1 and 30 years, both grid kinds, ensembles);
  2. the fast kernel (same source, FMA contraction + warp-parallel solve) meets the reference's criterion
     (step 10, rtol = sqrt(eps)) and stays within that tolerance over short horizons (20 steps) started from
     oracle states taken all along a 30-year trajectory and across a parameter ensemble;
  3. long fast runs are checked through determinism (chained launches / restarts are bitwise reproducible),
     sampler self-consistency, state invariants and climatology within the model's own sensitivity envelope.

Tolerance: rtol = sqrt(eps) = 1.49e-8 (Julia isapprox default) with an absolute floor of the same size
(|ref| < 1 compared absolutely), NaN masks compared separately.
"""
import numpy as np
import pytest

import ebm_b200 as ebm
from helpers import oracle_diag_miz, oracle_miz, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1.4901161193847656e-08   # sqrt(eps(Float64)): Julia's isapprox default
STATE = ("Ei", "Ew", "h", "D", "phi")


def _par(**kw):
    p = ebm.default_parameters("MIZ")
    p.update(kw)
    return p


def _zero(nx):
    z = np.zeros(nx)
    return ebm.Collection(Ei=z.copy(), Ew=z.copy(), h=z.copy(), D=z.copy(), phi=z.copy())


# Rounding-level perturbations of the first step's water enthalpy.  One perturbed oracle run is ONE sample of the
# model's sensitivity: over these eight the year-5 response of a single C5 member spans 2e-5 ... 2e-2, so the
# envelope is the largest response over a small perturbation ensemble, not a single draw.
PERTURBATIONS = (1e-14, -1e-14, 3e-14, -3e-14)


def _envelope(run_diag, ref, nx):
    """max over PERTURBATIONS of |run_diag(perturbed zero init) - ref|; NaN (a member that blows up under the
    perturbation) propagates, so such members drop out of the comparison."""
    env = None
    for eps in PERTURBATIONS:
        pin = _zero(nx)
        pin.Ew = pin.Ew + eps
        d = np.abs(run_diag(pin) - ref)
        env = d if env is None else np.where(np.isnan(env) | np.isnan(d), np.nan, np.maximum(env, d))
    return env


def _same(a, b):
    """bit-for-bit, NaN == NaN"""
    return np.array_equal(a, b, equal_nan=True)


def _check(a, ref, what, tol=RTOL):
    assert np.array_equal(np.isnan(a), np.isnan(ref)), f"{what}: NaN masks differ"
    err = rel_err(a, ref)
    assert err.max() < tol, (what, err.max(), np.unravel_index(err.argmax(), err.shape))


def test_fixture_setup_matches_reference_test_criterion():
    """test/runtests.jl:20-48: MIZ, SpaceTime{sin}(180, 2000, 1), zero init, F = 0; raw[var][10] of the ten
    variables, NaN -> 0, element-wise isapprox(rtol = sqrt(eps), atol = 0)."""
    st = ebm.SpaceTime(180, 2000, 1, "sin")
    par, f, init = _par(), ebm.Forcing(0.0), _zero(180)
    sols = ebm.integrate("MIZ", st, f, par, init)
    o = oracle_miz(st, [f], [par], [init], raw=True)
    for vi, v in enumerate(ebm.MIZ_VARS):
        a, b = np.nan_to_num(sols.raw[v][9]), np.nan_to_num(o["raw"][0, 9, vi])
        assert np.all(np.abs(a - b) <= RTOL * np.maximum(np.abs(a), np.abs(b))), v
    # known-answer probe values of SURVEY Appendix D (step 10 of the fixture run)
    assert abs(sols.raw.E[9][0] - 0.509) < 2e-3 and abs(sols.raw.E[9][-1] + 1.174) < 2e-3
    assert abs(np.nan_to_num(sols.raw.Ti[9])[-1] + 11.24) < 2e-2


def test_single_step_bitwise_chain():
    """step!(Val(:MIZ), ...) for 12 consecutive steps from the zero state: every stored variable of every step
    and the carried state are bit-identical to the oracle (NaN masks included)."""
    st = ebm.SpaceTime(180, 2000, 1, "sin")
    par, f = _par(), 0.75
    o = oracle_miz(st, [ebm.Forcing(f)], [par], [_zero(180)], lastonly=False, raw=True)
    v = _zero(180)
    for k in range(12):
        ebm.step("MIZ", st.t[k], f, v, st, par)
        for vi, name in enumerate(ebm.MIZ_VARS):
            assert _same(v[name], o["raw"][0, k, vi]), (k, name)
    assert v["newton_iters"] >= 0


@pytest.mark.parametrize("xfunc,nx", [("sin", 180), ("identity", 100)])
def test_strict_kernel_bitwise_one_year(xfunc, nx):
    """C1b with the literal-arithmetic kernel: all 2000 steps of the ten variables, the final state, the closure
    warm start and the Newton iteration count are bit-identical to the oracle, on both grid kinds."""
    st = ebm.SpaceTime(nx, 2000, 1, xfunc)
    par, f, init = _par(), ebm.Forcing(0.0), _zero(nx)
    o = oracle_miz(st, [f], [par], [init], lastonly=False, raw=True, seasonal=True)
    r = ebm.integrate_ensemble("MIZ", st, [f], [par], [init], lastonly=False, field_stride=1, strict=True)
    for vi, name in enumerate(ebm.MIZ_VARS):
        assert _same(r.raw[0, :, vi], o["raw"][0, :, vi]), name
    for k in STATE + ("T0",):
        assert _same(r.final[k], o[k]), k
    assert int(r.newton_iters[0]) == int(o["newton_iters"][0]) and int(r.nonconv[0]) == int(o["nonconv"][0])
    assert _same(r.seasonal[0, :, :2], o["seasonal"][0, :, :2])      # winter / summer snapshots are copies
    _check(r.seasonal[0, :, 2], o["seasonal"][0, :, 2], "annual mean", 1e-12)   # summation order only


HORIZON = 20


def test_fast_kernel_short_horizon_from_zero_state():
    """C1b setup: the first 20 steps of all ten variables within the reference's tolerance."""
    st = ebm.SpaceTime(180, 2000, 1, "sin")
    par, f, init = _par(), ebm.Forcing(0.0), _zero(180)
    o = oracle_miz(st, [f], [par], [init], lastonly=False, raw=True)
    r = ebm.integrate_ensemble("MIZ", st, [f], [par], [init], lastonly=False, field_stride=1, step_limit=HORIZON)
    for vi, v in enumerate(ebm.MIZ_VARS):
        _check(r.raw[0, :HORIZON, vi], o["raw"][0, :HORIZON, vi], v)
    assert np.isnan(r.raw[0, HORIZON:]).all()          # steps not taken stay NaN (undef in the reference)


def test_fast_kernel_short_horizons_along_thirty_year_trajectory():
    """C3 trajectory (docstring example, src/EnergyBalanceModel.jl:18-57): restart the fast kernel from the
    oracle's state (incl. the closure warm start) after 1, 2, 3, 5, 10, 20 and 30 years; 20 steps each."""
    par, f = _par(), ebm.Forcing(0.0)
    inits, T0s = [], []
    for years in (1, 2, 3, 5, 10, 20, 30):
        o = oracle_miz(ebm.SpaceTime(180, 2000, years, "sin"), [f], [par], [_zero(180)])
        inits.append(ebm.Collection({k: o[k][0] for k in STATE}))
        T0s.append(o["T0"][0])
    st = ebm.SpaceTime(180, 2000, 1, "sin")
    n = len(inits)
    o = oracle_miz(st, [f] * n, [par] * n, inits, T0=np.stack(T0s), lastonly=False, raw=True)
    r = ebm.integrate_ensemble("MIZ", st, [f] * n, [par] * n, inits, T0guess=np.stack(T0s), lastonly=False,
                               field_stride=1, step_limit=HORIZON)
    for vi, v in enumerate(ebm.MIZ_VARS):
        _check(r.raw[:, :HORIZON, vi], o["raw"][:, :HORIZON, vi], v)


def test_strict_kernel_bitwise_thirty_years():
    """C3 with the literal-arithmetic kernel: 30 years, last-year raw + all seasonal snapshots + final state
    bit-identical to the oracle."""
    st = ebm.SpaceTime(180, 2000, 30, "sin")
    par, f, init = _par(), ebm.Forcing(0.0), _zero(180)
    o = oracle_miz(st, [f], [par], [init], raw=True, seasonal=True)
    r = ebm.integrate_ensemble("MIZ", st, [f], [par], [init], field_stride=1, strict=True)
    assert _same(r.raw[0], o["raw"][0])
    assert _same(r.seasonal[0, :, :2], o["seasonal"][0, :, :2])
    for k in STATE + ("T0",):
        assert _same(r.final[k], o[k]), k
    assert int(r.newton_iters[0]) == int(o["newton_iters"][0])


def test_fast_kernel_thirty_years_climatology():
    """C3 with the fast kernel: Solutions layout, and the year-30 climate within the model's own sensitivity
    envelope, measured in the test with a perturbed oracle run (see also
    test_fast_kernel_divergence_is_bounded_by_the_models_own_sensitivity)."""
    st = ebm.SpaceTime(180, 2000, 30, "sin")
    par, f, init = _par(), ebm.Forcing(0.0), _zero(180)
    o = oracle_miz(st, [f], [par], [init], seasonal=True)
    r = ebm.integrate_ensemble("MIZ", st, [f], [par], [init], field_stride=1)
    sols = r.solutions(0, f, par, init, True)
    assert abs(sols.ts[0] - 29.00025) < 1e-12 and len(sols.ts) == 2000 and sols.raw.E.shape == (2000, 180)
    od = oracle_diag_miz(o["seasonal"], st.x)
    d = np.abs(r.diag[0, 29] - od[0, 29])
    # derived envelope: the oracle's own response to rounding-level perturbations of the first step's water enthalpy
    # (largest over PERTURBATIONS) -- the fast kernel may differ from the oracle by at most 10x that, per diagnostic
    env = _envelope(lambda pin: oracle_diag_miz(oracle_miz(st, [f], [par], [pin], seasonal=True)["seasonal"], st.x)[0, 29],
                    od[0, 29], 180)
    floor = np.array([1e-6, 1e-6, 1e-6, 0.0])[None, :]            # ice edge is quantised to the grid: no floor needed
    dx = float(np.diff(st.x).max())
    env[:, 3] = np.maximum(env[:, 3], dx)                          # ... but it moves by whole cells
    assert (d <= 10.0 * np.maximum(env, floor)).all(), (d, env)
    ice_cells = int((sols.raw.phi[-1] > 0).sum())
    assert 30 <= ice_cells <= 90                       # SURVEY Appendix D probe: ice cells 175 -> 57
    assert r.nonconv[0] == 0 and r.flags[0] == 0


def _ensemble(nmem):
    forcings, pars = [], []
    for m in range(nmem):
        forcings.append(ebm.Forcing(-2.0 + 4.0 * (m % 5) / 4.0))
        pars.append(_par(D=0.45 + 0.3 * (m % 7) / 6.0, B=1.8 + 0.1 * (m % 4), ai=0.35 + 0.02 * (m % 6),
                         k=1.5 + 0.25 * (m % 5), m1=50.4576 * (0.5 + 0.25 * (m % 3))))
    return forcings, pars


@pytest.mark.parametrize("nmem,nx,nt,xfunc", [(37, 180, 2000, "sin"), (9, 100, 1000, "identity"),
                                              (5, 50, 800, "sin"), (6, 250, 2000, "sin")])
def test_ensemble_strict_bitwise_and_fast_short_horizon(nmem, nx, nt, xfunc):
    """Ragged member counts, both grid kinds, other grid sizes, per-member parameters and forcing.
    Strict kernel: final state of every member after 1 year bit-identical.  Fast kernel: first 20 steps of the
    strided members' fields within tolerance."""
    st = ebm.SpaceTime(nx, nt, 1, xfunc)
    forcings, pars = _ensemble(nmem)
    inits = [_zero(nx) for _ in range(nmem)]
    o = oracle_miz(st, forcings, pars, inits, lastonly=False, raw=True)
    rs = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, strict=True)
    for k in STATE + ("T0",):
        assert _same(rs.final[k], o[k]), k
    assert np.array_equal(rs.newton_iters, o["newton_iters"])
    r = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, lastonly=False, field_stride=4, step_limit=HORIZON)
    sel = np.arange(0, nmem, 4)
    _check(r.raw[:, :HORIZON], o["raw"][sel, :HORIZON], "raw")


def test_multi_gpu_entry_point_matches_single_gpu_bitwise():
    """ebm_miz_run_multi (members dealt over the GPUs in packets): diagnostics, final state, counters, flags and the
    strided members' field outputs equal the single-GPU call's bit for bit.  Runs on one GPU too."""
    import torch
    ndev = min(torch.cuda.device_count(), 2)
    nmem, nx = 75, 60
    st = ebm.SpaceTime(nx, 400, 1, "sin")
    forcings, pars = _ensemble(nmem)
    inits = [_zero(nx) for _ in range(nmem)]
    ref = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, field_stride=4)
    r = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, field_stride=4, devices=list(range(ndev)), packet=8)
    assert _same(r.diag, ref.diag)
    for k in STATE + ("T0",):
        assert _same(r.final[k], ref.final[k]), k
    assert np.array_equal(r.newton_iters, ref.newton_iters) and np.array_equal(r.nonconv, ref.nonconv)
    assert np.array_equal(r.flags, ref.flags)
    assert r.seasonal.shape == ref.seasonal.shape and _same(r.seasonal, ref.seasonal) and _same(r.raw, ref.raw)


def test_multi_gpu_diagnostics_on_device_match_single_gpu_bitwise():
    """ebm_miz_run_multi with the diagnostics in device memory of GPU 0 (multi.diag_device = 0): the other GPU sends
    its rows there over NCCL.  Diagnostics, final state, counters, flags and field outputs equal the single-GPU call's
    bit for bit.  Runs on one GPU too."""
    import ctypes as C
    import torch
    from ebm_b200 import _lib
    ndev = min(torch.cuda.device_count(), 2)
    nmem, nx = 75, 60
    st = ebm.SpaceTime(nx, 400, 1, "sin")
    forcings, pars = _ensemble(nmem)
    ref = ebm.integrate_ensemble("MIZ", st, forcings, pars, [_zero(nx) for _ in range(nmem)], field_stride=4)
    lib = _lib.load()
    d_diag = torch.full((nmem, 1, 3, 4), float("nan"), dtype=torch.float64, device="cuda:0")
    seasonal, raw = np.empty_like(ref.seasonal), np.empty_like(ref.raw)
    final = {k: np.empty((nmem, nx)) for k in STATE + ("T0",)}
    iters, nonconv = np.zeros(nmem, dtype=np.int64), np.zeros(nmem, dtype=np.int64)
    flags = np.zeros(nmem, dtype=np.int32)
    i64 = C.POINTER(C.c_int64)
    out = _lib.MizOutputs(C.cast(d_diag.data_ptr(), C.POINTER(C.c_double)), _lib.dptr(seasonal), _lib.dptr(raw),
                          *[_lib.dptr(final[k]) for k in STATE + ("T0",)], iters.ctypes.data_as(i64),
                          nonconv.ctypes.data_as(i64), flags.ctypes.data_as(C.POINTER(C.c_int32)))
    par = np.array([[p[k] for k in ebm.MIZ_PAR_ORDER] for p in pars])
    forc = np.stack([f.row() for f in forcings])
    z = np.zeros((nmem, nx))
    grid, opt = _lib.make_grid(st), _lib.make_options(field_stride=4)
    multi = _lib.make_multi(devices=list(range(ndev)), diag_device=0, packet=8)
    _lib.check(lib.ebm_miz_run_multi(C.byref(grid), nmem, _lib.dptr(par), _lib.dptr(forc), *[_lib.dptr(z)] * 5, None,
                                     C.byref(opt), C.byref(multi), C.byref(out)))
    torch.cuda.synchronize()
    assert _same(d_diag.cpu().numpy(), ref.diag)
    for k in STATE + ("T0",):
        assert _same(final[k], ref.final[k]), k
    assert np.array_equal(iters, ref.newton_iters) and np.array_equal(nonconv, ref.nonconv)
    assert np.array_equal(flags, ref.flags)
    assert _same(seasonal, ref.seasonal) and _same(raw, ref.raw)


def test_sampler_self_consistency_and_diagnostics():
    """savesol! semantics on the device (infrastructure.jl:549-591): winter / summer snapshots are the raw steps
    winter.inx / summer.inx, the annual mean is the mean of the year's raw steps, and the L0 diagnostics equal
    hemispheric_mean / ice area / ice edge of those very fields.  (Self-consistency: independent of the
    trajectory's sensitivity.)"""
    nx, nmem = 180, 10
    st = ebm.SpaceTime(nx, 2000, 2, "sin")
    forcings, pars = _ensemble(nmem)
    r = ebm.integrate_ensemble("MIZ", st, forcings, pars, [_zero(nx)] * nmem, lastonly=False, field_stride=3)
    nsel = len(range(0, nmem, 3))
    assert r.raw.shape == (nsel, 4000, 10, nx) and r.seasonal.shape == (nsel, 2, 3, 10, nx)
    for y in range(2):
        assert _same(r.seasonal[:, y, 0], r.raw[:, y * 2000 + st.winter.inx - 1])
        assert _same(r.seasonal[:, y, 1], r.raw[:, y * 2000 + st.summer.inx - 1])
        mean = r.raw[:, y * 2000:(y + 1) * 2000].mean(axis=1)
        _check(r.seasonal[:, y, 2], mean, "annual mean", 1e-11)
    d = oracle_diag_miz(r.seasonal, st.x)
    sel = np.arange(0, nmem, 3)
    _check(r.diag[sel][..., :3], d[..., :3], "diag", 1e-11)
    assert np.abs(r.diag[sel][..., 3] - d[..., 3]).max() == 0.0


def test_ramp_forcing_and_chained_launches():
    """Forcing{false} per step on the device (strict run bit-identical to the oracle); splitting a fast run into
    launches (state + warm start carried through HBM) changes nothing."""
    st = ebm.SpaceTime(180, 2000, 3, "sin")
    forcings = [ebm.Forcing(0.0, 4.0, -2.0, (1, 0), (4.0, -6.0)), ebm.Forcing(1.5), ebm.Forcing(-1.0, 1.0, -1.0, (0, 1), (2.0, -2.0))]
    pars = [_par()] * 3
    inits = [_zero(180) for _ in range(3)]
    o = oracle_miz(st, forcings, pars, inits)
    s = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, strict=True)
    for k in STATE:
        assert _same(s.final[k], o[k]), k
    a = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, field_stride=1, want_raw=False)
    b = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, field_stride=1, want_raw=False, years_per_launch=1)
    for k in STATE + ("T0",):
        assert _same(a.final[k], b.final[k]), k
    assert _same(a.seasonal, b.seasonal) and _same(a.diag, b.diag)
    assert np.array_equal(a.newton_iters, b.newton_iters)


def test_restart_from_final_state_reproduces_long_run():
    """Checkpoint/restart (SURVEY 8f.3): a 2-year run == two 1-year runs chained through the returned state and
    the returned closure warm start T0 (the reference's persistent T0, src/miz.jl:47,64)."""
    par, f = _par(), ebm.Forcing(0.5)
    full = ebm.integrate_ensemble("MIZ", ebm.SpaceTime(180, 2000, 2, "sin"), [f], [par], [_zero(180)])
    st1 = ebm.SpaceTime(180, 2000, 1, "sin")
    a = ebm.integrate_ensemble("MIZ", st1, [f], [par], [_zero(180)])
    init2 = ebm.Collection({k: a.final[k][0] for k in STATE})
    b = ebm.integrate_ensemble("MIZ", st1, [f], [par], [init2], T0guess=a.final["T0"])
    for k in STATE + ("T0",):
        assert _same(full.final[k], b.final[k]), k


def test_state_invariants_large_ensemble():
    """Size-independent properties on a 4096-member parameter sweep: phi in [0,1], h >= 0, D in {0} U [Dmin,Dmax],
    Ei <= 0 <= Ew, finite state, closure converged everywhere; year-1 climate of spot-checked members within
    the sensitivity envelope of the oracle."""
    nmem, nx = 4096, 180
    st = ebm.SpaceTime(nx, 2000, 1, "sin")
    forcings, pars = _ensemble(nmem)
    r = ebm.integrate_ensemble("MIZ", st, forcings, pars, [_zero(nx)] * nmem)
    assert r.flags.max() == 0 and r.nonconv.max() == 0
    f = r.final
    assert (f["phi"] >= 0).all() and (f["phi"] <= 1).all() and (f["h"] >= 0).all()
    assert (f["Ei"] <= 0).all() and (f["Ew"] >= 0).all()
    D = f["D"]
    assert (((D == 0) | ((D >= 1.0) & (D <= 156.0)))).all()
    assert np.isfinite(r.diag).all()
    idx = list(range(0, nmem, 512))
    o = oracle_miz(st, [forcings[i] for i in idx], [pars[i] for i in idx], [_zero(nx)] * len(idx), seasonal=True)
    od = oracle_diag_miz(o["seasonal"], st.x)
    # envelope derived from the oracle's own sensitivity (perturbed run), member by member
    env = _envelope(lambda pin: oracle_diag_miz(oracle_miz(st, [forcings[i] for i in idx], [pars[i] for i in idx],
                                                           [pin] * len(idx), seasonal=True)["seasonal"], st.x)[:, 0, 2, 0],
                    od[:, 0, 2, 0], nx)
    assert (np.abs(r.diag[idx, 0, 2, 0] - od[:, 0, 2, 0]) <= 10.0 * np.maximum(env, 1e-6)).all()      # annual-mean hemispheric T


def test_c5_members_five_years():
    """BASELINE config C5 (SURVEY 8d): 8 evenly spaced members of the 16^5 = 1 048 576-member (D, B, ai, k, m1) tensor
    grid, sin grid, zero init, 5 years.  Literal kernel: final state, warm start and Newton counts bit-identical to
    the oracle (including which members blow up).  Fast kernel: on the members that stay finite, invariants hold, the
    closure converged and the year-5 hemispheric-mean temperature is within the model's sensitivity envelope."""
    import bench
    N, nsub, years = 16 ** 5, 8, 5
    idx = np.array([int(round(k * (N - 1) / (nsub - 1))) for k in range(nsub)])
    st, rows, _, _ = bench.miz_workload(ebm, N, np.asarray(idx, dtype=np.int64), years)
    pars = [ebm.Collection(dict(zip(ebm.MIZ_PAR_ORDER, r))) for r in rows]
    assert len({tuple(r) for r in rows}) == nsub                                 # distinct parameter sets
    forcings = [ebm.Forcing(0.0)] * nsub
    inits = [_zero(180) for _ in range(nsub)]
    o = oracle_miz(st, forcings, pars, inits, seasonal=True)
    rs = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits, strict=True)
    for k in STATE + ("T0",):
        assert _same(rs.final[k], o[k]), k
    assert np.array_equal(rs.newton_iters, o["newton_iters"]) and np.array_equal(rs.nonconv, o["nonconv"])
    r = ebm.integrate_ensemble("MIZ", st, forcings, pars, inits)
    # the reference algorithm itself blows up (non-finite state) on part of this sweep -- 2 of these 8 members within
    # 5 years in the oracle; such members are flagged, not an error.  Compare the members that stay finite in both.
    ofinite = np.isfinite(o["Ei"]).all(axis=1)
    assert np.array_equal(rs.flags == 0, ofinite)                                # literal kernel: same members blow up
    ok = (r.flags == 0) & ofinite
    assert ok.sum() >= nsub // 2
    f = r.final
    assert (f["phi"][ok] >= 0).all() and (f["phi"][ok] <= 1).all() and (f["h"][ok] >= 0).all()
    assert (f["Ei"][ok] <= 0).all() and (f["Ew"][ok] >= 0).all() and r.nonconv[ok].max() == 0
    od = oracle_diag_miz(o["seasonal"], st.x)
    env = _envelope(lambda pin: oracle_diag_miz(oracle_miz(st, forcings, pars, [pin] * nsub, seasonal=True)["seasonal"],
                                                st.x)[:, -1, 2, 0], od[:, -1, 2, 0], 180)
    okp = ok & np.isfinite(env)              # members that stay finite under every perturbation
    assert okp.sum() >= nsub // 2
    assert (np.abs(r.diag[okp, -1, 2, 0] - od[okp, -1, 2, 0]) <= 10.0 * np.maximum(env[okp], 1e-6)).all()


def test_fast_kernel_divergence_is_bounded_by_the_models_own_sensitivity(capsys):
    """Derived (not hand-picked) bound for the fast kernel over long horizons (round-1 VERDICT item 4).

    The MIZ model amplifies rounding-level differences, so `fast - oracle` cannot stay at rounding level; what can be
    asked is that it grows no faster than the ORACLE's own response to a perturbation of the same size.  For starts
    on the docstring trajectory (C3: after 1 and after 10 years) and horizons of 20, 200, 2000 and 20 000 steps:
        eps    = the fast kernel's one-step difference from the oracle, relative, from that start (>= 1 ulp)
        R(h)   = max over s in (+1, -1, +2, -2) of | oracle(x0 * (1 + s eps)) - oracle(x0) |  after h steps
                 (the model's sensitivity: one perturbed run is one sample of a chaotic divergence whose size varies
                 by an order of magnitude from sample to sample, so R is the largest of a small perturbation ensemble)
        F(h)   = | fast(x0) - oracle(x0) |                after h steps
    per state variable, max over cells, both normalised by max(|oracle|, 1).  Asserted: F(h) <= 10 * max(R(h), rtol)
    with rtol = sqrt(eps(Float64)), the reference's own equality criterion (test/runtests.jl:44)."""
    par, f = _par(), ebm.Forcing(0.0)
    iv = [ebm.MIZ_VARS.index(k) for k in STATE]
    lines = []
    for years0 in (1, 10):
        st0 = ebm.SpaceTime(180, 2000, years0, "sin")
        o0 = oracle_miz(st0, [f], [par], [_zero(180)])
        init = ebm.Collection({k: o0[k][0].copy() for k in STATE})
        T0 = o0["T0"]
        # one step of the fast kernel vs the oracle from this state
        st1 = ebm.SpaceTime(180, 2000, 1, "sin")
        ob = oracle_miz(st1, [f], [par], [init], T0=T0, lastonly=False, raw=True)
        g1 = ebm.integrate_ensemble("MIZ", st1, [f], [par], [init], T0guess=T0, lastonly=False, field_stride=1)
        one = max(float(rel_err(g1.raw[0, 0, v], ob["raw"][0, 0, v]).max()) for v in iv)
        eps = max(one, 2.0 ** -52)
        perts = [ebm.Collection({k: (init[k] * (1.0 + sgn * eps) if k != "phi" else init[k].copy()) for k in STATE})
                 for sgn in (1.0, -1.0, 2.0, -2.0)]
        ops = [oracle_miz(st1, [f], [par], [pt], T0=T0, lastonly=False, raw=True) for pt in perts]
        st10 = ebm.SpaceTime(180, 2000, 10, "sin")
        ob10 = oracle_miz(st10, [f], [par], [init], T0=T0)
        ops10 = [oracle_miz(st10, [f], [par], [pt], T0=T0) for pt in perts]
        g10 = ebm.integrate_ensemble("MIZ", st10, [f], [par], [init], T0guess=T0)
        for h in (20, 200, 2000, 20000):
            for k, v in zip(STATE, iv):
                if h <= 2000:
                    base, prs, fs = ob["raw"][0, h - 1, v], [q["raw"][0, h - 1, v] for q in ops], g1.raw[0, h - 1, v]
                else:
                    base, prs, fs = ob10[k][0], [q[k][0] for q in ops10], g10.final[k][0]
                scale = max(float(np.abs(base).max()), 1.0)
                R = max(float(np.abs(pr - base).max()) for pr in prs) / scale
                F = float(np.abs(fs - base).max()) / scale
                lines.append(f"start year {years0:2d} eps {eps:.1e} horizon {h:6d} {k:3s}: fast-oracle {F:.2e}  oracle sensitivity {R:.2e}")
                assert F <= 10.0 * max(R, RTOL), lines[-1]
    with capsys.disabled():
        print("\n" + "\n".join(lines))
