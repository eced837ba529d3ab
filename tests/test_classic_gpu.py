"""GPU parity tests for the classic path: libebm_cuda (through the C ABI / host mirror) vs the CPU oracle.

Tolerance (SURVEY.md 8c, BASELINE.json north_star): |gpu - ref| <= 1e-9 * max(|ref|, 1) at every compared
sample for the fast kernel; the strict kernel and the one-step entry point must be bit-identical to the
oracle (same operation order, same cos table, IEEE division, no FMA contraction).
"""
import numpy as np
import pytest

import ebm_b200 as ebm
from helpers import (assert_close, classic_branch_flags, cold_init, forcing_rows, oracle_classic, oracle_diag_classic, rel_err,
                     warm_init)

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _par(**kw):
    p = ebm.default_parameters("Classic")
    p.update(kw)
    return p


def test_single_step_debug_menu_bitwise():
    """The `debug` seam of step! (src/classic.jl:67-69) as a fixed menu of the step's per-cell locals
    (EBM_DEBUG_*: alpha, C, T0, S, mask): bit-identical to the oracle's locals; an expression is refused."""
    import oracle
    st = ebm.SpaceTime(100, 2000, 1)
    par = _par()
    row = [par[k] for k in ebm.CLASSIC_PAR_ORDER]
    E0 = np.linspace(60.0, -25.0, 100)
    E0[40] = 0.0                                      # alpha = 0 at E == 0, T0 = C / -Inf = -0.0
    Tg0 = np.linspace(12.0, -14.0, 100)
    for name in ("alpha", "C", "T0", "S", "mask"):
        o = oracle.classic_step(st.x, st.t, row, 7, 1.25, E0, Tg0, debug=name)
        v = ebm.Collection(E=E0.copy(), Tg=Tg0.copy())
        ebm.step("Classic", st.t[6], 1.25, v, st, par, debug=name)
        assert np.array_equal(v.debug, o["debug"]), name
        assert np.array_equal(v.E, o["E"]) and np.array_equal(v.Tg, o["Tg"]) and np.array_equal(v.T, o["T"])
    with pytest.raises(ValueError):
        ebm.step("Classic", st.t[6], 1.25, ebm.Collection(E=E0.copy(), Tg=Tg0.copy()), st, par, debug="C .- T0")


def test_single_step_bitwise():
    """step!(Val(:Classic), ...) one step: bit-identical to the oracle, warm and cold states."""
    st = ebm.SpaceTime(100, 2000, 1)
    par = _par()
    for init, f in ((warm_init(100), 0.0), (cold_init(100), 3.5)):
        o = oracle_classic(ebm.SpaceTime(100, 2000, 1), [ebm.Forcing(f)], [par], [init], lastonly=False, raw=True)
        v = ebm.Collection(E=init.E.copy(), Tg=init.Tg.copy())
        ebm.step("Classic", st.t[0], f, v, st, par)
        assert np.array_equal(v.E, o["raw"][0, 0, 0])
        assert np.array_equal(v.T, o["raw"][0, 0, 1])
        assert np.array_equal(v.h, o["raw"][0, 0, 2])


def test_strict_kernel_bitwise_one_year():
    """C1a with the literal-arithmetic kernel, run for two years: every step of E, T, h (the raw slots of both years)
    and the final Tg bit-identical."""
    st = ebm.SpaceTime(100, 2000, 2)
    par, f, init = _par(), ebm.Forcing(0.0), warm_init(100)
    o = oracle_classic(st, [f], [par], [init], lastonly=False, raw=True, seasonal=True)
    r = ebm.integrate_ensemble("Classic", st, [f], [par], [init], lastonly=False, field_stride=1, strict=True)
    assert np.array_equal(r.raw[0], o["raw"][0])
    assert np.array_equal(r.final["Tg"], o["Tg"])
    # winter / summer snapshots are copies of raw steps -> identical; annual mean differs only by summation order
    assert np.array_equal(r.seasonal[0, :, :2], o["seasonal"][0, :, :2])
    assert rel_err(r.seasonal[0, :, 2], o["seasonal"][0, :, 2]).max() < 1e-12


def test_fast_kernel_one_year_every_step():
    """C1a: classic 1-year, warm start, every step of E, T, h within 1e-9."""
    st = ebm.SpaceTime(100, 2000, 1)
    par, f, init = _par(), ebm.Forcing(0.0), warm_init(100)
    o = oracle_classic(st, [f], [par], [init], lastonly=False, raw=True)
    sols = ebm.integrate("Classic", st, f, par, init, lastonly=False)
    for vi, v in enumerate(("E", "T", "h")):
        err = rel_err(sols.raw[v], o["raw"][0, :, vi])
        assert err.max() < TOL, (v, err.max(), np.unravel_index(err.argmax(), err.shape))
    assert rel_err(sols.final["Tg"], o["Tg"][0]).max() < TOL
    assert len(sols.ts) == 2000 and abs(sols.ts[0] - 0.00025) < 1e-15


def test_fast_kernel_thirty_years_lastonly():
    """C2: 30-year spin-up, lastonly: last-year raw, all seasonal fields, final state."""
    st = ebm.SpaceTime(100, 2000, 30)
    par, f, init = _par(), ebm.Forcing(0.0), warm_init(100)
    o = oracle_classic(st, [f], [par], [init], lastonly=True, raw=True, seasonal=True)
    sols = ebm.integrate("Classic", st, f, par, init)
    for vi, v in enumerate(("E", "T", "h")):
        assert rel_err(sols.raw[v], o["raw"][0, :, vi]).max() < TOL, v
        for si, season in enumerate(("winter", "summer", "avg")):
            assert rel_err(sols.seasonal[season][v], o["seasonal"][0, :, si, vi]).max() < TOL, (v, season)
    assert abs(sols.ts[0] - 29.00025) < 1e-12
    # WE15-like climate at year 30 (SURVEY Appendix D probe)
    hm = ebm.hemispheric_mean(sols.seasonal.avg.T[29], st.x)
    assert 16.9 < hm < 17.1


def _ensemble(nmem, nx):
    forcings, pars, inits = [], [], []
    for m in range(nmem):
        F = -20.0 + 40.0 * (m // 2) / max(nmem // 2 - 1, 1)
        forcings.append(ebm.Forcing(F))
        pars.append(_par(D=0.45 + 0.3 * (m % 7) / 6.0, B=1.9 + 0.05 * (m % 5)))
        inits.append(warm_init(nx) if m % 2 == 0 else cold_init(nx))
    return forcings, pars, inits


@pytest.mark.parametrize("nmem,nx,nt,lastonly", [
    pytest.param(70, 100, 2000, True, id="70-100-2000"), pytest.param(33, 60, 1000, True, id="33-60-1000"),
    pytest.param(5, 37, 500, True, id="5-37-500"), pytest.param(40, 180, 2000, True, id="40-180-2000"),
    # raw output of every year (8-band and 16-band grids)
    pytest.param(8, 60, 1000, False, id="8-60-1000-all-years"), pytest.param(4, 180, 2000, False, id="4-180-2000-all-years")])
def test_ensemble_diag_fields_and_state(nmem, nx, nt, lastonly):
    """Ragged member counts / other grids: L0 diagnostics, L1/L2 fields of strided members, final state."""
    st = ebm.SpaceTime(nx, nt, 3)
    forcings, pars, inits = _ensemble(nmem, nx)
    o = oracle_classic(st, forcings, pars, inits, lastonly=lastonly, raw=True, seasonal=True)
    r = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=3, lastonly=lastonly)
    assert r.flags.max() == 0
    # E integrates cg_tau*Tg = 9800*Tg (classic.jl:48): a rounding difference of 1e-13 in the ghost-layer solve is
    # 1e-9 in the tendency.  At the BASELINE grid (nx = 100) everything stays under 1e-9; the finer 180-cell grid
    # (stiffer matrix, not a BASELINE configuration) is held to 1e-8.
    tol = TOL if nx <= 100 else 1e-8
    assert_close(r.final["E"], o["E"], tol, "final E")
    assert_close(r.final["Tg"], o["Tg"], tol, "final Tg")
    sel = np.arange(0, nmem, 3)
    # flagged-cell accounting (SURVEY 8c): cell-steps within 1e-6 of the branch threshold E = 0, or whose ice mask
    # differs from the oracle's, are counted, printed, must be rare and must stay under 1e-6
    flags = classic_branch_flags(r.raw, o["raw"][sel])
    nflag = assert_close(r.raw, o["raw"][sel], tol, "raw", flag=flags)
    print(f"classic ensemble {nmem} x nx {nx} x nt {nt}: {nflag // 3} flagged cell-steps of {flags.size // 3}")
    assert_close(r.seasonal, o["seasonal"][sel], tol, "seasonal")
    od = oracle_diag_classic(o["seasonal"], st.x)
    assert_close(r.diag[..., :2], od[..., :2], tol, "diag")
    # ice area / edge are step functions of the sign of E: equal unless a cell sits within 1e-9 of zero
    near0 = (np.abs(o["seasonal"][:, :, :, 0, :]) < 1e-9).any(axis=-1)
    mism = (np.abs(r.diag[..., 2:] - od[..., 2:]) > 1e-9).any(axis=-1)
    assert not (mism & ~near0).any()


def test_ramp_forcing_and_chained_launches():
    """Forcing{false} evaluated per step on the device; splitting the run into launches changes nothing."""
    st = ebm.SpaceTime(100, 2000, 6)
    forcings = [ebm.Forcing(0.0, 4.0, -2.0, (1, 1), (2.0, -3.0)), ebm.Forcing(-1.0, 1.0, -1.0, (0, 2), (1.0, -1.0)),
                ebm.Forcing(2.5)]
    pars = [_par()] * 3
    inits = [warm_init(100), cold_init(100), warm_init(100)]
    o = oracle_classic(st, forcings, pars, inits, seasonal=True)
    a = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=1, lastonly=False)
    b = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=1, lastonly=False, years_per_launch=2)
    assert rel_err(a.seasonal, o["seasonal"]).max() < TOL
    assert np.array_equal(a.final["E"], b.final["E"]) and np.array_equal(a.final["Tg"], b.final["Tg"])
    assert a.raw.shape[1] == 6 * 2000 and np.array_equal(a.raw, b.raw)
    assert np.array_equal(np.nan_to_num(a.seasonal), np.nan_to_num(b.seasonal))
    assert np.array_equal(a.diag, b.diag)


def test_energy_budget_and_thickness_invariants():
    """Size-independent properties on a 2048-member ensemble: h = -E/Lf*(E<0) >= 0, T = E/cw where E >= 0,
    finite state, and the two hysteresis branches are both populated."""
    nmem, nx = 2048, 100
    st = ebm.SpaceTime(nx, 2000, 2)
    par = _par()
    forcings = [ebm.Forcing(-20.0 + 40.0 * (m % 1024) / 1023.0) for m in range(nmem)]
    inits = [warm_init(nx) if m < 1024 else cold_init(nx) for m in range(nmem)]
    r = ebm.integrate_ensemble("Classic", st, forcings, [par] * nmem, inits, field_stride=64)
    assert r.flags.max() == 0 and np.isfinite(r.final["E"]).all() and np.isfinite(r.final["Tg"]).all()
    E, T, h = r.raw[:, :, 0], r.raw[:, :, 1], r.raw[:, :, 2]
    assert (h >= 0).all()
    assert np.allclose(h, np.where(E < 0, -E / par.Lf, 0.0), rtol=1e-14, atol=0)
    # T of step i is computed from E BEFORE that step's Euler update (classic.jl:51 precedes :53)
    Ep, Tn = E[:, :-1], T[:, 1:]
    assert np.allclose(Tn[Ep >= 0], Ep[Ep >= 0] / par.cw, rtol=1e-13, atol=0)
    assert (Tn[Ep < 0] <= 0).all()
    area = r.diag[:, -1, 2, 2]
    assert area[:1024].min() < 0.5 and area[1024:].max() > 5.0   # warm branch ice-free, cold branch snowball
    # spot-check 8 members against the oracle
    idx = list(range(0, nmem, 256))
    o = oracle_classic(st, [forcings[i] for i in idx], [par] * len(idx), [inits[i] for i in idx])
    assert rel_err(r.final["E"][idx], o["E"]).max() < TOL


def test_restart_through_checkpoint_file_is_exact(tmp_path):
    """SURVEY 8f.3: the classic model restarts exactly from the returned (E, Tg) -- the reference cannot, Tg is not a
    stored variable (infrastructure.jl:621).  4 years == 2 + 2 years through a checkpoint file, bit for bit."""
    par = _par()
    forcings = [ebm.Forcing(-3.0), ebm.Forcing(0.0, 4.0, -2.0, (1, 0), (2.0, -6.0))]   # constant, and a ramp over years 1..3
    inits = [cold_init(100), warm_init(100)]
    full = ebm.integrate_ensemble("Classic", ebm.SpaceTime(100, 2000, 4), forcings, [par] * 2, inits)
    st2 = ebm.SpaceTime(100, 2000, 2)
    a = ebm.integrate_ensemble("Classic", st2, forcings, [par] * 2, inits)
    path = str(tmp_path / "classic.ebm")
    ebm.save_state(path, a.final, years_done=2)
    state, years = ebm.load_state(path)
    inits2, _ = ebm.inits_from_state(state)
    b = ebm.integrate_ensemble("Classic", st2, forcings, [par] * 2, inits2, start_year=years)   # Forcing sees T + 2
    assert years == 2
    assert np.array_equal(full.final["E"], b.final["E"]) and np.array_equal(full.final["Tg"], b.final["Tg"])
    assert np.array_equal(full.diag[:, 2:], b.diag)


def test_c4_members_two_hundred_years():
    """BASELINE config C4 (SURVEY 8d): 32 evenly spaced members of the 65 536-member hysteresis sweep -- F = -20..+20,
    even members warm start, odd members cold start -- integrated for the full 200 years: final state and the last
    year's diagnostics against the oracle.  Tolerance 5e-9 here: after 400 000 steps the cells of the seasonal ice zone
    (|E| < 1, where E integrates cg_tau*Tg = 9800*Tg and a 1e-13 rounding difference in the ghost-layer solve is 1e-9
    in the tendency) sit at 1.4e-9 absolute; everything else stays under 1e-9, as do the 1-year and 30-year runs that
    the stated tolerance (BASELINE.json: "after one year") refers to.  The oracle's own two solvers (tridiagonal vs
    the reference's dense LU) differ by the same amount on such cells (SURVEY 8c probe: 7e-9 relative)."""
    N, H, nsub = 65536, 32768, 32
    idx = [int(round(k * (N - 1) / (nsub - 1))) for k in range(nsub)]
    st = ebm.SpaceTime(100, 2000, 200)
    par = _par()
    forcings = [ebm.Forcing(-20.0 + 40.0 * (m // 2) / (H - 1)) for m in idx]
    inits = [warm_init(100) if m % 2 == 0 else cold_init(100) for m in idx]
    o = oracle_classic(st, forcings, [par] * nsub, inits, seasonal=True)
    r = ebm.integrate_ensemble("Classic", st, forcings, [par] * nsub, inits)
    assert r.flags.max() == 0
    marginal = np.abs(o["E"]) < 1.0
    assert_close(r.final["E"], o["E"], 5e-9, "final E after 200 y")
    assert_close(np.where(marginal, 0.0, r.final["E"]), np.where(marginal, 0.0, o["E"]), TOL, "final E outside the seasonal ice zone")
    assert_close(r.final["Tg"], o["Tg"], TOL, "final Tg after 200 y")
    od = oracle_diag_classic(o["seasonal"][:, -1:], st.x)
    assert_close(r.diag[:, -1:, :, :2], od[..., :2], TOL, "year-200 mean T / mean E")
    near0 = (np.abs(o["seasonal"][:, -1:, :, 0, :]) < 1e-9).any(axis=-1)
    mism = (np.abs(r.diag[:, -1:, :, 2:] - od[..., 2:]) > 1e-9).any(axis=-1)
    assert not (mism & ~near0).any()
    # the sample covers both ends of the hysteresis loop: a nearly ice-free warm-branch member and snowball members
    area = r.diag[:, -1, 2, 2]
    assert area.min() < 0.5 and area.max() > 6.0


def test_c4_sweep_two_thousand_members_two_years():
    """BASELINE config C4 at width: every 32nd member of the 65 536-member hysteresis sweep (2048 members, both
    branches, F = -20..+20) through the launch-uniform-parameter instance, two years from the sweep's initial states
    (freeze-up of the cold branch, melt-back of the warm one): final state and every diagnostic against the oracle at
    the stated tolerance, member by member; flagged samples (enthalpy within 1e-6 of the branch threshold, or ice mask
    differing from the oracle's) are counted and must be rare."""
    N, H, stride = 65536, 32768, 32
    idx = list(range(0, N, stride))
    nsub = len(idx)
    st = ebm.SpaceTime(100, 2000, 2)
    par = _par()
    forcings = [ebm.Forcing(-20.0 + 40.0 * (m // 2) / (H - 1)) for m in idx]
    inits = [warm_init(100) if (m // stride) % 2 == 0 else cold_init(100) for m in idx]   # idx is even: alternate the branch
    o = oracle_classic(st, forcings, [par] * nsub, inits, seasonal=True)
    r = ebm.integrate_ensemble("Classic", st, forcings, [par] * nsub, inits)
    assert r.flags.max() == 0
    fE = (np.abs(o["E"]) < 1e-6) | ((r.final["E"] < 0) != (o["E"] < 0))
    nflag = assert_close(r.final["E"], o["E"], TOL, "final E after 2 y", flag=fE)
    assert_close(r.final["Tg"], o["Tg"], TOL, "final Tg after 2 y")
    od = oracle_diag_classic(o["seasonal"], st.x)
    assert_close(r.diag[..., :2], od[..., :2], TOL, "mean T / mean E, both years, three seasons")
    near0 = (np.abs(o["seasonal"][:, :, :, 0, :]) < 1e-9).any(axis=-1)
    mism = (np.abs(r.diag[..., 2:] - od[..., 2:]) > 1e-9).any(axis=-1)
    assert not (mism & ~near0).any()
    print(f"C4 sample: {nsub} members x 2 y, {nflag} flagged cells of {fE.size}; ice area range {r.diag[:, -1, 2, 2].min():.2f}..{r.diag[:, -1, 2, 2].max():.2f}")


def test_sweep_of_non_matrix_parameters_takes_the_table_driven_kernel():
    """A, B, cw, S1, ai, Fb, k, Lf may differ per member inside a 32-member group of the fast (table-driven) kernel --
    only D, cg, tau, S0, S2, a0, a2 build its shared tables.  70 members sweeping B, A, ai, k and the forcing."""
    nmem, nx = 70, 100
    st = ebm.SpaceTime(nx, 2000, 3)
    forcings = [ebm.Forcing(-6.0 + 12.0 * (m % 9) / 8.0) for m in range(nmem)]
    pars = [_par(B=1.9 + 0.05 * (m % 6), A=190.0 + (m % 4), ai=0.38 + 0.01 * (m % 5), k=1.8 + 0.1 * (m % 3)) for m in range(nmem)]
    inits = [warm_init(nx) if m % 2 == 0 else cold_init(nx) for m in range(nmem)]
    o = oracle_classic(st, forcings, pars, inits, raw=True, seasonal=True)
    lib = ebm._lib.load()
    n0 = lib.ebm_launch_count()
    r = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=5)
    assert lib.ebm_launch_count() > n0 and r.flags.max() == 0
    assert_close(r.final["E"], o["E"], TOL, "final E")
    assert_close(r.final["Tg"], o["Tg"], TOL, "final Tg")
    sel = np.arange(0, nmem, 5)
    assert_close(r.raw, o["raw"][sel], TOL, "raw")
    assert_close(r.seasonal, o["seasonal"][sel], TOL, "seasonal")
    assert_close(r.diag[..., :2], oracle_diag_classic(o["seasonal"], st.x)[..., :2], TOL, "diag")


def test_interleaved_parameter_sets_are_regrouped():
    """Three parameter sets (different D, a0) interleaved member by member, warm and cold starts mixed: the host entry
    point groups members by table-parameter set and regime before the launch; every output (diagnostics, strided
    fields, final state, flags) comes back in the caller's order."""
    nmem, nx = 192, 100
    st = ebm.SpaceTime(nx, 2000, 2)
    sets = [_par(), _par(D=0.5, a0=0.68), _par(D=0.7)]
    pars = [sets[m % 3] for m in range(nmem)]
    forcings = [ebm.Forcing(-8.0 + 16.0 * (m // 6) / (nmem // 6 - 1)) for m in range(nmem)]
    inits = [warm_init(nx) if (m // 3) % 2 == 0 else cold_init(nx) for m in range(nmem)]
    o = oracle_classic(st, forcings, pars, inits, raw=True, seasonal=True)
    r = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=7)
    assert r.flags.max() == 0
    assert_close(r.final["E"], o["E"], TOL, "final E")
    assert_close(r.final["Tg"], o["Tg"], TOL, "final Tg")
    sel = np.arange(0, nmem, 7)
    assert_close(r.raw, o["raw"][sel], TOL, "raw")
    assert_close(r.seasonal, o["seasonal"][sel], TOL, "seasonal")
    assert_close(r.diag[..., :2], oracle_diag_classic(o["seasonal"], st.x)[..., :2], TOL, "diag")


def test_device_entry_point_with_member_index():
    """ebm_classic_run_device (inputs resident in HBM, torch tensors as the allocator): the members are handed over
    in a shuffled order with member_index = original index of each slot; diagnostics and flags land at the original
    rows, and every member's result equals the host entry point's bit for bit (members are independent)."""
    import ctypes as C
    import torch
    from ebm_b200 import _lib
    nmem, nx, years = 96, 100, 2
    st = ebm.SpaceTime(nx, 2000, years)
    p = _par()
    par = np.tile([p[k] for k in ebm.CLASSIC_PAR_ORDER], (nmem, 1))
    forc = np.zeros((nmem, 10)); forc[:, :3] = np.linspace(-12.0, 12.0, nmem)[:, None]
    warm = (np.arange(nmem) % 3) != 0
    state = {"E": np.where(warm[:, None], 98.0, -9.5) * np.ones((nmem, nx)), "Tg": np.where(warm[:, None], 10.0, -10.0) * np.ones((nmem, nx))}
    ref = ebm.integrate_arrays("Classic", st, forc, par, state)
    perm = np.random.default_rng(5).permutation(nmem)                      # slot -> original index
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_par, d_forc = t(par[perm].T), t(forc[perm].T)
    d_E, d_Tg = t(state["E"][perm].T), t(state["Tg"][perm].T)
    d_diag = torch.full((nmem, years, 3, 4), float("nan"), dtype=torch.float64, device=dev)
    d_flags = torch.zeros(nmem, dtype=torch.int32, device=dev)
    d_idx = t(perm.astype(np.int64))
    lib = _lib.load()
    grid, opt = _lib.make_grid(st), _lib.make_options(device=0)
    args = _lib.ClassicDeviceArgs(nmem, d_par.data_ptr(), d_forc.data_ptr(), d_E.data_ptr(), d_Tg.data_ptr(),
                                  d_diag.data_ptr(), None, None, d_flags.data_ptr(), d_idx.data_ptr())
    _lib.check(lib.ebm_classic_run_device(C.byref(grid), C.byref(args), C.byref(opt), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert np.array_equal(d_diag.cpu().numpy(), ref.diag)                  # rows at the original member index
    assert int(d_flags.max().item()) == 0
    E_fin = np.empty((nmem, nx)); E_fin[perm] = d_E.cpu().numpy().T        # state stays in slot order
    Tg_fin = np.empty((nmem, nx)); Tg_fin[perm] = d_Tg.cpu().numpy().T
    assert np.array_equal(E_fin, ref.final["E"]) and np.array_equal(Tg_fin, ref.final["Tg"])


@pytest.mark.parametrize("rows,cols", [(70001, 37), (37, 70001), (1, 5), (2100000, 3)])
def test_transpose_device_layout_helper(rows, cols):
    """ebm_transpose_device: [rows][cols] -> [cols][rows] for member counts beyond 65535*32 on either axis."""
    import ctypes as C
    import torch
    from ebm_b200 import _lib
    lib = _lib.load()
    src = torch.arange(rows * cols, dtype=torch.float64, device="cuda").reshape(rows, cols)
    dst = torch.empty((cols, rows), dtype=torch.float64, device="cuda")
    _lib.check(lib.ebm_transpose_device(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), rows, cols,
                                        C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert torch.equal(dst, src.t().contiguous())


@pytest.mark.parametrize("nx", [180, 208, 130])
def test_sixteen_band_table_driven_instance(nx):
    """104 < nx <= 208 with uniform table-building parameters: the 16-band instance of the table-driven kernel
    (8 warps per CTA).  Forcing, B and the initial branch vary per member; fields of every 6th member."""
    nmem = 40
    st = ebm.SpaceTime(nx, 2000, 2)
    forcings = [ebm.Forcing(-8.0 + 16.0 * m / (nmem - 1)) for m in range(nmem)]
    pars = [_par(B=2.0 + 0.05 * (m % 4)) for m in range(nmem)]
    inits = [warm_init(nx) if m % 2 == 0 else cold_init(nx) for m in range(nmem)]
    o = oracle_classic(st, forcings, pars, inits, raw=True, seasonal=True)
    r = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=6)
    assert r.flags.max() == 0
    tol = 1e-8                                     # finer grids: see test_ensemble_diag_fields_and_state
    assert_close(r.final["E"], o["E"], tol, "final E")
    assert_close(r.final["Tg"], o["Tg"], tol, "final Tg")
    sel = np.arange(0, nmem, 6)
    assert_close(r.raw, o["raw"][sel], tol, "raw")
    assert_close(r.seasonal, o["seasonal"][sel], tol, "seasonal")
    assert_close(r.diag[..., :2], oracle_diag_classic(o["seasonal"], st.x)[..., :2], tol, "diag")


@pytest.mark.parametrize("nx,lastonly", [pytest.param(230, True, id="230"), pytest.param(250, True, id="250"),
                                         pytest.param(250, False, id="250-all-years")])   # raw output of both years
def test_band_kernel_large_grids(nx, lastonly):
    """208 < nx <= 256: the band kernel (16 cells per band, 16 members per CTA).  nx = 230 needs 15 bands -- an odd
    count, which the launcher pads to whole warps (ADVICE r1: no thread may shadow another thread's band)."""
    nmem = 20 if lastonly else 5
    st = ebm.SpaceTime(nx, 2000, 2)
    forcings = [ebm.Forcing(-8.0 + 16.0 * m / (nmem - 1)) for m in range(nmem)]
    pars = [_par(B=2.0 + 0.05 * (m % 4)) for m in range(nmem)]
    inits = [warm_init(nx) if m % 2 == 0 else cold_init(nx) for m in range(nmem)]
    o = oracle_classic(st, forcings, pars, inits, lastonly=lastonly, raw=True, seasonal=True)
    r = ebm.integrate_ensemble("Classic", st, forcings, pars, inits, field_stride=4, lastonly=lastonly)
    assert r.flags.max() == 0
    tol = 2e-8                                     # finer grids: see test_ensemble_diag_fields_and_state
    assert_close(r.final["E"], o["E"], tol, "final E")
    assert_close(r.final["Tg"], o["Tg"], tol, "final Tg")
    sel = np.arange(0, nmem, 4)
    assert_close(r.raw, o["raw"][sel], tol, "raw")
    assert_close(r.seasonal, o["seasonal"][sel], tol, "seasonal")
    assert_close(r.diag[..., :2], oracle_diag_classic(o["seasonal"], st.x)[..., :2], tol, "diag")


def _ndev():
    return ebm._lib.load().ebm_device_count()


@pytest.mark.parametrize("diag_on_device", [False, True])
def test_multi_gpu_entry_point_matches_single_gpu_bitwise(diag_on_device):
    """ebm_classic_run_multi (one host thread + stream per GPU inside the library, members dealt in packets after the
    regime sort): every output row equals the single-GPU call's bit for bit.  With diag_on_device the diagnostics of
    the other GPU arrive in device memory of GPU 0 over NCCL (communicator owned by the library).  Runs on one GPU
    too (one device = the degenerate deal)."""
    import ctypes as C
    import torch
    from ebm_b200 import _lib
    ndev = min(_ndev(), 2)
    nmem, nx, years = 200, 100, 2
    st = ebm.SpaceTime(nx, 2000, years)
    p = _par()
    par = np.tile([p[k] for k in ebm.CLASSIC_PAR_ORDER], (nmem, 1))
    forc = np.zeros((nmem, 10)); forc[:, :3] = np.linspace(-15.0, 15.0, nmem)[:, None]
    warm = (np.arange(nmem) % 3) != 0
    state = {"E": np.where(warm[:, None], 98.0, -9.5) * np.ones((nmem, nx)), "Tg": np.where(warm[:, None], 10.0, -10.0) * np.ones((nmem, nx))}
    ref = ebm.integrate_arrays("Classic", st, forc, par, state, field_stride=7)
    if not diag_on_device:
        r = ebm.integrate_arrays("Classic", st, forc, par, state, devices=list(range(ndev)), packet=16, field_stride=7)
        assert np.array_equal(r.diag, ref.diag)
        # field outputs: rows of the members whose ORIGINAL index is a multiple of the stride, whatever GPU ran them
        assert r.seasonal.shape == ref.seasonal.shape and np.array_equal(r.seasonal, ref.seasonal, equal_nan=True)
        assert np.array_equal(r.raw, ref.raw, equal_nan=True)
    else:
        lib = _lib.load()
        d_diag = torch.full((nmem, years, 3, 4), float("nan"), dtype=torch.float64, device="cuda:0")
        E_fin, Tg_fin = np.empty((nmem, nx)), np.empty((nmem, nx))
        flags = np.zeros(nmem, dtype=np.int32)
        out = _lib.ClassicOutputs(C.cast(d_diag.data_ptr(), C.POINTER(C.c_double)), None, None, _lib.dptr(E_fin), _lib.dptr(Tg_fin),
                                  flags.ctypes.data_as(C.POINTER(C.c_int32)))
        grid, opt = _lib.make_grid(st), _lib.make_options()
        multi = _lib.make_multi(devices=list(range(ndev)), diag_device=0, packet=16)
        _lib.check(lib.ebm_classic_run_multi(C.byref(grid), nmem, _lib.dptr(np.ascontiguousarray(par)), _lib.dptr(np.ascontiguousarray(forc)),
                                             _lib.dptr(state["E"]), _lib.dptr(state["Tg"]), C.byref(opt), C.byref(multi), C.byref(out)))
        torch.cuda.synchronize()
        assert np.array_equal(d_diag.cpu().numpy(), ref.diag)

        class R: pass
        r = R(); r.final = {"E": E_fin, "Tg": Tg_fin}; r.flags = flags
    assert np.array_equal(r.final["E"], ref.final["E"]) and np.array_equal(r.final["Tg"], ref.final["Tg"])
    assert np.array_equal(r.flags, ref.flags)


def test_wave_balanced_launch_is_bit_identical():
    """A member count that leaves the last wave of CTAs nearly empty takes the wave-balanced launch (ranges of CTAs on
    several streams, advancing in chunks of years): bit-identical to one launch."""
    import os, subprocess, sys
    code = r"""
import sys, numpy as np
sys.path.insert(0, %r)
import ebm_b200 as ebm
lib = ebm._lib.load()
slots = 148 * 3
nmem, nx, years = (slots + 40) * 16, 100, 8
st = ebm.SpaceTime(nx, 2000, years)
p = ebm.default_parameters("Classic")
par = np.tile([p[k] for k in ebm.CLASSIC_PAR_ORDER], (nmem, 1))
forc = np.zeros((nmem, 10)); forc[:, :3] = np.linspace(-18.0, 18.0, nmem)[:, None]
warm = (np.arange(nmem) %% 2) == 0
state = {"E": np.where(warm[:, None], 98.0, -9.5) * np.ones((nmem, nx)), "Tg": np.where(warm[:, None], 10.0, -10.0) * np.ones((nmem, nx))}
n0 = lib.ebm_launch_count()
r = ebm.integrate_arrays("Classic", st, forc, par, state)
print("LAUNCHES", lib.ebm_launch_count() - n0)
np.save(sys.argv[1], np.concatenate([r.final["E"].ravel(), r.final["Tg"].ravel(), np.nan_to_num(r.diag).ravel()]))
""" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))),)
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        outs = []
        for tag, env in (("a", {}), ("b", {"EBM_NO_WAVE_BALANCE": "1"})):
            path = os.path.join(tmp, tag + ".npy")
            r = subprocess.run([sys.executable, "-c", code, path], env=dict(os.environ, **env), capture_output=True, text=True)
            assert r.returncode == 0, r.stderr[-2000:]
            outs.append((np.load(path), int(r.stdout.split("LAUNCHES")[1].split()[0])))
        (a, la), (b, lb) = outs
        assert np.array_equal(a, b)
        assert la > lb    # the balanced path really ran: many chunked launches instead of a few


@pytest.mark.parametrize("xfunc,nx", [("sin", 100), ("sin", 60), ("identity", 100), ("sin", 180)])
def test_generic_stencil_extension(xfunc, nx):
    """ebm_options_t.classic_stencil = 1 (SURVEY 8f-4): the classic model with the generic flux-form stencil in kappa --
    a non-symmetric tridiagonal matrix on non-uniform grids.  Fast kernel (table-driven and per-member-coefficient
    instances, 8 and 16 bands) within tolerance of the oracle, literal kernel bit-identical; the default (0) keeps the
    reference's behaviour (get_diffop whatever the grid)."""
    nmem = 36
    st = ebm.SpaceTime(nx, 2000, 2, xfunc)
    forcings = [ebm.Forcing(-10.0 + 20.0 * m / (nmem - 1)) for m in range(nmem)]
    pars = [_par(B=2.0 + 0.05 * (m % 4)) if m < 32 else _par(D=0.5 + 0.05 * (m % 4)) for m in range(nmem)]   # last group: per-member D
    inits = [warm_init(nx) if m % 2 == 0 else cold_init(nx) for m in range(nmem)]
    o = oracle_classic(st, forcings, pars, inits, raw=True, seasonal=True, stencil=1)
    state = {"E": np.stack([i.E for i in inits]), "Tg": np.stack([i.Tg for i in inits])}
    from helpers import classic_rows
    r = ebm.integrate_arrays("Classic", st, forcing_rows(forcings), classic_rows(pars), state, field_stride=5, classic_stencil=1)
    assert r.flags.max() == 0
    tol = TOL if nx <= 100 else 1e-8
    assert_close(r.final["E"], o["E"], tol, "final E")
    assert_close(r.final["Tg"], o["Tg"], tol, "final Tg")
    sel = np.arange(0, nmem, 5)
    assert_close(r.raw, o["raw"][sel], tol, "raw")
    assert_close(r.diag[..., :2], oracle_diag_classic(o["seasonal"], st.x)[..., :2], tol, "diag")
    rs = ebm.integrate_arrays("Classic", st, forcing_rows(forcings[:4]), classic_rows(pars[:4]), {k: v[:4] for k, v in state.items()},
                              strict=True, classic_stencil=1)
    assert np.array_equal(rs.final["E"], o["E"][:4]) and np.array_equal(rs.final["Tg"], o["Tg"][:4])
    if xfunc == "sin":       # the default still reproduces the reference's behaviour on this grid
        od = oracle_classic(st, forcings[:4], pars[:4], inits[:4])
        rd = ebm.integrate_arrays("Classic", st, forcing_rows(forcings[:4]), classic_rows(pars[:4]), {k: v[:4] for k, v in state.items()})
        assert_close(rd.final["E"], od["E"], tol, "default stencil")


def test_integrate_grids_per_member_grids():
    """SURVEY 8f-4, second half: members on different grids (nx, nt, duration) in one call.  integrate_grids groups the
    members by SpaceTime (a launch integrates one grid) and addresses the results by the caller's member index; a
    member's result is bit-identical to integrating it alone, and within tolerance of the oracle."""
    p = ebm.default_parameters("Classic")
    specs = [(100, 2000, 1), (60, 1000, 2), (100, 2000, 1), (150, 2000, 1), (60, 1000, 2), (37, 500, 1)]
    sts = [ebm.SpaceTime(nx, nt, dur) for nx, nt, dur in specs]
    forcings = [ebm.Forcing(-6.0 + 3.0 * m) for m in range(len(specs))]
    pars = [p] * len(specs)
    inits = [ebm.Collection(E=np.full(st.nx, 98.0 if m % 2 == 0 else -9.5), Tg=np.full(st.nx, 10.0 if m % 2 == 0 else -10.0))
             for m, st in enumerate(sts)]
    res = ebm.integrate_grids("Classic", sts, forcings, pars, inits)
    assert len(res.groups) == 4 and [len(g[1]) for g in res.groups] == [2, 2, 1, 1]
    for m, st in enumerate(sts):
        one = ebm.integrate_ensemble("Classic", st, [forcings[m]], [pars[m]], [inits[m]])
        got = res.member(m)
        assert (got["spacetime"].nx, got["spacetime"].nt, got["spacetime"].dur) == (st.nx, st.nt, st.dur)
        assert got["diag"].shape == (st.dur, 3, 4)
        for k in ("E", "Tg"):
            assert np.array_equal(got["final"][k], one.final[k][0]), (m, k)
        assert np.array_equal(got["diag"], one.diag[0], equal_nan=True)
        o = oracle_classic(st, [forcings[m]], [pars[m]], [inits[m]])
        tol = 1e-9 if st.nx <= 100 else 1e-8
        assert_close(got["final"]["E"], o["E"][0], tol, f"member {m} E")


def test_launch_uniform_parameter_instance_is_bit_identical():
    """A forcing sweep (every member has the same 15 parameters) takes the launch-uniform-parameter instance of the
    kernel: member constants derived on the host and read as constant-bank operands.  Same bits as the per-member
    instance (EBM_NO_UPAR=1), warm and cold starts, constant and ramp forcing, with field output."""
    import os
    nmem, nx = 96, 100
    st = ebm.SpaceTime(nx, 2000, 2)
    par = _par()
    forcings = [ebm.Forcing(-18.0 + 36.0 * m / (nmem - 1)) if m % 5 else ebm.Forcing(-2.0, 6.0, 1.0, holdyrs=(0, 0), rates=(4.0, -5.0))
                for m in range(nmem)]
    inits = [warm_init(nx) if m % 2 == 0 else cold_init(nx) for m in range(nmem)]
    runs = []
    for flag in (None, "1"):
        if flag is None:
            os.environ.pop("EBM_NO_UPAR", None)
        else:
            os.environ["EBM_NO_UPAR"] = flag
        try:
            runs.append(ebm.integrate_ensemble("Classic", st, forcings, [par] * nmem, inits, field_stride=16))
        finally:
            os.environ.pop("EBM_NO_UPAR", None)
    a, b = runs
    for k in ("E", "Tg"):
        assert np.array_equal(a.final[k], b.final[k]), k
    assert np.array_equal(a.diag, b.diag, equal_nan=True)
    assert np.array_equal(a.seasonal, b.seasonal, equal_nan=True) and np.array_equal(a.raw, b.raw, equal_nan=True)
