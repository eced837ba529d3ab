#!/usr/bin/env python
"""bench.py -- member-years/s of the classic-EBM hysteresis ensemble (BASELINE.json config C4) on B200.

One "step" = one full pass of the hot path over the workload: N_members x 200 simulated years of the
classic EBM (nx=100, nt=2000), L0 diagnostics for every member-year.

  value  : device-resident throughput (inputs already in HBM, ebm_classic_run_device on torch's stream),
           CUDA-event timed, max over ranks; plus the NCCL gather of the diagnostics when N > 1.
  e2e    : same metric through the host-buffer C-ABI call ebm_classic_run (pinned host inputs, H2D, kernel,
           D2H of diagnostics + final state inside the timed region).
  roofline : FP64.  achieved = 37 FLOP/cell-step x nx x nt x member-years of one launch / its duration;
           peak = DFMA throughput measured in this run (MEASURED_PEAKS.json has no FP64 entry).
  cpu_baseline : the C oracle (a port of the reference's algorithm, tridiagonal solve) with OpenMP on all
           host cores, on a bounded sample of the same workload.

  kernel_ms_per_rank : CUDA-event time of the integrate call on every rank (min / max / all): load balance.
  strong   : (N > 1) the fixed 65 536-member sweep dealt over the N ranks -- strong scaling beside the weak headline.
  miz      : the C5 MIZ parameter sweep, 131 072 members x 5 years per GPU (N = 8: the full 16^5 grid), a few steps:
           value, roofline, e2e, cpu_baseline, NaN census (value_finite_members counts finite members only).

Every rank integrates the members `ebm.member_deal` hands it: 32-member packets dealt round-robin after a sort by
initial regime (a contiguous cut gives one rank all the expensive members; round-1 VERDICT).

`--impl reference` times that CPU implementation alone (rank 0 only).

`--dump-outputs DIR` writes what the last timed step of the headline pass (and of the MIZ sub-record) returned, for a
fixed seeded sample of members, so that two builds of the project can be compared output for output: the inputs are
the same from run to run for the same arguments.  Sampled members whose outputs are not finite are left out.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_CELL_STEP = {"classic": 37.0, "miz": 173.0}   # SURVEY.md Appendix E
NOMINAL_FP64_TFLOPS = 37.2                               # 148 SM x 64 FMA/clk x 2 x 1.965 GHz


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="classic", choices=["classic", "miz"])
    ap.add_argument("--members", type=int, default=0, help="members per GPU (default: 65536 classic, 131072 miz)")
    ap.add_argument("--years", type=int, default=0, help="simulated years (default: 200 classic, 50 miz)")
    ap.add_argument("--cpu-sample-members", type=int, default=0)
    ap.add_argument("--order", default="interleaved", choices=["branch", "interleaved"],
                    help="classic member order: SURVEY 8d's C4 definition (even members warm start, odd members cold start; "
                         "default) or branch-major (all warm starts, then all cold starts)")
    ap.add_argument("--miz-members", type=int, default=131072, help="members per GPU of the MIZ sub-record")
    ap.add_argument("--miz-years", type=int, default=5, help="simulated years of the MIZ sub-record")
    ap.add_argument("--no-extra", action="store_true", help="skip the strong-scaling and MIZ sub-records")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (diagnostics, final state, flags) "
                         "for a fixed seeded sample of members as DIR/<workload>_<name>.npy, float64, under 64 MB in all "
                         "(rank 0's members only; members with non-finite outputs left out)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ----------------------------------------------------------------------------- workloads
ORDER = "interleaved"


def classic_workload(ebm, nmem_total, m, years):
    """C4: H = nmem_total/2 forcings F = -20..+20, each run from a warm and from a cold start, for the global member
    indices `m`.  Member order "interleaved" (SURVEY 8d, default): F_m = -20 + 40*(m//2)/(H-1), even m warm start, odd m
    cold start; "branch": F_m = -20 + 40*(m mod H)/(H-1), first half warm, second half cold."""
    st = ebm.SpaceTime(100, 2000, years)
    p = ebm.default_parameters("Classic")
    prow = np.array([p[k] for k in ebm.CLASSIC_PAR_ORDER])
    H = max(nmem_total // 2, 1)
    m = np.asarray(m, dtype=np.int64)
    count = len(m)
    if ORDER == "interleaved":
        F = -20.0 + 40.0 * (m // 2) / max(H - 1, 1)
        warm = (m % 2) == 0
    else:
        F = -20.0 + 40.0 * (m % H) / max(H - 1, 1)
        warm = m < H
    par = np.repeat(prow[None, :], count, axis=0)
    forc = np.zeros((count, 10))
    forc[:, 0] = forc[:, 1] = forc[:, 2] = F
    E0 = np.where(warm[:, None], 98.0, -9.5) * np.ones((count, st.nx))
    Tg0 = np.where(warm[:, None], 10.0, -10.0) * np.ones((count, st.nx))
    return st, par, forc, (E0, Tg0)


def classic_cost_key(nmem_total):
    """Regime of every member's initial state (0 warm / ice free, 2 cold / snowball): what the member costs."""
    m = np.arange(nmem_total)
    warm = (m % 2) == 0 if ORDER == "interleaved" else m < max(nmem_total // 2, 1)
    return np.where(warm, 0, 2)


def miz_workload(ebm, nmem_total, m, years):
    """C5: 16^5 tensor grid over (D, B, ai, k, m1) when nmem_total = 2^20 (row-major); zero init, F = 0."""
    st = ebm.SpaceTime(180, 2000, years, "sin")
    p = ebm.default_parameters("MIZ")
    order = list(ebm.MIZ_PAR_ORDER)
    prow = np.array([p[k] for k in order])
    m = np.asarray(m, dtype=np.int64)
    count = len(m)
    par = np.repeat(prow[None, :], count, axis=0)
    n = max(int(round(nmem_total ** 0.2)), 1)
    idx = [(m // n ** (4 - q)) % n for q in range(5)]
    lin = lambda lo, hi, i: lo + (hi - lo) * i / max(n - 1, 1)
    par[:, order.index("D")] = lin(0.45, 0.75, idx[0])
    par[:, order.index("B")] = lin(1.8, 2.4, idx[1])
    par[:, order.index("ai")] = lin(0.35, 0.45, idx[2])
    par[:, order.index("k")] = lin(1.5, 2.5, idx[3])
    par[:, order.index("m1")] = p["m1"] * lin(0.5, 2.0, idx[4])
    forc = np.zeros((count, 10))
    z = np.zeros((count, st.nx))
    return st, par, forc, (z, z, z, z, z)


# ----------------------------------------------------------------------------- clocks sampling
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nme in enumerate(names):
                if len(r) > 2 + k and r[2 + k].lower().startswith("active"):
                    reasons.add(nme)
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[6]) for r in self.rows if len(r) > 6 and r[6].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------- CPU arm
PUBLISHED_MIZ_MY_PER_S = 0.256   # the reference's only figure: 60 000 MIZ steps in 1:57 (src/EnergyBalanceModel.jl:57-61)


def host_threads():
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the oracle sets its own count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_run(workload, nmem_total, years, sample_members, threads, solver=0):
    """Oracle (port of the reference algorithm) with OpenMP over members on a strided sample of the workload
    (alternating even / odd members, so that both branches of C4 are sampled)."""
    import ebm_b200 as ebm
    import oracle
    sample_members = max(1, min(sample_members, nmem_total))
    stride = max(nmem_total // sample_members, 1)
    k = np.arange(sample_members)
    idx = np.minimum(k * stride + (k % 2), nmem_total - 1)
    if workload == "classic":
        st, par, forc, (E0, Tg0) = classic_workload(ebm, nmem_total, idx, years)
        t0 = time.perf_counter()
        oracle.classic_run(st.x, st.t, years, st.winter.inx, st.summer.inx, par, forc, E0, Tg0,
                           want_seasonal=True, nthreads=threads, solver=solver)
    else:
        st, par, forc, init = miz_workload(ebm, nmem_total, idx, years)
        t0 = time.perf_counter()
        oracle.miz_run(st.x, st.t, years, st.winter.inx, st.summer.inx, st.grid_kind, par, forc,
                       *init, want_seasonal=True, nthreads=threads)
    dt = time.perf_counter() - t0
    return len(idx) * years / dt, dt, f"{len(idx)} members (stride {stride}, even and odd alternating) x {years} years, seasonal sampling on"


def cpu_baseline(workload, nmem_total, years, threads, sample_members=0, target_s=20.0):
    """B-cpu of BASELINE.md 3: the oracle on all host cores, on a sample sized for >= ~10 s of CPU work (a short
    probe fixes the rate first), plus -- classic only -- B-ref-proxy (dense LU of the nx x nx matrix every step, as
    the reference's `\\` does, one thread) and B-pub (the reference's one published figure)."""
    probe_members = max(2 * threads, 8)
    yrs = years if workload == "classic" else min(years, 5)
    if not sample_members:
        v0, _, _ = cpu_run(workload, nmem_total, min(yrs, 2), probe_members, threads)
        sample_members = int(max(probe_members, min(nmem_total, v0 * target_s / yrs)))
        sample_members = max(threads, sample_members // threads * threads)
    v, dt, desc = cpu_run(workload, nmem_total, yrs, sample_members, threads)
    out = {"value": v, "unit": "member-years/s", "cores": threads, "kind": "port", "sample": desc, "seconds": dt,
           "note": "C oracle restating src/classic.jl / src/miz.jl (tridiagonal solve / semi-smooth Newton, OpenMP over "
                   "members); Julia is not installed, the reference itself cannot run",
           "published_reference": {"value": PUBLISHED_MIZ_MY_PER_S, "unit": "member-years/s", "what": "MIZ, nx=180, nt=2000, "
                                   "60 000 steps in 1:57 on the author's machine, 1 thread (src/EnergyBalanceModel.jl:57-61)"}}
    if workload == "classic":
        vp, dtp, descp = cpu_run("classic", nmem_total, 2, 4, 1, solver=1)
        out["reference_proxy"] = {"value": vp, "unit": "member-years/s", "cores": 1, "seconds": dtp, "sample": descp,
                                  "what": "same oracle with the dense LU of the nx x nx matrix every step, as "
                                          "classic.jl:55-63 does, one thread (BASELINE.md B-ref-proxy)"}
    return out


def reference_arm(args, nmem, years):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    world = args.gpus
    total = nmem * world
    sample = args.cpu_sample_members or (8 * threads if args.workload == "classic" else 2 * threads)
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt, desc = cpu_run(args.workload, total, years, sample, threads)
        if i >= args.warmup:
            vals.append((v, dt))
    value = sum(v * dt for v, dt in vals) / sum(dt for _, dt in vals)   # member-years / seconds over the K steps
    ms = 1e3 * sum(dt for _, dt in vals) / len(vals)
    line = {
        "impl": "reference", "metric": "member_years_per_sec", "value": value, "unit": "member-years/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, nmem, years, args.gpus),
        "cpu_baseline": {"value": value, "unit": "member-years/s", "cores": threads, "kind": "port", "sample": desc,
                         "note": "C oracle restating src/classic.jl / src/miz.jl (tridiagonal solve instead of the "
                                 "reference's dense LU); Julia is not installed, the reference itself cannot run"},
        "e2e": {"value": value, "unit": "member-years/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(workload, nmem, years, gpus):
    if workload == "classic":
        return {"workload": "C4 classic-EBM hysteresis ensemble: F=-20..+20 W/m^2, warm+cold start branches", "member_order": ORDER,
                "members_per_gpu": nmem, "members_total": nmem * gpus, "years": years, "nx": 100, "nt": 2000,
                "sharding": "32-member packets dealt round-robin over the ranks after a sort by initial regime (member_deal)",
                "outputs": "L0 diagnostics (3 seasons x 4 scalars per member-year) + final state",
                "l2": "flushed between timed iterations (256 MiB write); state is register-resident in any case"}
    return {"workload": "C5 MIZ parameter-sweep ensemble over (D,B,ai,k,m1), zero init, F=0",
            "members_per_gpu": nmem, "members_total": nmem * gpus, "years": years, "nx": 180, "nt": 2000,
            "grid": "sin", "outputs": "L0 diagnostics + final state",
            "l2": "flushed between timed iterations (256 MiB write)"}


# ----------------------------------------------------------------------------- GPU arm
class Env:
    """torch / library handles shared by the passes of one bench process."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        import ebm_b200 as ebm
        from ebm_b200 import _lib
        self.torch, self.dist, self.ebm, self._lib = torch, dist, ebm, _lib
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.lib = _lib.load()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
        self.stream = torch.cuda.current_stream()
        self.peak_tf, self.peak_mhz = ebm.fp64_peak(self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()


def device_pass(env, workload, nmem_total, years, steps, warmup, sample_clocks=False, dump_dir=None, dump_bytes=0):
    """W warm-up + K timed steps of one workload; every rank integrates the members `member_deal` hands it.
    Returns the measurements (max over ranks where it is a time) and what the e2e / CPU legs need.  With `dump_dir`,
    rank 0 writes a sample of the last timed step's outputs there (dump_outputs)."""
    torch, dist, ebm, _lib, lib, dev = env.torch, env.dist, env.ebm, env._lib, env.lib, env.dev
    world, rank = env.world, env.rank
    key = classic_cost_key(nmem_total) if workload == "classic" else None
    index = [ebm.member_deal(nmem_total, world, r, key=key) for r in range(world)]
    mine = index[rank]
    nmem = len(mine)
    build = classic_workload if workload == "classic" else miz_workload
    st, par, forc, init = build(ebm, nmem_total, mine, years)
    nx, nt = st.nx, st.nt
    grid = _lib.make_grid(st)
    opt = _lib.make_options(device=env.local, lastonly=True, field_stride=0)
    # device-resident inputs (member index fastest), allocated by torch.  member_deal hands over whole packets of
    # one regime in regime order, which is the layout the classic kernels want (lanes of a warp = members of a regime)
    f64 = torch.float64
    d_par = torch.from_numpy(np.ascontiguousarray(par.T)).to(dev)
    d_forc = torch.from_numpy(np.ascontiguousarray(forc.T)).to(dev)
    d_init = [torch.from_numpy(np.ascontiguousarray(a.T)).to(dev) for a in init]
    nstate = len(init) + (1 if workload == "miz" else 0)
    d_state = [torch.empty((nx, nmem), dtype=f64, device=dev) for _ in range(nstate)]
    d_diag = torch.full((nmem, years, 3, 4), float("nan"), dtype=f64, device=dev)
    d_flags = torch.zeros(nmem, dtype=torch.int32, device=dev)
    d_i64 = torch.zeros((2, nmem), dtype=torch.int64, device=dev)
    stream = env.stream
    if workload == "classic":
        dargs = _lib.ClassicDeviceArgs(nmem, d_par.data_ptr(), d_forc.data_ptr(), d_state[0].data_ptr(),
                                       d_state[1].data_ptr(), d_diag.data_ptr(), None, None, d_flags.data_ptr(), None)
        run_dev = lambda: _lib.check(lib.ebm_classic_run_device(C.byref(grid), C.byref(dargs), C.byref(opt),
                                                                C.c_void_p(stream.cuda_stream)))
    else:
        dargs = _lib.MizDeviceArgs(nmem, d_par.data_ptr(), d_forc.data_ptr(), *[t.data_ptr() for t in d_state],
                                   d_diag.data_ptr(), None, None, d_i64[0].data_ptr(), d_i64[1].data_ptr(),
                                   d_flags.data_ptr())
        run_dev = lambda: _lib.check(lib.ebm_miz_run_device(C.byref(grid), C.byref(dargs), C.byref(opt),
                                                            C.c_void_p(stream.cuda_stream)))
    kern_ev = []

    def step(timed):
        env.flush.fill_(1)                                 # L2 flush
        for k, a in enumerate(d_init):                     # restore the batch's initial state (device copy)
            d_state[k].copy_(a)
        if workload == "miz":
            d_state[-1].zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_dev()
        e1.record(stream)
        if world > 1:                                      # NCCL over NVLink: gather the ensemble diagnostics to rank 0
            ebm.gather_member_rows(d_diag, nmem_total, dst=0, index=index)
        if timed:
            kern_ev.append((e0, e1))

    for _ in range(warmup):
        step(False)
    env.barrier()
    sampler = ClockSampler(env.local) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    launches0 = lib.ebm_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(steps):
        step(True)
    t1.record(stream)
    env.barrier()
    launches = lib.ebm_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    if dump_dir is not None and rank == 0:
        if workload == "classic":
            outs = {"diag": d_diag, "E_final": d_state[0].T, "Tg_final": d_state[1].T, "flags": d_flags}
        else:
            outs = {"diag": d_diag, **{f"{v}_final": t.T for v, t in zip(("Ei", "Ew", "h", "D", "phi", "T0"), d_state)},
                    "newton_iters": d_i64[0], "nonconv": d_i64[1], "flags": d_flags}
        dump_outputs(dump_dir, workload, mine, outs, dump_bytes)
    ms_total = t0.elapsed_time(t1)
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in kern_ev]))
    k_all = [k_ms]
    if world > 1:
        tt = torch.tensor([ms_total], dtype=f64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt.item())
        kk = [torch.zeros(1, dtype=f64, device=dev) for _ in range(world)]
        dist.all_gather(kk, torch.tensor([k_ms], dtype=f64, device=dev))
        k_all = [float(t.item()) for t in kk]
    finite = torch.isfinite(d_state[0]).all(dim=0)         # members whose final state is finite
    cnt = torch.tensor([int(finite.sum().item()), int((d_flags != 0).sum().item())], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(cnt)
    ms_per_step = ms_total / steps
    value = nmem_total * years / (ms_per_step * 1e-3)
    flop_launch = FLOP_PER_CELL_STEP[workload] * nx * nt * float(years) * nmem
    achieved = flop_launch / (max(k_all) * 1e-3) / 1e12
    diag_bytes = d_diag.numel() * 8
    res = {"value": value, "ms_per_step": ms_per_step, "steps": steps, "warmup": warmup, "launches": int(launches),
           "clocks": clocks, "finite_members": int(cnt[0].item()), "flagged_members": int(cnt[1].item()),
           "members_total": nmem_total, "members_this_rank": nmem, "years": years,
           "kernel_ms_per_rank": {"min": min(k_all), "max": max(k_all), "all": k_all},
           "achieved_tflops": achieved, "diag_bytes": diag_bytes, "max_kernel_ms": max(k_all),
           "mean_T_last_year_member0": float(d_diag[0, -1, 2, 0].item()) if nmem else None}
    res["_e2e_inputs"] = (st, par, forc, init, nmem)
    return res


DUMP_BYTES = {"headline": 44_000_000, "miz": 16_000_000}   # under 64 MB in all, .npy headers included


def dump_outputs(out_dir, workload, mine, outs, max_bytes):
    """Write `outs` (name -> device tensor, member index first) for a sample of this rank's members as
    out_dir/<workload>_<name>.npy in float64, plus <workload>_member_index.npy (global member indices of the rows).
    The sample is drawn with a fixed seed from the member count alone and sized to `max_bytes`, so two builds of the
    project run with the same arguments sample the same members.  Sampled members with a non-finite value in any
    output are left out (members of the MIZ sweep whose state blows up, as it does in the reference algorithm; the
    JSON line counts them as nan_members), so every value written is finite and comparable."""
    import torch
    nmem = len(mine)
    per_member = 8 * (1 + sum(int(np.prod(t.shape[1:])) for t in outs.values()))
    count = max(1, min(nmem, max_bytes // per_member))
    pos = np.sort(np.random.default_rng(0).choice(nmem, size=count, replace=False))
    sel = {name: t.index_select(0, torch.from_numpy(pos).to(t.device)) for name, t in outs.items()}
    finite = torch.stack([torch.isfinite(s.reshape(count, -1)).all(dim=1) for s in sel.values()]).all(dim=0).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{workload}_member_index.npy"),
            np.asarray(mine, dtype=np.int64)[pos[finite]].astype(np.float64))
    for name, s in sel.items():
        np.save(os.path.join(out_dir, f"{workload}_{name}.npy"), s.cpu().numpy()[finite].astype(np.float64))


def roofline_record(env, workload, res, traffic):
    frac = res["achieved_tflops"] / env.peak_tf
    kernel = ("classic_uniform_kernel<13,8,16,168,...,UPAR> (launch-uniform parameters: member constants as constant-bank "
              "operands; ensembles with per-member parameters take the table-driven / per-member-coefficient instances)"
              if workload == "classic" else "miz_fast_kernel<6>")
    return {"bound": "fp64", "achieved": res["achieved_tflops"], "peak": env.peak_tf, "unit": "TFLOP/s", "frac": frac,
            "traffic": traffic.get(workload, {}).get("bytes") if traffic else None,
            "traffic_source": traffic.get(workload, {}).get("source") if traffic else None,
            "peak_source": "measured in this run by ebm_fp64_peak (dependent-free DFMA chains); MEASURED_PEAKS.json has no FP64 entry",
            "peak_nominal": NOMINAL_FP64_TFLOPS, "frac_of_nominal": res["achieved_tflops"] / NOMINAL_FP64_TFLOPS,
            "kernel": kernel, "kernel_ms": res["max_kernel_ms"],
            "algorithmic_flop_per_cell_step": FLOP_PER_CELL_STEP[workload],
            "hbm_output_stream": {"bytes_per_launch": res["diag_bytes"],
                                  "achieved_gbs": res["diag_bytes"] / (res["max_kernel_ms"] * 1e-3) / 1e9,
                                  "peak_gbs": _measured_hbm()}}


def _traffic():
    """DRAM bytes of one launch of the default configurations, captured with ncu (profiles/r2_traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return None


def main():
    args = parse()
    global ORDER
    ORDER = args.order
    nmem = args.members or (65536 if args.workload == "classic" else 131072)
    years = args.years or (200 if args.workload == "classic" else 50)
    if args.impl == "reference":
        reference_arm(args, nmem, years)
        return
    env = Env()
    world, rank = env.world, env.rank
    total = nmem * world
    traffic = _traffic()

    # ---- headline: K timed steps of the requested workload, weak scaling (nmem members per GPU)
    res = device_pass(env, args.workload, total, years, args.steps, args.warmup, sample_clocks=True,
                      dump_dir=args.dump_outputs, dump_bytes=DUMP_BYTES["headline"])
    roof = roofline_record(env, args.workload, res, traffic if (args.members == 0 and args.years == 0) else None)
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(env, args.workload, res["_e2e_inputs"], years, total)
    cpu = None
    if rank == 0 and not args.no_cpu:
        cpu = cpu_baseline(args.workload, total, years, host_threads(), args.cpu_sample_members)

    # ---- sub-records (default classic run only): strong scaling of the fixed 65 536-member sweep, and the MIZ sweep
    strong = miz = None
    if args.workload == "classic" and not args.no_extra:
        if world == 1:
            strong = {"members_total": total, "value": res["value"], "unit": "member-years/s",
                      "note": "N = 1: the strong-scaling run is the headline run"}
        else:
            sres = device_pass(env, "classic", nmem, years, min(args.steps, 3), 1)
            strong = {"members_total": nmem, "members_per_gpu": nmem // world, "years": years, "value": sres["value"],
                      "unit": "member-years/s", "ms_per_step": sres["ms_per_step"], "steps": sres["steps"], "warmup": 1,
                      "kernel_ms_per_rank": sres["kernel_ms_per_rank"],
                      "note": "the fixed 65 536-member sweep (SURVEY 8e) dealt over the N ranks; NCCL gather inside the timed step"}
        mz_members, mz_years = args.miz_members, args.miz_years
        mres = device_pass(env, "miz", mz_members * world, mz_years, min(args.steps, 3), 1,
                           dump_dir=args.dump_outputs, dump_bytes=DUMP_BYTES["miz"])
        mroof = roofline_record(env, "miz", mres, traffic)
        me2e = None if args.no_e2e else run_e2e(env, "miz", mres["_e2e_inputs"], mz_years, mz_members * world)
        mcpu = cpu_baseline("miz", mz_members * world, mz_years, host_threads()) if (rank == 0 and not args.no_cpu) else None
        fin = mres["finite_members"]
        miz = {"metric": "member_years_per_sec", "value": mres["value"], "unit": "member-years/s",
               "value_finite_members": mres["value"] * fin / max(mres["members_total"], 1),
               "nan_members": mres["members_total"] - fin, "flagged_members": mres["flagged_members"],
               "ms_per_step": mres["ms_per_step"], "steps": mres["steps"], "warmup": 1,
               "config": workload_config("miz", mz_members, mz_years, world), "roofline": mroof,
               "kernel_ms_per_rank": mres["kernel_ms_per_rank"], "e2e": me2e, "cpu_baseline": mcpu,
               "gpu_launches": mres["launches"],
               "note": "members whose state is non-finite at the end (the reference algorithm itself blows up for part of "
                       "this sweep, DESIGN.md 2) are counted in `value` and excluded from `value_finite_members`"}

    if rank == 0:
        line = {
            "metric": "member_years_per_sec", "value": res["value"], "unit": "member-years/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, nmem, years, world),
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": res["launches"], "clocks": res["clocks"],
            "kernel_ms_per_rank": res["kernel_ms_per_rank"],
            "nan_members": res["members_total"] - res["finite_members"], "flagged_members": res["flagged_members"],
            "strong": strong, "miz": miz,
        }
        print(json.dumps(line))
    if world > 1:
        env.dist.destroy_process_group()


def _measured_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh).get("hbm_gbs")
    except Exception:
        return 6650.0


def run_e2e(env, workload, inputs, years, total):
    """The same metric through the host-buffer C ABI: pinned host inputs -> H2D -> (regime sort) -> kernel -> D2H of the
    diagnostics and the final state, all inside the timed region; one untimed call first (the library keeps its device
    workspace between calls), then ONE timed call -- a step is seconds long, so one call is already a stable sample."""
    torch, dist, _lib, lib = env.torch, env.dist, env._lib, env.lib
    st, par, forc, init, nmem = inputs
    nx = st.nx
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_par, h_forc = pin(par), pin(forc)
    h_init = [pin(a) for a in init]
    h_diag = torch.empty((nmem, years, 3, 4), dtype=torch.float64).pin_memory()
    nfin = len(init) + (1 if workload == "miz" else 0)
    h_fin = [torch.empty((nmem, nx), dtype=torch.float64).pin_memory() for _ in range(nfin)]
    grid = _lib.make_grid(st)
    opt = _lib.make_options(device=env.local, lastonly=True, field_stride=0)
    P = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_double))
    if workload == "classic":
        out = _lib.ClassicOutputs(P(h_diag), None, None, P(h_fin[0]), P(h_fin[1]), None)
        call = lambda: _lib.check(lib.ebm_classic_run(C.byref(grid), nmem, P(h_par), P(h_forc), P(h_init[0]), P(h_init[1]),
                                                      C.byref(opt), C.byref(out)))
    else:
        out = _lib.MizOutputs(P(h_diag), None, None, *[P(t) for t in h_fin], None, None, None)
        call = lambda: _lib.check(lib.ebm_miz_run(C.byref(grid), nmem, P(h_par), P(h_forc), *[P(t) for t in h_init], None,
                                                  C.byref(opt), C.byref(out)))
    h2d = sum(t.numel() * 8 for t in [h_par, h_forc] + h_init)
    d2h = h_diag.numel() * 8 + sum(t.numel() * 8 for t in h_fin)
    call()
    env.barrier()
    t0 = time.perf_counter()
    call()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if env.world > 1:
        tt = torch.tensor([dt], dtype=torch.float64, device=env.dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    return {"value": total * years / dt, "unit": "member-years/s", "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(d2h), "seconds_per_step": dt, "steps": 1, "untimed_calls_before": 1,
            "api": "ebm_classic_run (host-buffer C ABI)" if workload == "classic" else "ebm_miz_run (host-buffer C ABI)",
            "result_check": {"mean_T_last_year_member0": float(h_diag[0, -1, 2, 0])}}


if __name__ == "__main__":
    main()
