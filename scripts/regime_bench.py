#!/usr/bin/env python
"""dev: throughput of the classic kernel on regime-homogeneous ensembles (what each code path costs).

    python scripts/regime_bench.py [--members 32768] [--years 10] [--regimes snow,free,partial,c4]

snow: cold start (every cell ice, stays a snowball), F = -20..+20; free: warm start, F = +14..+20 (ice free after the
spin-up); partial: warm start, F = -8..+8 (seasonal / perennial polar ice); c4: the bench.py C4 mix.  The state is
spun up for `--spinup` years first so that the timed launches see the regime's steady state.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--members", type=int, default=32768)
    ap.add_argument("--years", type=int, default=10)
    ap.add_argument("--spinup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--regimes", default="snow,free,partial,c4")
    a = ap.parse_args()
    import torch
    import ebm_b200 as ebm
    from ebm_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    p = ebm.default_parameters("Classic")
    prow = np.array([p[k] for k in ebm.CLASSIC_PAR_ORDER])
    n = a.members
    out = {"members": n, "years": a.years}
    for regime in a.regimes.split(","):
        m = np.arange(n)
        if regime == "snow":
            F, warm = -20.0 + 40.0 * m / (n - 1), np.zeros(n, bool)
        elif regime == "free":
            F, warm = 14.0 + 6.0 * m / (n - 1), np.ones(n, bool)
        elif regime == "partial":
            F, warm = -8.0 + 16.0 * m / (n - 1), np.ones(n, bool)
        else:
            F, warm = -20.0 + 40.0 * (m // 2) / (n // 2 - 1), (m % 2) == 0
        # sorted by regime of the initial state, like ebm_classic_run does
        order = np.argsort(~warm, kind="stable")
        F, warm = F[order], warm[order]
        forc = np.zeros((10, n)); forc[0] = forc[1] = forc[2] = F
        par = np.repeat(prow[:, None], n, axis=1)
        E0 = np.where(warm[None, :], 98.0, -9.5) * np.ones((100, n))
        Tg0 = np.where(warm[None, :], 10.0, -10.0) * np.ones((100, n))
        d_par, d_forc = torch.from_numpy(par).to(dev), torch.from_numpy(forc).to(dev)
        d_E, d_Tg = torch.from_numpy(E0).to(dev), torch.from_numpy(Tg0).to(dev)
        stream = torch.cuda.current_stream()

        def run(years, start):
            st = ebm.SpaceTime(100, 2000, years)
            grid = _lib.make_grid(st)
            opt = _lib.make_options(device=0, lastonly=True, field_stride=0, start_year=start)
            d_diag = torch.empty((n, years, 3, 4), dtype=torch.float64, device=dev)
            dargs = _lib.ClassicDeviceArgs(n, d_par.data_ptr(), d_forc.data_ptr(), d_E.data_ptr(), d_Tg.data_ptr(),
                                           d_diag.data_ptr(), None, None, None, None)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            _lib.check(lib.ebm_classic_run_device(C.byref(grid), C.byref(dargs), C.byref(opt), C.c_void_p(stream.cuda_stream)))
            e1.record(stream)
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), d_diag

        if a.spinup > 0:
            run(a.spinup, 0)
        best = 1e30
        for r in range(a.reps):
            ms, dg = run(a.years, a.spinup + r * a.years)
            best = min(best, ms)
        E = d_E.cpu().numpy()
        ice = (E < 0).sum(axis=0)
        out[regime] = {"my_per_s": n * a.years / (best * 1e-3), "ms": best,
                       "end_state": {"ice_free": float((ice == 0).mean()), "snowball": float((ice == 100).mean()),
                                     "partial": float(((ice > 0) & (ice < 100)).mean())},
                       "checksum_meanT_last": float(dg[:, -1, 2, 0].double().mean().item())}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
