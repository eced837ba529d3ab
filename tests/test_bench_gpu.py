"""bench.py --dump-outputs on a small C4 ensemble and MIZ sweep: the files hold what the timed device path returned in
its last step, for the members they name (classic: against the oracle at the stated tolerance), and only finite values
(MIZ members whose state blows up are left out)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import ebm_b200 as ebm
import oracle
from helpers import assert_close, oracle_diag_classic

pytestmark = pytest.mark.gpu
TOL = 1e-9


def test_bench_dump_outputs(tmp_path):
    out = tmp_path / "dump"
    nmem, years, mz_nmem = 512, 2, 1024   # 1024 = 4^5: the MIZ sweep's grid has interior points
    r = subprocess.run([sys.executable, bench.__file__, "--members", str(nmem), "--years", str(years), "--steps", "3",
                        "--warmup", "1", "--no-e2e", "--no-cpu", "--miz-members", str(mz_nmem), "--miz-years", "1",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["miz"]["steps"] == 3
    names = sorted(os.listdir(out))
    assert sum(os.path.getsize(out / f) for f in names) < 64e6
    d = {f[:-len(".npy")]: np.load(out / f) for f in names}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in d.values())

    # small ensembles are written whole; member_index maps rows to the sweep's global member indices
    m = d["classic_member_index"].astype(np.int64)
    assert np.array_equal(np.sort(m), np.arange(nmem))
    assert d["classic_diag"].shape == (nmem, years, 3, 4) and d["classic_E_final"].shape == (nmem, 100)
    assert d["classic_flags"].max() == 0
    st, par, forc, (E0, Tg0) = bench.classic_workload(ebm, nmem, m, years)
    o = oracle.classic_run(st.x, st.t, years, st.winter.inx, st.summer.inx, par, forc, E0, Tg0, want_seasonal=True)
    fE = (np.abs(o["E"]) < 1e-6) | ((d["classic_E_final"] < 0) != (o["E"] < 0))
    assert_close(d["classic_E_final"], o["E"], TOL, "dumped final E", flag=fE)
    assert_close(d["classic_Tg_final"], o["Tg"], TOL, "dumped final Tg")
    od = oracle_diag_classic(o["seasonal"], st.x)
    assert_close(d["classic_diag"][..., :2], od[..., :2], TOL, "dumped mean T / mean E")

    # the whole MIZ sweep is sampled; members with non-finite outputs are left out, so at most the finite ones remain
    mm = d["miz_member_index"].astype(np.int64)
    nkeep = len(mm)
    assert 0 < nkeep <= mz_nmem - line["miz"]["nan_members"]
    assert len(np.unique(mm)) == nkeep and mm.min() >= 0 and mm.max() < mz_nmem
    assert d["miz_diag"].shape == (nkeep, 1, 3, 4)
    for v in ("Ei", "Ew", "h", "D", "phi", "T0"):
        assert d[f"miz_{v}_final"].shape == (nkeep, 180), v
    assert d["miz_newton_iters"].max() > 0
