"""dev: per-phase cycle breakdown of the classic kernel (CTA 0) at full residency (444 CTAs), by regime.
run: EBM_CUDA_LIB=energybalancemodel.jl_b200/lib/libebm_cuda_pt.so python scripts/dev_phase_timing2.py   (library: scripts/dev_phase_timing.sh)"""
import ctypes as C, sys, time
sys.path.insert(0, ".")
import numpy as np
import ebm_b200 as ebm
from ebm_b200 import _lib

lib = _lib.load()
lib.ebm_debug_phase_cycles.argtypes = [C.POINTER(C.c_uint64)]
nmem, years = 7104, 2
st = ebm.SpaceTime(100, 2000, years)
p = ebm.default_parameters("Classic")
par = np.repeat(np.array([[p[k] for k in ebm.CLASSIC_PAR_ORDER]]), nmem, axis=0)
names = ["physics", "elim+reduce", "barrier1 wait", "interface", "barrier2 wait", "backsub"]
for label, F, warm, spin in (("ice-free (F=+15, warm)", 15.0, True, 0), ("seasonal ice (F=0, warm)", 0.0, True, 20), ("snowball (F=-10, cold)", -10.0, False, 0)):
    forc = np.zeros((nmem, 10)); forc[:, :3] = F
    E0 = np.full((nmem, 100), 98.0 if warm else -9.5); Tg0 = np.full((nmem, 100), 10.0 if warm else -10.0)
    for yrs in ([spin, years] if spin else [years]):
        stt = ebm.SpaceTime(100, 2000, yrs)
        diag = np.empty((nmem, yrs, 3, 4)); Ef = np.empty((nmem, 100)); Tgf = np.empty((nmem, 100))
        out = _lib.ClassicOutputs(_lib.dptr(diag), None, None, _lib.dptr(Ef), _lib.dptr(Tgf), None)
        grid = _lib.make_grid(stt); opt = _lib.make_options()
        buf = (C.c_uint64 * 64)()
        lib.ebm_debug_phase_cycles(buf)   # reset
        t0 = time.time()
        _lib.check(lib.ebm_classic_run(C.byref(grid), nmem, _lib.dptr(par), _lib.dptr(forc), _lib.dptr(E0), _lib.dptr(Tg0), C.byref(opt), C.byref(out)))
        dt = time.time() - t0
        E0, Tg0 = Ef.copy(), Tgf.copy()
    rc = lib.ebm_debug_phase_cycles(buf)
    a = np.array(list(buf), dtype=np.float64).reshape(8, 8)[:6, :4] / (2000 * years)
    print(f"== {label}: wall {dt:.3f}s rc={rc}; ice area last year {diag[0,-1,2,2]:.2f}; cycles per step by phase x warp (CTA 0):")
    for k, n in enumerate(names):
        print(f"   {n:14s} " + " ".join(f"{v:8.0f}" for v in a[k]))
    print(f"   {'total':14s} " + " ".join(f"{v:8.0f}" for v in a.sum(axis=0)))
