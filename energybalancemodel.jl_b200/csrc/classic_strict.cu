// classic_strict.cu -- literal-arithmetic classic step on the GPU (one thread per member).
//
// Same operation order as the reference (src/classic.jl:43-65, SURVEY.md Appendix A): IEEE division,
// no FMA contraction (every op is an explicit __d*_rn intrinsic), masks as selects, and the
// tridiagonal solve in the LU order a dense `\` without row swaps reduces to.  State and scratch
// live in global memory; this kernel exists for parity debugging (ebm_options_t.strict) and for the
// one-step entry point ebm_classic_step -- it is not the fast path (classic_uniform.cu is).
#include "ebm_internal.cuh"

namespace {

struct Lit {  // literal IEEE ops, never contracted
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
};

struct ClassicStatics {
  double dt, cg_tau, dt_tau, dc, M, kLf, dtD, one_dttau;
};

__device__ __forceinline__ ClassicStatics make_statics(const double* p, long long stride, int nt) {
  ClassicStatics s;
  const double D = p[0 * stride], B = p[2 * stride], k = p[11 * stride], Lf = p[12 * stride];
  const double cg = p[13 * stride], tau = p[14 * stride];
  s.dt = Lit::div(1.0, (double)nt);        // infrastructure.jl:128
  s.cg_tau = Lit::div(cg, tau);            // classic.jl:18
  s.dt_tau = Lit::div(s.dt, tau);          // :19
  s.dc = Lit::mul(s.dt_tau, s.cg_tau);     // :20
  s.M = Lit::add(B, s.cg_tau);             // :27
  s.kLf = Lit::mul(k, Lf);                 // :29
  s.dtD = Lit::mul(s.dt, D);               // :21 (dt*D)
  s.one_dttau = Lit::add(1.0, s.dt_tau);
  return s;
}

// One literal step for member m.  E, Tg, and scratch arrays are strided by `stride` (member-fastest
// layout [nx][nmem]); T is written to Tout (same stride).  ti = 1-based year index.
__device__ void classic_step_literal(const EbmGridTables& g, const double* p, long long pstride,
                                     const ClassicStatics& s, int ti, double f,
                                     double* E, double* Tg, double* Tout, double* dg, double* y, double* w,
                                     long long stride, int dbg_which = 0, double* dbg = nullptr) {
  const int nx = g.nx;
  const double A = p[1 * pstride], cw = p[3 * pstride], S0 = p[4 * pstride], S1 = p[5 * pstride];
  const double S2 = p[6 * pstride], a0 = p[7 * pstride], a2 = p[8 * pstride], ai = p[9 * pstride];
  const double Fb = p[10 * pstride], cg = p[13 * pstride];
  const double sc0 = Lit::mul(S1, g.ctab[ti - 1]);  // S1*cos(2*pi*t_i)
  const double sc1 = Lit::mul(S1, g.ctab[ti]);      // column i+1 (nt+1 := 1)
  for (int j = 0; j < nx; ++j) {
    const double xj = g.x[j], x2j = g.x2[j];
    const double Sb = Lit::sub(S0, Lit::mul(S2, x2j));
    const double Si = Lit::sub(Sb, Lit::mul(sc0, xj));
    const double Sn = Lit::sub(Sb, Lit::mul(sc1, xj));
    const double aw = Lit::sub(a0, Lit::mul(a2, x2j));                                   // :28
    double Ej = E[j * stride];
    const double Tgj = Tg[j * stride];
    const double alpha = Ej > 0.0 ? aw : (Ej < 0.0 ? ai : 0.0);                          // :47
    const double C = Lit::add(Lit::sub(Lit::add(Lit::mul(alpha, Si), Lit::mul(s.cg_tau, Tgj)), A), f);  // :48
    const double T0 = Lit::div(C, Lit::sub(s.M, Lit::div(s.kLf, Ej)));                   // :50
    const double Tj = Lit::add(Ej >= 0.0 ? Lit::div(Ej, cw) : 0.0, (Ej < 0.0 && T0 < 0.0) ? T0 : 0.0);  // :51
    Tout[j * stride] = Tj;
    Ej = Lit::add(Ej, Lit::mul(s.dt, Lit::add(Lit::sub(C, Lit::mul(s.M, Tj)), Fb)));     // :53
    E[j * stride] = Ej;
    const bool mk = (T0 < 0.0) && (Ej < 0.0);
    if (dbg != nullptr)   // debug menu of the step seam (include/ebm_cuda.h EBM_DEBUG_*; classic.jl:67-69)
      dbg[j * stride] = dbg_which == EBM_DEBUG_ALPHA ? alpha : dbg_which == EBM_DEBUG_C ? C : dbg_which == EBM_DEBUG_T0 ? T0
                      : dbg_which == EBM_DEBUG_S ? Si : dbg_which == EBM_DEBUG_MASK ? (mk ? 1.0 : 0.0) : nan("");
    const double gg = Lit::sub(s.M, Lit::div(s.kLf, Ej));
    // kappa diagonal: (1+dt_tau) - ((dt*D)*diffop_jj)/cg, diffop_jj = -l3, l3 = -l1 - l2 (infrastructure.jl:485-488)
    const double l1 = j > 0 ? -g.lam_lo[j] : 0.0, l2 = j < nx - 1 ? -g.lam_hi[j] : 0.0;
    const double l3 = Lit::sub(-l1, l2);
    const double kd = Lit::sub(s.one_dttau, Lit::div(Lit::mul(s.dtD, -l3), cg));
    dg[j * stride] = Lit::sub(kd, mk ? Lit::div(s.dc, gg) : 0.0);                        // :56
    const double r1 = Ej >= 0.0 ? Lit::div(Ej, cw) : 0.0;
    const double r2 = mk ? Lit::div(Lit::add(Lit::sub(Lit::mul(ai, Sn), A), f), gg) : 0.0;
    y[j * stride] = Lit::add(Tgj, Lit::mul(s.dt_tau, Lit::add(r1, r2)));                 // :58-62 (rhs)
  }
  // tridiagonal solve, LU order: l = a/w; w' = d - l*c; y' = r - l*y; x = (y - c*x')/w
  w[0] = dg[0];
  for (int j = 1; j < nx; ++j) {
    const double off = -Lit::div(Lit::mul(s.dtD, g.lam_lo[j]), cg);      // kappa sub-diagonal: row j, column j-1
    const double sup = -Lit::div(Lit::mul(s.dtD, g.lam_hi[j - 1]), cg);  // super-diagonal of row j-1 (the same value with get_diffop)
    const double l = Lit::div(off, w[(j - 1) * stride]);
    w[j * stride] = Lit::sub(dg[j * stride], Lit::mul(l, sup));
    y[j * stride] = Lit::sub(y[j * stride], Lit::mul(l, y[(j - 1) * stride]));
  }
  double xn = Lit::div(y[(nx - 1) * stride], w[(nx - 1) * stride]);
  Tg[(nx - 1) * stride] = xn;
  for (int j = nx - 2; j >= 0; --j) {
    const double off = -Lit::div(Lit::mul(s.dtD, g.lam_hi[j]), cg);
    xn = Lit::div(Lit::sub(y[j * stride], Lit::mul(off, xn)), w[j * stride]);
    Tg[j * stride] = xn;
  }
}

// hemispheric_mean in the reference's loop order (utilities.jl:397-403)
template <typename F>
__device__ double hemi_mean(const double* x, int nx, F val) {
  double acc = 0.0;
  for (int i = 0; i < nx - 1; ++i)
    acc = Lit::add(acc, Lit::div(Lit::mul(Lit::add(val(i), val(i + 1)), Lit::sub(x[i + 1], x[i])), 2.0));
  return acc;
}

__global__ void classic_strict_kernel(const ClassicKArgs a, double* ws) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= a.nmem) return;
  const long long nmem = a.nmem;
  const int nx = a.nx, nt = a.nt;
  const size_t plane = (size_t)nx * nmem;
  double* dg = ws + 0 * plane + m; double* y = ws + 1 * plane + m; double* w = ws + 2 * plane + m;
  double* Tc = ws + 3 * plane + m; double* sE = ws + 4 * plane + m; double* sT = ws + 5 * plane + m;
  double* sH = ws + 6 * plane + m;
  double* E = a.E + m; double* Tg = a.Tg + m;
  const double* p = a.par + m;
  const ClassicStatics s = make_statics(p, nmem, nt);
  const double Lf = p[12 * nmem];
  const double* fr = a.forc + m;
  const long long mo = a.orig != nullptr ? a.orig[m] : m;   // original member index: output rows
  const bool sel = ebm_field_selected(a, mo);
  const long long msel = sel ? ebm_field_row(a, mo) : 0;
  const long long nraw = ebm_nraw(nt, a.dur, a.lastonly);
  for (int j = 0; j < nx; ++j) { sE[j * nmem] = 0.0; sT[j * nmem] = 0.0; sH[j * nmem] = 0.0; }

  for (int year = a.year0; year < a.year0 + a.nyears; ++year) {
    for (int ti = 1; ti <= nt; ++ti) {
      const double f = ebm_forcing_at([&](int r) { return fr[r * nmem]; }, (long long)(year + a.start_year) * nt + ti, nt);
      classic_step_literal(a.g, p, nmem, s, ti, f, E, Tg, Tc, dg, y, w, nmem);
      for (int j = 0; j < nx; ++j) {
        const double Ej = E[j * nmem];
        sE[j * nmem] += Ej; sT[j * nmem] += Tc[j * nmem];
        sH[j * nmem] += (Ej < 0.0 ? Lit::div(-Ej, Lf) : 0.0);
      }
      const int season = ebm_season(a, ti, nt);
      if (sel && a.raw != nullptr && ebm_raw_year(year, a.dur, a.lastonly)) {
        double* o = a.raw + ebm_raw_offset(msel, nraw, ebm_raw_slot(year, ti, nt, a.lastonly), EBM_CLASSIC_NVAR, nx);
        for (int j = 0; j < nx; ++j) {
          const double Ej = E[j * nmem];
          o[j] = Ej; o[nx + j] = Tc[j * nmem]; o[2 * nx + j] = Ej < 0.0 ? Lit::div(-Ej, Lf) : 0.0;  // :65
        }
      }
      if (season >= 0) {
        const bool avg = season == 2;
        const double dnt = (double)nt;
        auto vE = [&](int j) { return avg ? Lit::div(sE[j * nmem], dnt) : E[j * nmem]; };
        auto vT = [&](int j) { return avg ? Lit::div(sT[j * nmem], dnt) : Tc[j * nmem]; };
        auto vH = [&](int j) {
          if (avg) return Lit::div(sH[j * nmem], dnt);
          const double Ej = E[j * nmem];
          return Ej < 0.0 ? Lit::div(-Ej, Lf) : 0.0;
        };
        if (sel && a.seasonal != nullptr) {
          double* o = a.seasonal + ebm_seasonal_offset(msel, a.dur, year, season, EBM_CLASSIC_NVAR, nx);
          for (int j = 0; j < nx; ++j) { o[j] = vE(j); o[nx + j] = vT(j); o[2 * nx + j] = vH(j); }
        }
        if (a.diag != nullptr) {
          double edge = 2.0;   // no ice
          for (int j = 0; j < nx; ++j) if (vE(j) < 0.0) { edge = a.g.x[j]; break; }
          ebm_store_diag(a.diag, mo, a.dur, year, season, hemi_mean(a.g.x, nx, vT), hemi_mean(a.g.x, nx, vE),
                         hemi_mean(a.g.x, nx, [&](int j) { return vE(j) < 0.0 ? 1.0 : 0.0; }), edge);
        }
      }
      if (ti == nt) for (int j = 0; j < nx; ++j) { sE[j * nmem] = 0.0; sT[j * nmem] = 0.0; sH[j * nmem] = 0.0; }
    }
  }
  if (a.flags != nullptr) {
    bool bad = false;
    for (int j = 0; j < nx; ++j) bad = bad || ebm_state_bad(E[j * nmem]) || ebm_state_bad(Tg[j * nmem]);
    if (bad) atomicOr(a.flags + mo, 1);
  }
}

// one step, one member: contiguous [nx] arrays (stride 1); scratch = 3*nx doubles
__global__ void classic_single_step_kernel(EbmGridTables g, const double* par15, int ti, double f,
                                           double* E, double* Tg, double* T, double* h, double* scratch,
                                           int dbg_which, double* dbg) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  const ClassicStatics s = make_statics(par15, 1, g.nt);
  classic_step_literal(g, par15, 1, s, ti, f, E, Tg, T, scratch, scratch + g.nx, scratch + 2 * g.nx, 1, dbg_which, dbg);
  const double Lf = par15[12];
  for (int j = 0; j < g.nx; ++j) h[j] = E[j] < 0.0 ? Lit::div(-E[j], Lf) : 0.0;  // classic.jl:65
}

}  // namespace

int ebm_launch_classic_strict(const ClassicKArgs& a, cudaStream_t stream) {
  double* ws = nullptr;
  const size_t bytes = sizeof(double) * 7 * (size_t)a.nx * (size_t)a.nmem;
  EBM_CUDA_TRY(cudaMallocAsync(&ws, bytes, stream));
  const int threads = 64;
  const long long blocks = (a.nmem + threads - 1) / threads;
  classic_strict_kernel<<<(unsigned)blocks, threads, 0, stream>>>(a, ws);
  cudaError_t e = cudaGetLastError();
  cudaFreeAsync(ws, stream);
  EBM_CUDA_TRY(e);
  ebm_count_launch();
  return EBM_OK;
}

int ebm_launch_classic_single_step(const EbmGridTables& g, const double* par15, int ti, double f,
                                   double* E, double* Tg, double* T, double* h, cudaStream_t stream,
                                   int dbg_which, double* dbg) {
  double* scratch = nullptr;
  EBM_CUDA_TRY(cudaMallocAsync(&scratch, sizeof(double) * 3 * (size_t)g.nx, stream));
  classic_single_step_kernel<<<1, 32, 0, stream>>>(g, par15, ti, f, E, Tg, T, h, scratch, dbg_which, dbg);
  cudaError_t e = cudaGetLastError();
  cudaFreeAsync(scratch, stream);
  EBM_CUDA_TRY(e);
  ebm_count_launch();
  return EBM_OK;
}
