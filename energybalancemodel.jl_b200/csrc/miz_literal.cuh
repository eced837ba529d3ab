// miz_literal.cuh -- the marginal-ice-zone (MIZ) ensemble step kernel written in the reference's operation order.
// Included by miz_strict.cu and compiled with -fmad=false: literal arithmetic, IEEE division, serial Thomas solve in
// the oracle's order -- bit-identical to the oracle; used for parity debugging (ebm_options_t.strict) and by the
// one-step entry point ebm_miz_step.  The production fast kernel, same mapping with the arithmetic restructured for
// the FP64 pipe, is miz_kernel.cu.
//
// Replaces, for a whole ensemble and many years per launch, the reference's
//   integrate loop            src/infrastructure.jl:630-634
//   step!(::Val{:MIZ})        src/miz.jl:150-196        (arithmetic spec: SURVEY.md Appendix B)
//   solveTi / T0eq            src/miz.jl:33-68          (closure: semi-smooth Newton, tridiagonal Jacobian)
//   diffusion!                src/infrastructure.jl:495-527 (identity grid and generic flux-form stencil)
//   savesol! / annual_mean    src/infrastructure.jl:536-591
//
// Mapping (B200: 148 SMs x 4 sub-partitions, 16 FP64 lanes each, 64K registers per SM):
//   * one WARP integrates one member; lane l owns the K contiguous cells j = l*K .. l*K+K-1 (K = ceil(nx/32)).
//     The six state vectors (Ei, Ew, h, D, phi and the closure's warm start T0) stay in registers for the
//     whole launch -- years of steps -- and nothing but sampled output touches HBM.
//   * there is no CTA barrier in the time loop and no shared-memory traffic between lanes: neighbour
//     temperatures cross lanes with two shuffles per stencil evaluation, and the Newton convergence test is a
//     warp vote, so every member takes exactly the iterations it needs (no lock-step across members).
//   * the closure's linear system (tridiagonal, strictly diagonally dominant) is solved by one lane, serial Thomas
//     in the oracle's order, through shared memory.
//   * geometry tables (x, x^2, trapezoid weights, stencil coefficients) are per-CTA shared memory laid out
//     [cell-in-lane][lane] (bank-conflict free); member parameters are warp-uniform registers.
//   * the insolation cos(2*pi*t) comes from a per-step table built on the host (same libm as the oracle).
#pragma once
#include <math.h>

#include "ebm_internal.cuh"


namespace {

constexpr int kWarpsPerCta = 1;

// Julia min(a, b): NaN-propagating (SURVEY Appendix C.6)
__device__ __forceinline__ double jl_min(double a, double b) {
  if (a != a || b != b) return a + b;
  if (a == b) return (__double2hiint(a) < 0) ? a : b;   // min(0.0, -0.0) = -0.0
  return a < b ? a : b;
}
// Julia clamp(x, lo, hi) = ifelse(x > hi, hi, ifelse(x < lo, lo, x)); NaN passes through
__device__ __forceinline__ double jl_clamp(double x, double lo, double hi) { return x > hi ? hi : (x < lo ? lo : x); }

struct MizPar {   // miz_paramset, src/infrastructure.jl:436-441
  double D, A, B, cw, S0, S1, S2, a0, a2, ai, Fb, k, Lf, Tm, m1, m2, alpha, rl, Dmin, Dmax, hmin, kappa;
};

// per-CTA geometry tables, [i][lane] for cell j = lane*K + i
template <int K>
struct MizTabs {
  double x[K * 32], x2[K * 32], wts[K * 32];
  double cu[K * 32], cl[K * 32];   // stencil coefficient towards j+1 / j-1
  // literal stencils: generic (mxxph, mxxmh, phmmh, diffx[j+1], diffx[j]) / identity (lam_hi, lam_lo)
  double mxxph[K * 32], mxxmh[K * 32], phmmh[K * 32], dxp[K * 32], dxm[K * 32];
  double scratch[6][K * 32];   // serial Thomas: jl, jd, ju, rhs, w, y
};

template <int K>
struct MizMember {
  // state
  double Ei[K], Ew[K], h[K], D[K], phi[K], T0[K];
  // per-year accumulators for the L0 diagnostics of the annual-mean fields (hemispheric mean is linear)
  double accT, accE, accP;
  unsigned icebits;
};

// ---- diffusion of a temperature profile held K cells per lane (increment only: D * nabla^2 T) -----------------
// tb[i] are the lane's cells; neighbours come from the adjacent lanes.  Zero flux at both ends: the difference
// (generic stencil, infrastructure.jl:522) / the get_diffop coefficient towards a missing neighbour is 0.
template <int K>
__device__ __forceinline__ void miz_diffusion(const MizTabs<K>& tb_, const MizPar& p, int kind, int nx, int lane,
                                              const double (&tb)[K], double (&out)[K]) {
  const double left = ebm_shfl_up1(tb[K - 1]);    // cell j-1 of my first cell (garbage for lane 0: masked)
  const double right = ebm_shfl_dn1(tb[0]);       // cell j+1 of my last cell
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int s = i * 32 + lane;
    const double tm = (i == 0) ? left : tb[i - 1];
    const double tp = (i == K - 1) ? right : tb[i + 1];
    const int j = lane * K + i;
    if (kind == 1) {
      const double dTp = (j < nx - 1) ? tp - tb[i] : 0.0;       // diffT[i]   (:522-523)
      const double dTm = (j > 0) ? tb[i] - tm : 0.0;            // diffT[i-1]
      out[i] = p.D * (tb_.mxxph[s] * dTp / tb_.dxp[s] - tb_.mxxmh[s] * dTm / tb_.dxm[s]) / tb_.phmmh[s];   // :524
    } else {
      // (par.D * get_diffop(nx)) * temp, CSC mat-vec accumulated in column order (:497)
      const double lm = tb_.cl[s], lp = tb_.cu[s];              // lambda towards j-1 / j+1 (0 at the ends)
      const double l1 = (j > 0) ? -lm : 0.0, l2 = (j < nx - 1) ? -lp : 0.0;
      const double l3 = -l1 - l2;
      double acc = 0.0;
      if (j > 0) acc += (p.D * lm) * tm;
      acc += (p.D * (-l3)) * tb[i];
      if (j < nx - 1) acc += (p.D * lp) * tp;
      out[i] = acc;
    }
  }
}

// ---- tridiagonal solve: rows (jl, jd, ju) x = rhs, K rows per lane ------------------------------------------------
// On return rhs holds the solution.  Literal Thomas in the oracle's order (one lane), through shared memory.
template <int K>
__device__ __forceinline__ void miz_tridiag(MizTabs<K>& tabs, int nx, int lane, const double (&jl)[K],
                                            const double (&jd)[K], const double (&ju)[K], double (&rhs)[K]) {
  double* sl = tabs.scratch[0]; double* sd = tabs.scratch[1]; double* su = tabs.scratch[2];
  double* sr = tabs.scratch[3]; double* w = tabs.scratch[4]; double* y = tabs.scratch[5];
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = lane * K + i;
    sl[j] = jl[i]; sd[j] = jd[i]; su[j] = ju[i]; sr[j] = rhs[i];
  }
  __syncwarp();
  if (lane == 0) {
    w[0] = sd[0]; y[0] = sr[0];
    for (int j = 1; j < nx; ++j) {
      const double l = sl[j] / w[j - 1];
      w[j] = sd[j] - l * su[j - 1];
      y[j] = sr[j] - l * y[j - 1];
    }
    double dl = y[nx - 1] / w[nx - 1];
    sr[nx - 1] = dl;
    for (int j = nx - 2; j >= 0; --j) { dl = (y[j] - su[j] * dl) / w[j]; sr[j] = dl; }
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = lane * K + i;
    rhs[i] = (j < nx) ? sr[j] : 0.0;
  }
  __syncwarp();
}

// ---- closure: solveTi (src/miz.jl:47-68) ----------------------------------------------------------------------------
// Residual T0eq (:33-45) is piecewise linear in T0 with a tridiagonal generalised Jacobian
//   J = -diag(k/hp + B) + L*diag(phi*[T0 < Tm]),   L = D*nabla^2 stencil,
// so a semi-smooth Newton iteration stopped at max|res| <= tol (reference: abstol 1e-8) finds the root the
// reference's TrustRegion solver is asked for.  Returns the number of Newton iterations; *fail if not converged.
template <int K>
__device__ __forceinline__ int miz_solveTi(MizTabs<K>& tabs, const MizPar& p, int kind, int nx, int lane,
                                           double f, double c2pt, const double (&h)[K], const double (&Tw)[K],
                                           const double (&phi)[K], double (&T0)[K], double (&Ti)[K], double tol,
                                           int maxit, int* fail) {
  double hp[K], ins[K];
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int s = i * 32 + lane;
    hp[i] = (h[i] == 0.0) ? p.hmin : h[i];                                          // :51
    const double xj = tabs.x[s];
    ins[i] = p.ai * (p.S0 - p.S1 * xj * c2pt - p.S2 * tabs.x2[s]);                  // solar on ice, :11
  }
  int it = 0;
  *fail = 0;
  for (;;) {
    double tb[K], dif[K], res[K];
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const double ti = jl_min(T0[i], p.Tm);                                        // ice_temp :31
      tb[i] = ti * phi[i] + (1 - phi[i]) * Tw[i];                                   // Tbar! :21-25
    }
    miz_diffusion<K>(tabs, p, kind, nx, lane, tb, dif);
    bool ok = true, nan = false;
#pragma unroll
    for (int i = 0; i < K; ++i) {
      double v = p.k * (p.Tm - T0[i]) / hp[i];                                      // :39 SCM
      v = v + ins[i];                                                               // :40
      v = v + ((-p.A) - p.B * (T0[i] - p.Tm));                                      // :41 OLR
      v = v + dif[i];                                                               // :42
      v = v + f;                                                                    // :43
      res[i] = v;
      if (lane * K + i < nx) {
        const double av = fabs(v);
        nan = nan || (av != av);
        ok = ok && (av <= tol);
      }
    }
    const bool anynan = __any_sync(kFull, nan);
    const bool allok = __all_sync(kFull, ok);
    if (!anynan && allok) break;
    if (anynan || it >= maxit) { *fail = 1; break; }
    // Jacobian rows
    double g[K], jl[K], jd[K], ju[K];
#pragma unroll
    for (int i = 0; i < K; ++i) g[i] = (T0[i] < p.Tm) ? phi[i] : 0.0;
    const double gleft = ebm_shfl_up1(g[K - 1]), gright = ebm_shfl_dn1(g[0]);
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const int s = i * 32 + lane;
      const int j = lane * K + i;
      const double gm = (i == 0) ? gleft : g[i - 1];
      const double gp = (i == K - 1) ? gright : g[i + 1];
      double lo, up, di;
      if (kind == 1) {   // oracle miz_diff_coeffs
        up = (j < nx - 1) ? p.D * tabs.mxxph[s] / tabs.dxp[s] / tabs.phmmh[s] : 0.0;
        lo = (j > 0) ? p.D * tabs.mxxmh[s] / tabs.dxm[s] / tabs.phmmh[s] : 0.0;
        di = -(lo + up);
      } else {
        const double lm = tabs.cl[s], lp = tabs.cu[s];
        const double l1 = (j > 0) ? -lm : 0.0, l2 = (j < nx - 1) ? -lp : 0.0;
        const double l3 = -l1 - l2;
        lo = (j > 0) ? p.D * lm : 0.0; up = (j < nx - 1) ? p.D * lp : 0.0; di = p.D * (-l3);
      }
      jd[i] = -(p.k / hp[i] + p.B) + di * g[i];
      jl[i] = (j > 0 && j < nx) ? lo * gm : 0.0;
      ju[i] = (j < nx - 1) ? up * gp : 0.0;
      res[i] = (j < nx) ? -res[i] : 0.0;
    }
    miz_tridiag<K>(tabs, nx, lane, jl, jd, ju, res);
#pragma unroll
    for (int i = 0; i < K; ++i) T0[i] += res[i];
    ++it;
  }
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const double ti = jl_min(T0[i], p.Tm);                                          // :65
    Ti[i] = (h[i] == 0.0) ? 0.0 : ti;                                               // :66 zeroref!(Ti, h)
  }
  return it;
}

// ---- field output of one step for a member with L1/L2 output: savesol! (infrastructure.jl:549-591) ----------------------
// v[var][i] = the ten stored variables of this lane's cells (order of include/ebm_cuda.h EBM_MV_*)
template <int K>
__device__ __forceinline__ void miz_store_fields(const MizKArgs& a, int lane, long long msel, int year, int ti,
                                                 int season, const double (&v)[EBM_MIZ_NVAR][K]) {
  const int nx = a.nx, nt = a.nt;
  // the one step of ebm_miz_step (single_ti) has one raw slot
  if (a.raw != nullptr && (a.single_ti > 0 || ebm_raw_year(year, a.dur, a.lastonly))) {
    const long long nraw = a.single_ti > 0 ? 1 : ebm_nraw(nt, a.dur, a.lastonly);
    const long long rawidx = a.single_ti > 0 ? 0 : ebm_raw_slot(year, ti, nt, a.lastonly);
    double* o = a.raw + ebm_raw_offset(msel, nraw, rawidx, EBM_MIZ_NVAR, nx);
#pragma unroll
    for (int q = 0; q < EBM_MIZ_NVAR; ++q)
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const int j = lane * K + i;
        if (j < nx) o[(long long)q * nx + j] = v[q][i];
      }
  }
  if (a.seasonal != nullptr) {
    double* yr = a.seasonal + ebm_seasonal_offset(msel, a.dur, year, 0, EBM_MIZ_NVAR, nx);
    // the annual-mean slot doubles as the running sum of the year (annusol.raw -> crossmean, :556-559, :583-588)
    double* av = yr + 2LL * EBM_MIZ_NVAR * nx;
#pragma unroll
    for (int q = 0; q < EBM_MIZ_NVAR; ++q)
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const int j = lane * K + i;
        if (j < nx) {
          double* c = av + (long long)q * nx + j;
          const double sum = (ti == 1) ? v[q][i] : *c + v[q][i];
          *c = (ti == nt) ? sum / (double)nt : sum;
          if (season == 0 || season == 1) yr[((long long)season * EBM_MIZ_NVAR + q) * nx + j] = v[q][i];
        }
      }
  }
}

// ---- the kernel --------------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(kWarpsPerCta * 32) miz_warp_kernel(const MizKArgs a) {
  __shared__ MizTabs<K> tabs;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nx = a.nx, nt = a.nt, kind = a.g.kind;
  const long long nmem = a.nmem;

  for (int s = threadIdx.x; s < K * 32; s += blockDim.x) {
    const int i = s >> 5, l = s & 31;
    const int j = l * K + i;
    const bool v = j < nx;
    tabs.x[s] = v ? a.g.x[j] : 0.0;
    tabs.x2[s] = v ? a.g.x2[j] : 0.0;
    tabs.wts[s] = v ? a.g.wts[j] : 0.0;
    double cu = 0.0, cl = 0.0;
    if (v) {
      if (kind == 1) {
        cu = (j < nx - 1) ? a.g.mxxph[j] / a.g.diffx[j + 1] / a.g.phmmh[j] : 0.0;
        cl = (j > 0) ? a.g.mxxmh[j] / a.g.diffx[j] / a.g.phmmh[j] : 0.0;
      } else {
        cu = a.g.lam_hi[j]; cl = a.g.lam_lo[j];
      }
    }
    tabs.cu[s] = cu; tabs.cl[s] = cl;
    tabs.mxxph[s] = v ? a.g.mxxph[j] : 0.0; tabs.mxxmh[s] = v ? a.g.mxxmh[j] : 0.0;
    tabs.phmmh[s] = v ? a.g.phmmh[j] : 1.0;
    tabs.dxp[s] = v ? a.g.diffx[j + 1] : 1.0; tabs.dxm[s] = v ? a.g.diffx[j] : 1.0;
  }
  __syncthreads();

  const long long m = (long long)blockIdx.x * kWarpsPerCta + warp;
  if (m >= nmem) return;   // whole warp; no CTA barrier follows

  MizPar p;
  {
    const double* q = a.par + m;
    p.D = q[0 * nmem]; p.A = q[1 * nmem]; p.B = q[2 * nmem]; p.cw = q[3 * nmem]; p.S0 = q[4 * nmem];
    p.S1 = q[5 * nmem]; p.S2 = q[6 * nmem]; p.a0 = q[7 * nmem]; p.a2 = q[8 * nmem]; p.ai = q[9 * nmem];
    p.Fb = q[10 * nmem]; p.k = q[11 * nmem]; p.Lf = q[12 * nmem]; p.Tm = q[13 * nmem]; p.m1 = q[14 * nmem];
    p.m2 = q[15 * nmem]; p.alpha = q[16 * nmem]; p.rl = q[17 * nmem]; p.Dmin = q[18 * nmem]; p.Dmax = q[19 * nmem];
    p.hmin = q[20 * nmem]; p.kappa = q[21 * nmem];
  }
  double fr[EBM_NFORCING];
#pragma unroll
  for (int r = 0; r < EBM_NFORCING; ++r) fr[r] = (a.single_ti > 0) ? 0.0 : a.forc[(long long)r * nmem + m];
  const auto frow = [&](int r) { return fr[r]; };
  const bool constf = ebm_forcing_const(frow);

  const double dt = 1.0 / nt;
  const double Tm_m2 = pow(p.Tm, p.m2);                                     // wlat :71 -- `Tm^m2` binds to Tm (sic)
  const double denom_dn = p.Lf * p.alpha * (p.Dmin * p.Dmin) * p.hmin;      // psinplus :127

  MizMember<K> s;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = lane * K + i;
    const bool v = j < nx;
    const long long o = (long long)j * nmem + m;
    s.Ei[i] = v ? a.Ei[o] : 0.0; s.Ew[i] = v ? a.Ew[o] : 0.0; s.h[i] = v ? a.h[o] : 0.0;
    s.D[i] = v ? a.D[o] : 0.0; s.phi[i] = v ? a.phi[o] : 0.0; s.T0[i] = v ? a.T0[o] : 0.0;
  }
  s.accT = s.accE = s.accP = 0.0;
  s.icebits = 0u;

  const bool sel = ebm_field_selected(a, m) && (a.seasonal != nullptr || a.raw != nullptr);
  const long long msel = sel ? ebm_field_row(a, m) : 0;
  long long iters_total = 0, fails_total = 0;

  const int ti_first = a.single_ti > 0 ? a.single_ti : 1;
  const int ti_last = a.single_ti > 0 ? a.single_ti : nt;

  const long long step_stop = a.step_limit > 0 ? (long long)a.step_limit : 0x7fffffffffffffffLL;
  for (int year = a.year0; year < a.year0 + a.nyears; ++year) {
    for (int ti = ti_first; ti <= ti_last; ++ti) {
      if ((long long)year * nt + ti > step_stop) break;   // ebm_options_t.step_limit (warp-uniform)
      const double c2pt = __ldg(a.g.ctab + (ti - 1));                       // cos(2*pi*t)
      double f = fr[0];
      if (a.single_ti > 0) f = a.single_f;
      else if (!constf)
        f = ebm_forcing_at(frow, (long long)(year + a.start_year) * nt + ti, nt);
      const int season = ebm_season(a, ti, nt);

      // ---- temperatures (miz.jl:156-158)
      double Tw[K], Ti[K];
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const double v = p.Tm + s.Ew[i] / ((1 - s.phi[i]) * p.cw);          // water_temp :30
        Tw[i] = (v != v) ? 0.0 : v;                                         // :157
      }
      int fail = 0;
      iters_total += miz_solveTi<K>(tabs, p, kind, nx, lane, f, c2pt, s.h, Tw, s.phi, s.T0, Ti, a.tol, a.maxit, &fail);
      fails_total += fail;

      // ---- fluxes (:160-164)
      double n[K], tb[K], dif[K];
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const double v = s.phi[i] / (p.alpha * (s.D[i] * s.D[i]));          // num :84
        n[i] = (s.D[i] == 0.0) ? 0.0 : v;                                   // :85
        tb[i] = Ti[i] * s.phi[i] + (1 - s.phi[i]) * Tw[i];                  // Tbar(Ti, Tw, phi)
      }
      miz_diffusion<K>(tabs, p, kind, nx, lane, tb, dif);

      double out[EBM_MIZ_NVAR][K];
      double dgT = 0.0, dgE = 0.0, dgP = 0.0, dgX = 2.0;
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const int sidx = i * 32 + lane;
        const double xj = tabs.x[sidx], x2j = tabs.x2[sidx];
        const double Ei = s.Ei[i], Ew = s.Ew[i], h = s.h[i], D = s.D[i], phi = s.phi[i];
        const double ins = p.S0 - p.S1 * xj * c2pt - p.S2 * x2j;                              // :11
        const double Lolr = p.A + p.B * (tb[i] - p.Tm);                                      // :99
        const double sol_i = 0.0 + p.ai * ins;                                               // solar(ice)
        const double sol_w = 0.0 + (p.a0 - p.a2 * x2j) * ins;                                // solar(water) :14
        const double difz = 0.0 + dif[i];
        const double Fvi = sol_i - Lolr + difz + p.Fb + f;                                   // :100
        const double Fvw = sol_w - Lolr + difz + p.Fb + f;
        const double wl = p.m1 * (Tw[i] - Tm_m2);                                            // :71
        double Flat = phi * h * p.Lf * wl * kPi / (p.alpha * D);                             // :104
        if (D == 0.0) Flat = 0.0;                                                            // :105
        const double rEi = Ei + (phi * Fvi + Flat) * dt;                                     // :137,148,166
        const double rEw = Ew + ((1 - phi) * Fvw - Flat) * dt;                               // :138,148,167
        // redistributeE :109-117
        const double cEi = jl_clamp(rEi, -INFINITY, 0.0), cEw = jl_clamp(rEw, 0.0, INFINITY);
        const double psiEidt = rEi - cEi, psiEwdt = rEw - cEw;
        double Ei_n = cEi + psiEwdt;
        const double Ew_n = cEw + psiEidt;
        // area_lead :90-93 (n from the start of the step)
        const double d2rl = D + 2.0 * p.rl;
        const double ring = p.alpha * n[i] * (d2rl * d2rl - D * D);
        const double Al = jl_min(ring, 1.0 - phi);
        // split_psiEw :120-125 on psiEwdt/dt (:173)
        const double psiEw = psiEwdt / dt;
        double Ql = Al / (1 - phi) * psiEw;
        if (phi == 1.0) Ql = 0.0;
        const double Qp = psiEw - Ql;
        const double dn = dt * (-Qp / denom_dn);                                             // :127,174
        // D_t :140-146
        const double lat_melt = -kPi / 2.0 * p.alpha * wl;                                   // :141 (sic)
        double lat_grow = -D / (2 * p.Lf * h * phi) * Ql;                                    // :142
        const double D3 = D * D * D;
        const double weld = p.kappa * p.alpha / 4 * phi * D3;                                // :143
        if (h == 0.0) lat_grow = 0.0;                                                        // :144
        const double Dt = lat_melt + lat_grow + weld;                                        // :145
        const double rD = D + Dt * dt;                                                       // :175
        // average :129-134
        const double total = n[i] + dn;
        double Dn = (n[i] * rD + dn * p.Dmin) / total;
        if (total == 0.0) Dn = 0.0;
        Dn = jl_clamp(Dn, p.Dmin, p.Dmax);                                                   // :177
        if (Ei_n == 0.0) Dn = 0.0;                                                           // :178
        double rh = h + (-1 / p.Lf * Fvi) * dt;                                              // :139,179
        rh = jl_clamp(rh, 0.0, INFINITY);                                                    // :180
        double hn = (n[i] * rh + dn * p.hmin) / total;                                       // :181
        if (total == 0.0) hn = 0.0;
        // concentration :74-80
        double ph = -Ei_n / (p.Lf * hn);
        if (hn == 0.0) ph = 0.0;
        if (ph > 1.0) ph = 1.0;
        if (hn == 0.0) Ei_n = 0.0;                                                           // :185
        const double En = ph * Ei_n + (1 - ph) * Ew_n;                                       // :186
        const double Tn = Ti[i] * ph + (1 - ph) * Tw[i];                                     // :187
        s.Ei[i] = Ei_n; s.Ew[i] = Ew_n; s.D[i] = Dn; s.h[i] = hn; s.phi[i] = ph;

        // ---- sampling
        const bool real = lane * K + i < nx;
        const double wj = tabs.wts[sidx];
        s.accT = fma(wj, Tn, s.accT); s.accE = fma(wj, En, s.accE); s.accP = fma(wj, ph, s.accP);
        if (ph > 0.0 && real) s.icebits |= 1u << i;
        if (season == 0 || season == 1) {
          dgT = fma(wj, Tn, dgT); dgE = fma(wj, En, dgE); dgP = fma(wj, ph, dgP);
          if (ph > 0.0 && real) dgX = fmin(dgX, xj);
        } else if (season == 2) {
          if (((s.icebits >> i) & 1u) != 0u) dgX = fmin(dgX, xj);
        }
        if (sel) {
          out[EBM_MV_T][i] = Tn; out[EBM_MV_Ei][i] = Ei_n;
          out[EBM_MV_Ti][i] = (Ei_n == 0.0) ? NAN : Ti[i];                                   // :193
          out[EBM_MV_D][i] = Dn; out[EBM_MV_n][i] = n[i]; out[EBM_MV_h][i] = hn; out[EBM_MV_phi][i] = ph;
          out[EBM_MV_E][i] = En; out[EBM_MV_Ew][i] = Ew_n;
          out[EBM_MV_Tw][i] = (ph > 0.99) ? NAN : Tw[i];                                     // :194
        }
      }
      if (sel) miz_store_fields<K>(a, lane, msel, year, ti, season, out);
      if (season >= 0 && a.diag != nullptr) {
        if (season == 2) {   // annual means: mean over the year of the hemispheric means (linear)
          dgT = s.accT / (double)nt; dgE = s.accE / (double)nt; dgP = s.accP / (double)nt;
        }
        const double t0 = ebm_warp_sum(dgT), t1 = ebm_warp_sum(dgE), t2 = ebm_warp_sum(dgP), t3 = ebm_warp_min(dgX);
        if (lane == 0) ebm_store_diag(a.diag, m, a.dur, year, season, t0, t1, t2, t3);
      }
      if (ti == nt) { s.accT = s.accE = s.accP = 0.0; s.icebits = 0u; }
    }
  }

  // ---- final state
  bool bad = false;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = lane * K + i;
    if (j < nx) {
      const long long o = (long long)j * nmem + m;
      a.Ei[o] = s.Ei[i]; a.Ew[o] = s.Ew[i]; a.h[o] = s.h[i]; a.D[o] = s.D[i]; a.phi[o] = s.phi[i]; a.T0[o] = s.T0[i];
      bad = bad || ebm_state_bad(s.Ei[i]) || ebm_state_bad(s.Ew[i]) || ebm_state_bad(s.h[i]) || ebm_state_bad(s.D[i]) ||
            ebm_state_bad(s.phi[i]);
    }
  }
  bad = __any_sync(kFull, bad);
  if (lane == 0) {
    if (a.newton_iters != nullptr) a.newton_iters[m] += iters_total;
    if (a.nonconv != nullptr) a.nonconv[m] += fails_total;
    if (bad && a.flags != nullptr) a.flags[m] |= 1;
  }
}

template <int K>
int miz_launch_k(const MizKArgs& a, cudaStream_t stream) {
  const long long blocks = (a.nmem + kWarpsPerCta - 1) / kWarpsPerCta;
  if (blocks > 0x7fffffffLL) { ebm_set_error("miz: too many members (%lld)", a.nmem); return EBM_ERR_INVALID; }
  miz_warp_kernel<K><<<(unsigned)blocks, kWarpsPerCta * 32, 0, stream>>>(a);
  EBM_CUDA_TRY(cudaGetLastError());
  ebm_count_launch();
  return EBM_OK;
}

int miz_launch_any(const MizKArgs& a, cudaStream_t stream) {
  if (a.nx < 3) { ebm_set_error("miz: nx must be >= 3"); return EBM_ERR_INVALID; }
  if (a.nx <= 64) return miz_launch_k<2>(a, stream);
  if (a.nx <= 128) return miz_launch_k<4>(a, stream);
  if (a.nx <= 192) return miz_launch_k<6>(a, stream);
  if (a.nx <= 256) return miz_launch_k<8>(a, stream);
  ebm_set_error("miz: nx=%d > 256 not supported by the register-resident kernel", a.nx);
  return EBM_ERR_UNSUPPORTED;
}

}  // namespace
