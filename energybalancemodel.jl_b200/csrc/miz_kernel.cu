// miz_kernel.cu -- production (fast) flavour of the marginal-ice-zone (MIZ) ensemble step kernel, and the launch dispatch.
//
// Replaces, for a whole ensemble and many years per launch, the reference's
//   integrate loop            src/infrastructure.jl:630-634
//   step!(::Val{:MIZ})        src/miz.jl:150-196        (arithmetic spec: SURVEY.md Appendix B)
//   solveTi / T0eq            src/miz.jl:33-68          (closure: semi-smooth Newton, tridiagonal Jacobian)
//   diffusion!                src/infrastructure.jl:495-527 (identity grid and generic flux-form stencil)
//   savesol! / annual_mean    src/infrastructure.jl:536-591
// The literal-order twin of this kernel (bit-identical to the oracle) is miz_literal.cuh / miz_strict.cu; the
// algebra here is the same step with
//   * every division turned into a reciprocal (MUFU.RCP64H seed + one cubic step) times a product, reciprocals
//     shared between quotients with the same denominator, constant quotients hoisted per member; denominators that
//     the reference masks afterwards (zeroref!: D == 0, h == 0, n + dn == 0, phi == 1) are replaced by 1 BEFORE
//     the reciprocal so that open-water cells never enter the IEEE slow path (they did 13 times per cell-step in the
//     literal flavour: 0/0 everywhere); unmasked special operands still take the literal x / y (rare branch);
//   * the closure residual folded to (k/hp + B)*(Tm - T0) + (ai*S - A + f) + D nabla^2 Tbar, k/hp computed once
//     per step, stencil coefficients pre-scaled by the member's D in per-warp shared memory;
//   * FMA contraction.
// Mapping (B200: 148 SMs x 4 sub-partitions x 16 FP64 lanes, 64K registers per SM):
//   * one WARP integrates one member; lane l owns the K contiguous cells j = l*K .. l*K+K-1 (K = ceil(nx/32)); the
//     six state vectors (Ei, Ew, h, D, phi, closure warm start T0) stay in registers for the whole launch;
//   * no CTA barrier and no shared-memory exchange in the time loop: neighbour temperatures cross lanes with two
//     shuffles per stencil evaluation, Newton convergence is a warp vote (every member iterates as often as it
//     needs), the tridiagonal Jacobian system is solved partitioned -- K rows per lane with a left spike, parallel
//     cyclic reduction over shuffles for the 32 interface unknowns, local back substitution;
//   * geometry tables are per-CTA shared memory laid out [cell-in-lane][lane] (bank-conflict free);
//   * cos(2*pi*t) comes from a per-step table built on the host (same libm as the oracle).
// Results agree with the oracle to rounding over short horizons; the MIZ dynamics amplify rounding differences
// (DESIGN.md "MIZ sensitivity"), so long runs are compared through the literal kernel instead.
#include <math.h>
#include <type_traits>
#include <string.h>

#include "ebm_internal.cuh"

namespace {

constexpr int kWarps = 4;                   // members per CTA
constexpr int kGC = 3;                      // cells per statement-major group when K allows it (DESIGN.md 4.3)

// c ? a : b as one SELP with both operands evaluated: the compiler otherwise branches around "expensive" operands,
// which splits the unrolled per-cell code into scheduling regions and serialises the K cells of a lane
__device__ __forceinline__ double keep(double v) {
  // an empty asm "touches" the operand: it must be computed before the select and cannot be sunk into a conditional
  // arm; the select itself stays a plain predicate select (2 FSEL, no predicate materialisation)
  asm("" : "+d"(v));
  return v;
}
__device__ __forceinline__ double sel(bool c, double a, double b) { return c ? keep(a) : keep(b); }
// c ? 0 : b and c ? 1 : b as bit masks on the two words (2 LOP3 each; the mask of a condition is shared by all its
// uses): ptxas lowers a select against an immediate 0.0 / 1.0 to "materialise the constant + two predicated moves",
// 3-4 instructions per select and a third of this kernel's instruction count (profiles/r2_miz_fast_ncu.txt)
__device__ __forceinline__ double sel0(bool c, double b) {
  const int m = c ? 0 : -1;
  return __hiloint2double(__double2hiint(b) & m, __double2loint(b) & m);
}
__device__ __forceinline__ double sel1(bool c, double b) {
  const int m = c ? 0 : -1;
  return __hiloint2double((__double2hiint(b) & m) | (0x3ff00000 & ~m), __double2loint(b) & m);
}
// zero / sign tests on the integer pipe (the FP64 pipe is the bottleneck); +0 and -0 are both zero
__device__ __forceinline__ bool is_zero(double v) { return ((__double2hiint(v) & 0x7fffffff) | __double2loint(v)) == 0; }   // one LOP3 with predicate output
// x / y with y an ordinary non-zero number (no denormal / huge denominators: DESIGN.md 4.3)
__device__ __forceinline__ double div_n(double x, double y) { return x * ebm_rcp(y); }
// x / y with y zero or ordinary: IEEE results for y == +-0 (x/0 = +-Inf, 0/0 = NaN/0 = NaN), branch free
__device__ __forceinline__ double div_z(double x, double y) {
  const bool z = is_zero(y);
  const double q = x * ebm_rcp(sel1(z, y));
  const double inf = __hiloint2double(0x7ff00000 | ((__double2hiint(x) ^ __double2hiint(y)) & 0x80000000), 0);
  const double zq = (is_zero(x) || x != x) ? __longlong_as_double(0x7ff8000000000000LL) : inf;
  return sel(z, zq, q);
}

template <int K>
struct Tabs {   // per CTA, [i][lane] for cell j = lane*K + i
  double x[K * 32], x2[K * 32], wts[K * 32];
  double lo[kWarps][K * 32], up[kWarps][K * 32];   // member's D times the stencil coefficient towards j-1 / j+1
  double cst[kWarps][56];                          // member constants (warp-uniform: broadcast loads, not registers)
  double cold[kWarps][7 * K * 32];                 // Ei, Ew, D, h, Tw, 1/(1-phi), 1/hp: touched once or twice per step
};

// indices into Tabs::cst
enum { cA, cB, ccw, cS0, cS1, cS2, ca0, ca2, cai, cFb, ck, cLf, cTm, cm1, calpha, cDmin, cDmax, chmin,
       cTm_m2, cinv_alpha, cc_dn, cc_melt, cc_weld, cc_flat, cdt_Lf, ctwoLf, ctworl,
       cinv_cw, cinv_Lf, cinv_hmin, cc_r1, cc_r2, cc_wl0, ccBF, cF0, cNCST = cF0 + EBM_NFORCING };

// ---- D nabla^2 of a profile held K cells per lane:  up*(T[j+1]-T[j]) - lo*(T[j]-T[j-1])  (infrastructure.jl:495-527)
template <int K>
__device__ __forceinline__ void diffuse(const double* __restrict__ lo, const double* __restrict__ up, int lane,
                                        const double (&tb)[K], double (&out)[K]) {
  const double left = ebm_shfl_up1(tb[K - 1]);
  const double right = ebm_shfl_dn1(tb[0]);
  // d[i] = T[j] - T[j-1] for the lane's cells, d[K] towards the next lane: each difference serves two cells
  double d[K + 1];
  d[0] = tb[0] - left;
#pragma unroll
  for (int i = 1; i < K; ++i) d[i] = tb[i] - tb[i - 1];
  d[K] = right - tb[K - 1];
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int s = i * 32 + lane;
    out[i] = fma(up[s], d[i + 1], -lo[s] * d[i]);   // a zero coefficient silences the missing neighbour
  }
}

// ---- tridiagonal solve across the warp, K rows per lane; rhs -> solution -----------------------------------------------
// row(i, jl, jd, ju) produces row i on demand, so the three coefficient vectors never live in registers at once
template <int K, class RowFn>
__device__ __forceinline__ void tridiag(int lane, RowFn row, double (&rhs)[K]) {
  // local forward elimination:  x_i + q_i x_{i+1} + s_i xL = y_i   (xL = last unknown of the previous lane)
  // Pivots in determinant form: P_i = w_0 ... w_i obeys P_i = d_i P_{i-1} - (l_i u_{i-1}) P_{i-2} -- one dependent FMA
  // per row instead of FMA -> reciprocal -> product (the K reciprocals 1/w_i = P_{i-1}/P_i are then independent of
  // each other; |w| <= 2 D / dx^2 + k/hmin + B ~ 1e5, so P stays far inside the double range for K <= 8)
  double q[K], s[K];
  {
    double Pm2 = 1.0, Pm1 = 1.0, jup = 0.0;
#pragma unroll
    for (int i = 0; i < K; ++i) {
      double jl_i, jd_i, ju_i;
      row(i, jl_i, jd_i, ju_i);
      const double P = (i == 0) ? jd_i : fma(jd_i, Pm1, -((jl_i * jup) * Pm2));
      const double iw = Pm1 * ebm_rcp(P);
      s[i] = jl_i * iw;                       // tq_i, turned into the spike below
      q[i] = ju_i * iw;
      rhs[i] = rhs[i] * iw;
      Pm2 = Pm1; Pm1 = P; jup = ju_i;
    }
#pragma unroll
    for (int i = 1; i < K; ++i) {
      rhs[i] = fma(-s[i], rhs[i - 1], rhs[i]);
      s[i] = -s[i] * s[i - 1];
    }
  }
  // reduce row 0 to  x_0 = al - be*xL - ga*z   (z = my last unknown)
  double al = rhs[K - 2], be = s[K - 2], ga = q[K - 2];
#pragma unroll
  for (int i = K - 3; i >= 0; --i) {
    al = fma(-q[i], al, rhs[i]);
    be = fma(-q[i], be, s[i]);
    ga = -q[i] * ga;
  }
  // interface row of this lane:  A z_{l-1} + B z_l + C z_{l+1} = R, from the next lane's (al, be, ga)
  const double nal = ebm_shfl_dn1(al), nbe = ebm_shfl_dn1(be), nga = ebm_shfl_dn1(ga);
  const double ql = (lane == 31) ? 0.0 : q[K - 1];
  double A = (lane == 0) ? 0.0 : s[K - 1];
  double C = -ql * nga;
  double R = fma(-ql, nal, rhs[K - 1]);
  {
    const double ib = ebm_rcp(fma(-ql, nbe, 1.0));
    A *= ib; C *= ib; R *= ib;
  }
  // parallel cyclic reduction, rows kept normalised (B = 1); out-of-range neighbours are identity rows
#pragma unroll
  for (int st = 1; st < 32; st <<= 1) {
    // couplings shrink quadratically (products of 2^k original ones): the last steps are usually no-ops
    if (st >= 4 && !__any_sync(kFull, fabs(A) + fabs(C) > 1e-19)) break;
    const double Au = __shfl_up_sync(kFull, A, st), Cu = __shfl_up_sync(kFull, C, st), Ru = __shfl_up_sync(kFull, R, st);
    const double Ad = __shfl_down_sync(kFull, A, st), Cd = __shfl_down_sync(kFull, C, st), Rd = __shfl_down_sync(kFull, R, st);
    const double a_ = (lane >= st) ? A : 0.0, c_ = (lane + st < 32) ? C : 0.0;
    const double ib = ebm_rcp(fma(-a_, Cu, fma(-c_, Ad, 1.0)));
    const double Rn = fma(-a_, Ru, fma(-c_, Rd, R));
    A = -(a_ * Au) * ib;
    C = -(c_ * Cd) * ib;
    R = Rn * ib;
  }
  const double z = R;
  const double zup = ebm_shfl_up1(z);              // every lane executes the shuffle (full mask)
  const double xL = (lane == 0) ? 0.0 : zup;
  double xn = z;
  rhs[K - 1] = z;
#pragma unroll
  for (int i = K - 2; i >= 0; --i) {
    xn = fma(-q[i], xn, fma(-s[i], xL, rhs[i]));
    rhs[i] = xn;
  }
}

// ---- field output of one cell for a member with L1/L2 output: savesol! (infrastructure.jl:549-591) --------------------
// v = the ten stored variables of cell j (order of include/ebm_cuda.h EBM_MV_*)
__device__ __forceinline__ void store_cell(const MizKArgs& a, int j, long long msel, int year, int ti, int season,
                                           const double (&v)[EBM_MIZ_NVAR]) {
  const int nx = a.nx, nt = a.nt;
  if (a.raw != nullptr && (!a.lastonly || year == a.dur - 1)) {   // not ebm_raw_year: -70 to +11 instructions
    double* o = a.raw + ebm_raw_offset(msel, ebm_nraw(nt, a.dur, a.lastonly), ebm_raw_slot(year, ti, nt, a.lastonly),
                                       EBM_MIZ_NVAR, nx) + j;
#pragma unroll
    for (int q = 0; q < EBM_MIZ_NVAR; ++q) o[(long long)q * nx] = v[q];
  }
  if (a.seasonal != nullptr) {
    double* yr = a.seasonal + ebm_seasonal_offset(msel, a.dur, year, 0, EBM_MIZ_NVAR, nx) + j;
    // the annual-mean slot doubles as the running sum of the year (annusol.raw -> crossmean, :556-559, :583-588)
    double* av = yr + 2LL * EBM_MIZ_NVAR * nx;
#pragma unroll
    for (int q = 0; q < EBM_MIZ_NVAR; ++q) {
      double* c = av + (long long)q * nx;
      const double sum = (ti == 1) ? v[q] : *c + v[q];
      *c = (ti == nt) ? sum / (double)nt : sum;
      if (season == 0 || season == 1) yr[((long long)season * EBM_MIZ_NVAR + q) * nx] = v[q];
    }
  }
}

template <int K, int MINB>
__global__ void __launch_bounds__(kWarps * 32, MINB) miz_fast_kernel(const MizKArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Tabs<K>& tabs = *reinterpret_cast<Tabs<K>*>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nx = a.nx, nt = a.nt, kind = a.g.kind;
  const long long nmem = a.nmem;
  const long long m_raw = (long long)blockIdx.x * kWarps + warp;
  const long long m = m_raw < nmem ? m_raw : nmem - 1;

  for (int s = threadIdx.x; s < K * 32; s += blockDim.x) {
    const int i = s >> 5, l = s & 31;
    const int j = l * K + i;
    const bool v = j < nx;
    tabs.x[s] = v ? a.g.x[j] : 0.0;
    tabs.x2[s] = v ? a.g.x2[j] : 0.0;
    tabs.wts[s] = v ? a.g.wts[j] : 0.0;
  }
  {
    const double Dm = a.par[0 * nmem + m];
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const int j = lane * K + i;
      double cu = 0.0, cl = 0.0;
      if (j < nx) {   // not a shared helper: every formulation tried reorders this kernel's code
        if (kind == 1) {   // generic flux-form stencil, infrastructure.jl:510-524
          cu = (j < nx - 1) ? a.g.mxxph[j] / a.g.diffx[j + 1] / a.g.phmmh[j] : 0.0;
          cl = (j > 0) ? a.g.mxxmh[j] / a.g.diffx[j] / a.g.phmmh[j] : 0.0;
        } else {           // get_diffop, infrastructure.jl:480-489
          cu = a.g.lam_hi[j]; cl = a.g.lam_lo[j];
        }
      }
      tabs.up[warp][i * 32 + lane] = Dm * cu;
      tabs.lo[warp][i * 32 + lane] = Dm * cl;
    }
  }
  __syncthreads();
  if (m_raw >= nmem) return;   // whole warp; no CTA barrier follows
  const double* __restrict__ lo = tabs.lo[warp];
  const double* __restrict__ up = tabs.up[warp];

  // ---- member constants (miz_paramset, infrastructure.jl:436-441) -> per-warp shared memory
  const int nt_ = nt;
  const double dt = 1.0 / nt_, ntd = (double)nt_;
  if (lane == 0) {
    const double* q = a.par + m;
    double* c = tabs.cst[warp];
    const double pLf = q[12 * nmem], pTm = q[13 * nmem], pm2 = q[15 * nmem], palpha = q[16 * nmem], prl = q[17 * nmem];
    const double pDmin = q[18 * nmem], phmin = q[20 * nmem], pkappa = q[21 * nmem];
    c[cA] = q[1 * nmem]; c[cB] = q[2 * nmem]; c[ccw] = q[3 * nmem]; c[cS0] = q[4 * nmem]; c[cS1] = q[5 * nmem];
    c[cS2] = q[6 * nmem]; c[ca0] = q[7 * nmem]; c[ca2] = q[8 * nmem]; c[cai] = q[9 * nmem]; c[cFb] = q[10 * nmem];
    c[ck] = q[11 * nmem]; c[cLf] = pLf; c[cTm] = pTm; c[cm1] = q[14 * nmem]; c[calpha] = palpha;
    c[cDmin] = pDmin; c[cDmax] = q[19 * nmem]; c[chmin] = phmin;
    c[cTm_m2] = pow(pTm, pm2);                                               // wlat :71 -- `Tm^m2` binds to Tm (sic)
    c[cinv_alpha] = 1.0 / palpha;
    c[cc_dn] = dt / (pLf * palpha * (pDmin * pDmin) * phmin);               // psinplus :127 times dt (:174)
    c[cc_melt] = -kPi / 2.0 * palpha;                                        // :141 (sic)
    c[cc_weld] = pkappa * palpha / 4;                                        // :143
    c[cc_flat] = pLf * kPi * (1.0 / palpha);                                 // :104
    c[cdt_Lf] = dt / pLf;                                                    // :139
    c[ctwoLf] = 2 * pLf;
    c[ctworl] = 2.0 * prl;
    c[cinv_cw] = 1.0 / c[ccw]; c[cinv_Lf] = 1.0 / pLf; c[cinv_hmin] = ebm_rcp(phmin);
    c[cc_r1] = 4.0 * prl; c[cc_r2] = 4.0 * prl * prl;                        // (D + 2 rl)^2 - D^2 = 4 rl D + 4 rl^2  (:91)
    c[cc_wl0] = -c[cm1] * c[cTm_m2];                                         // wlat = m1*Tw - m1*Tm^m2       (:71)
    c[ccBF] = c[cB] * pTm + c[cFb];
    for (int r = 0; r < EBM_NFORCING; ++r) c[cF0 + r] = a.forc[(long long)r * nmem + m];
  }
  __syncwarp();
  const double* cst = tabs.cst[warp];   // re-read after every STEP_FENCE: constants are CSE'd within a phase only
#define CST(name) (cst[c##name])
#define STEP_FENCE() asm volatile("" ::: "memory")
  const auto frow = [&](int r) { return cst[cF0 + r]; };
  const bool constf = ebm_forcing_const(frow);

  // Ei, Ew and D are read and written once per step (outside the closure): they live in thread-private shared
  // memory [array][i][lane]; h, phi and the warm start T0 stay in registers
  double* const cold = tabs.cold[warp] + lane;
#define EI(i) cold[(0 * K + (i)) * 32]
#define EW(i) cold[(1 * K + (i)) * 32]
#define DD(i) cold[(2 * K + (i)) * 32]
#define HH(i) cold[(3 * K + (i)) * 32]
#define TW(i) cold[(4 * K + (i)) * 32]
#define ROM(i) cold[(5 * K + (i)) * 32]   /* 1/(1-phi) of this step (1 where phi == 1) */
#define RHP(i) cold[(6 * K + (i)) * 32]   /* 1/hp, hp = h or hmin where h == 0: carried from the step that made h */
  double phi[K], T0[K];
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = lane * K + i;
    const bool v = j < nx;
    const long long o = (long long)j * nmem + m;
    EI(i) = v ? a.Ei[o] : 0.0; EW(i) = v ? a.Ew[o] : 0.0; HH(i) = v ? a.h[o] : 0.0;
    DD(i) = v ? a.D[o] : 0.0; phi[i] = v ? a.phi[o] : 0.0; T0[i] = v ? a.T0[o] : 0.0;
    const double h0 = HH(i);
    RHP(i) = sel(is_zero(h0), cst[cinv_hmin], ebm_rcp(sel1(is_zero(h0), h0)));   // same expression as in the step
  }
  double accT = 0.0, accE = 0.0, accP = 0.0;   // running hemispheric sums of the year (annual means are linear)
  unsigned icebits = 0u;

  const bool sel_m = ebm_field_selected(a, m) && (a.seasonal != nullptr || a.raw != nullptr);
  const long long msel = sel_m ? ebm_field_row(a, m) : 0;
  long long iters_total = 0, fails_total = 0;
  const long long step_stop = a.step_limit > 0 ? (long long)a.step_limit : 0x7fffffffffffffffLL;
  const double tol = a.tol;
  const int maxit = a.maxit;

  for (int year = a.year0; year < a.year0 + a.nyears; ++year) {
    for (int ti = 1; ti <= nt; ++ti) {
      if ((long long)year * nt + ti > step_stop) break;   // ebm_options_t.step_limit (warp-uniform)
      STEP_FENCE();
      const double S1c = CST(S1) * __ldg(a.g.ctab + (ti - 1));                   // S1*cos(2*pi*t)
      double f = cst[cF0];
      if (!constf)
        f = ebm_forcing_at(frow, (long long)(year + a.start_year) * nt + ti, nt);
      const double fA = f - CST(A);
      const int season = ebm_season(a, ti, nt);

      // ---- temperatures and the closure's per-step constants (miz.jl:156-158, :33-60)
      double omTw[K], kb[K], c0[K];
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const int s = i * 32 + lane;
        const double om = 1 - phi[i];
        const bool one = phi[i] == 1.0;
        const double r_om = ebm_rcp(sel1(one, om));                         // shared by water_temp and split_psiEw
        ROM(i) = r_om;
        const double ew = EW(i);
        // Ew / ((1-phi) cw) (:30); phi == 1: the IEEE quotient by +0 (NaN for Ew == 0 or NaN, else +-Inf)
        const double qz = (is_zero(ew) || ew != ew) ? __longlong_as_double(0x7ff8000000000000LL)
                                                     : __hiloint2double(0x7ff00000 | (__double2hiint(ew) & 0x80000000), 0);
        const double v = CST(Tm) + sel(one, qz, ew * r_om * CST(inv_cw));
        const double tw = sel0(v != v, v);                                 // :157
        TW(i) = tw;
        omTw[i] = om * tw;
        kb[i] = fma(CST(k), RHP(i), CST(B));                                   // k/hp + B, hp = h or hmin (:51)
        const double S = fma(-CST(S2), tabs.x2[s], fma(-S1c, tabs.x[s], CST(S0)));   // :11
        c0[i] = fma(CST(ai), S, fA);                                             // ai*S - A + f
      }
      // ---- solveTi: semi-smooth Newton on  (k/hp + B)(Tm - T0) + c0 + D nabla^2(phi*min(T0,Tm) + (1-phi)Tw) = 0
      int it = 0, fail = 0;
      for (;;) {
        double tb[K], res[K];
#pragma unroll
        for (int i = 0; i < K; ++i) tb[i] = fma((T0[i] < CST(Tm)) ? T0[i] : CST(Tm), phi[i], omTw[i]);   // Tbar! :21-25
        diffuse<K>(lo, up, lane, tb, res);
        bool ok = true, nan = false;
#pragma unroll
        for (int i = 0; i < K; ++i) {
          const double v = fma(kb[i], CST(Tm) - T0[i], c0[i] + res[i]);          // T0eq :39-43
          res[i] = -v;
          const double av = (lane * K + i < nx) ? fabs(v) : 0.0;
          nan = nan || ((__double2hiint(av) & 0x7ff00000) == 0x7ff00000);   // NaN or Inf residual
          ok = ok && (av <= tol);
        }
        if (__all_sync(kFull, ok)) break;
        if (__any_sync(kFull, nan) || it >= maxit) { fail = 1; break; }
        // generalised Jacobian  J = -diag(k/hp + B) + L*diag(phi*[T0 < Tm])
        double g[K];
#pragma unroll
        for (int i = 0; i < K; ++i) {
          g[i] = (T0[i] < CST(Tm)) ? phi[i] : 0.0;
          res[i] = (lane * K + i >= nx) ? 0.0 : res[i];
        }
        const double gleft = ebm_shfl_up1(g[K - 1]), gright = ebm_shfl_dn1(g[0]);
        tridiag<K>(lane, [&](int i, double& jl, double& jd, double& ju) {
          const int s = i * 32 + lane;
          const double l = lo[s], u = up[s];
          jd = fma(-(l + u), g[i], -kb[i]);
          jl = l * ((i == 0) ? gleft : g[i - 1]);
          ju = u * ((i == K - 1) ? gright : g[i + 1]);
        }, res);
        // The residual is piecewise linear: if the step leaves the active set [T0 < Tm] (where phi != 0) unchanged,
        // the new T0 is the root to rounding (|res| ~ 1e-12 << tol) and the confirming residual evaluation the
        // reference performs is skipped; the iteration count is the same either way.
        bool changed = false, bad = false;
#pragma unroll
        for (int i = 0; i < K; ++i) {
          const double tn = T0[i] + res[i];
          changed = changed || (!is_zero(phi[i]) && ((T0[i] < CST(Tm)) != (tn < CST(Tm))));
          bad = bad || (tn != tn);
          T0[i] = tn;
        }
        ++it;
        if (__any_sync(kFull, bad)) { fail = 1; break; }
        if (!__any_sync(kFull, changed)) break;
      }
      iters_total += it;
      fails_total += fail;

      // ---- fluxes, enthalpy, floe size, thickness, concentration (:160-187)
      STEP_FENCE();
      double Ti[K], tb[K], dif[K];
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const double tmin = (T0[i] < CST(Tm)) ? T0[i] : ((T0[i] != T0[i]) ? T0[i] : CST(Tm));   // min(T0, Tm) :65
        Ti[i] = is_zero(HH(i)) ? 0.0 : tmin;                                            // :66
        tb[i] = fma(Ti[i], phi[i], omTw[i]);
      }
      diffuse<K>(lo, up, lane, tb, dif);

      double dgT = 0.0, dgE = 0.0, dgP = 0.0, dgX = 2.0;
      // two instantiations: the hot one (no sampling this step, no field output) is straight-line code
      auto cells = [&](auto slow_tag) {
      constexpr bool SLOW = decltype(slow_tag)::value;
      constexpr int GC = (K % kGC == 0) ? kGC : 2;   // cells per statement-major group (K is even)
      // ptxas keeps the source order to a large extent and a warp issues in order: written cell after cell, the six
      // ~100-instruction dependent chains of a lane run one after the other (static schedule: 2.6 issue cycles per FP64
      // instruction).  Statement-major over groups of GC cells -- every statement for the group's cells before the
      // next statement -- gives the warp GC independent chains; the arithmetic of every cell is unchanged.
#pragma unroll
      for (int g0 = 0; g0 < K; g0 += GC) {
        constexpr int G = GC;
#define FORG _Pragma("unroll") for (int g = 0; g < G; ++g)
#define I (g0 + g)
        double xj[G], x2j[G], Eio[G], Ewo[G], ho[G], Do[G], pho[G], om[G], S[G], common[G], Fvi[G], Fvw[G], wl[G], rD[G];
        double an[G], n[G], Flat[G], rEi[G], rEw[G], cEi[G], cEw[G], psiEw_dt[G], Ei_n[G], Ew_n[G], ring[G], Al[G];
        double psiEw[G], Ql[G], dn[G], lat_grow[G], Dt[G], rDn[G], total[G], rt[G], Dn[G], rh[G], hn[G], r_hn[G], ph[G];
        double omn[G], En[G], Tn[G], tw[G];
        bool noD[G], noh[G], one[G], tz[G], hz[G];
        FORG { const int sidx = I * 32 + lane; xj[g] = tabs.x[sidx]; x2j[g] = tabs.x2[sidx]; }
        FORG { Eio[g] = EI(I); Ewo[g] = EW(I); ho[g] = HH(I); Do[g] = DD(I); pho[g] = phi[I]; tw[g] = TW(I); }
        FORG om[g] = 1 - pho[g];
        FORG { noD[g] = is_zero(Do[g]); noh[g] = is_zero(ho[g]); one[g] = pho[g] == 1.0; }
        FORG S[g] = fma(-CST(S2), x2j[g], fma(-S1c, xj[g], CST(S0)));
        FORG common[g] = fma(-CST(B), tb[I], dif[I]) + CST(cBF);                       // -(A + B(Tb-Tm)) + diffusion + Fb (+ fA below)
        FORG Fvi[g] = c0[I] + common[g];                                               // :99-100 (ice)
        FORG Fvw[g] = fma(fma(-CST(a2), x2j[g], CST(a0)), S[g], fA) + common[g];       // (water)
        FORG wl[g] = fma(CST(m1), tw[g], CST(c_wl0));                                  // :71
        FORG rD[g] = ebm_rcp(sel1(noD[g], Do[g]));
        FORG an[g] = sel0(noD[g], pho[g] * (rD[g] * rD[g]));                           // alpha * n
        FORG n[g] = an[g] * CST(inv_alpha);                                            // num :84-85
        FORG Flat[g] = sel0(noD[g], (pho[g] * ho[g]) * (wl[g] * CST(c_flat)) * rD[g]); // :104-105
        FORG rEi[g] = fma(fma(pho[g], Fvi[g], Flat[g]), dt, Eio[g]);                   // :137,148,166
        FORG rEw[g] = fma(fma(om[g], Fvw[g], -Flat[g]), dt, Ewo[g]);                   // :138,148,167
        FORG { cEi[g] = rEi[g] > 0.0 ? 0.0 : rEi[g]; cEw[g] = rEw[g] < 0.0 ? 0.0 : rEw[g]; }   // redistributeE :110-111
        FORG psiEw_dt[g] = rEw[g] - cEw[g];
        FORG Ei_n[g] = cEi[g] + psiEw_dt[g];
        FORG Ew_n[g] = cEw[g] + (rEi[g] - cEi[g]);
        FORG ring[g] = an[g] * fma(CST(c_r1), Do[g], CST(c_r2));                       // area_lead :91
        FORG Al[g] = (ring[g] < om[g]) ? ring[g] : om[g];                              // :92
        FORG psiEw[g] = psiEw_dt[g] * ntd;                                             // psiEwdt / dt (:173)
        FORG Ql[g] = sel0(one[g], Al[g] * ROM(I) * psiEw[g]);                          // split_psiEw :121-122
        FORG dn[g] = -(psiEw[g] - Ql[g]) * CST(c_dn);                                  // :127,174
        FORG lat_grow[g] = sel0(noh[g], div_z(-Do[g], sel1(noh[g], CST(twoLf) * ho[g] * pho[g])) * Ql[g]);   // :142,144
        FORG Dt[g] = fma(CST(c_melt), wl[g], lat_grow[g]) + CST(c_weld) * pho[g] * (Do[g] * Do[g] * Do[g]);  // :141-145
        FORG rDn[g] = fma(Dt[g], dt, Do[g]);                                           // :175
        FORG total[g] = n[g] + dn[g];
        FORG tz[g] = is_zero(total[g]);
        FORG rt[g] = ebm_rcp(sel1(tz[g], total[g]));
        FORG Dn[g] = sel0(tz[g], fma(n[g], rDn[g], dn[g] * CST(Dmin)) * rt[g]);        // average :131-132
        FORG Dn[g] = sel(Dn[g] > CST(Dmax), CST(Dmax), sel(Dn[g] < CST(Dmin), CST(Dmin), Dn[g]));   // clamp (NaN stays NaN) :177
        FORG Dn[g] = sel0(is_zero(Ei_n[g]), Dn[g]);                                    // :178
        FORG rh[g] = fma(-Fvi[g], CST(dt_Lf), ho[g]);                                  // :139,179
        FORG rh[g] = rh[g] < 0.0 ? 0.0 : rh[g];                                        // :180
        FORG hn[g] = sel0(tz[g], fma(n[g], rh[g], dn[g] * CST(hmin)) * rt[g]);         // :181
        FORG hz[g] = is_zero(hn[g]);
        FORG r_hn[g] = ebm_rcp(sel1(hz[g], hn[g]));
        FORG RHP(I) = sel(hz[g], CST(inv_hmin), r_hn[g]);                              // next step's 1/hp (:51)
        FORG ph[g] = sel0(hz[g], -Ei_n[g] * r_hn[g] * CST(inv_Lf));                    // concentration :75-76
        FORG { if (ph[g] > 1.0) ph[g] = 1.0; }                                         // :77
        FORG Ei_n[g] = sel0(hz[g], Ei_n[g]);                                           // :185
        FORG omn[g] = 1 - ph[g];
        FORG En[g] = fma(ph[g], Ei_n[g], omn[g] * Ew_n[g]);                            // :186
        FORG Tn[g] = fma(Ti[I], ph[g], omn[g] * tw[g]);                                // :187
        FORG { EI(I) = Ei_n[g]; EW(I) = Ew_n[g]; DD(I) = Dn[g]; HH(I) = hn[g]; phi[I] = ph[g]; }

        // ---- sampling
        FORG {
        const int i = I;
        const int sidx = i * 32 + lane;
        const bool real = lane * K + i < nx;
        const double wj = tabs.wts[sidx];
        accT = fma(wj, Tn[g], accT); accE = fma(wj, En[g], accE); accP = fma(wj, ph[g], accP);
        icebits |= (unsigned)(ph[g] > 0.0 && real) << i;
        if (SLOW) {
        if (season == 0 || season == 1) {
          dgT = fma(wj, Tn[g], dgT); dgE = fma(wj, En[g], dgE); dgP = fma(wj, ph[g], dgP);
          if (ph[g] > 0.0 && real) dgX = fmin(dgX, xj[g]);
        } else if (season == 2) {
          if (((icebits >> i) & 1u) != 0u) dgX = fmin(dgX, xj[g]);
        }
        if (sel_m && real) {
          double v[EBM_MIZ_NVAR];
          v[EBM_MV_T] = Tn[g]; v[EBM_MV_Ei] = Ei_n[g];
          v[EBM_MV_Ti] = is_zero(Ei_n[g]) ? NAN : Ti[i];                              // :193
          v[EBM_MV_D] = Dn[g]; v[EBM_MV_n] = n[g]; v[EBM_MV_h] = hn[g]; v[EBM_MV_phi] = ph[g];
          v[EBM_MV_E] = En[g]; v[EBM_MV_Ew] = Ew_n[g];
          v[EBM_MV_Tw] = (ph[g] > 0.99) ? NAN : tw[g];                                // :194
          store_cell(a, lane * K + i, msel, year, ti, season, v);
        }
        }   // SLOW
        }
#undef FORG
#undef I
      }
      };    // cells
      if (sel_m || season >= 0) cells(std::true_type{}); else cells(std::false_type{});
      if (season >= 0 && a.diag != nullptr) {
        if (season == 2) {   // annual means: mean over the year of the hemispheric means (linear)
          dgT = accT / ntd; dgE = accE / ntd; dgP = accP / ntd;
        }
        const double t0 = ebm_warp_sum(dgT), t1 = ebm_warp_sum(dgE), t2 = ebm_warp_sum(dgP), t3 = ebm_warp_min(dgX);
        if (lane == 0) ebm_store_diag(a.diag, m, a.dur, year, season, t0, t1, t2, t3);
      }
      if (ti == nt) { accT = accE = accP = 0.0; icebits = 0u; }
    }
  }

  // ---- final state
  bool bad = false;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = lane * K + i;
    if (j < nx) {
      const long long o = (long long)j * nmem + m;
      const double ei = EI(i), ew = EW(i), dd = DD(i);
      a.Ei[o] = ei; a.Ew[o] = ew; a.h[o] = HH(i); a.D[o] = dd; a.phi[o] = phi[i]; a.T0[o] = T0[i];
      bad = bad || ebm_state_bad(ei) || ebm_state_bad(ew) || ebm_state_bad(HH(i)) || ebm_state_bad(dd) ||
            ebm_state_bad(phi[i]);
    }
  }
  bad = __any_sync(kFull, bad);
  if (lane == 0) {
    if (a.newton_iters != nullptr) a.newton_iters[m] += iters_total;
    if (a.nonconv != nullptr) a.nonconv[m] += fails_total;
    if (bad && a.flags != nullptr) a.flags[m] |= 1;
  }
}

template <int K, int MINB>
int launch_k(const MizKArgs& a, cudaStream_t stream) {
  const long long blocks = (a.nmem + kWarps - 1) / kWarps;
  if (blocks > 0x7fffffffLL) { ebm_set_error("miz: too many members (%lld)", a.nmem); return EBM_ERR_INVALID; }
  auto kern = miz_fast_kernel<K, MINB>;
  EBM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Tabs<K>)));
  EBM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  kern<<<(unsigned)blocks, kWarps * 32, sizeof(Tabs<K>), stream>>>(a);
  EBM_CUDA_TRY(cudaGetLastError());
  ebm_count_launch();
  return EBM_OK;
}

}  // namespace

int ebm_launch_miz_fast(const MizKArgs& a, cudaStream_t stream) {
  if (a.nx < 3) { ebm_set_error("miz: nx must be >= 3"); return EBM_ERR_INVALID; }
  if (a.nx <= 64) return launch_k<2, 4>(a, stream);
  if (a.nx <= 128) return launch_k<4, 4>(a, stream);
  if (a.nx <= 192) return launch_k<6, 3>(a, stream);   // 3 resident CTAs per SM (168 registers): fastest measured
  if (a.nx <= 256) return launch_k<8, 2>(a, stream);
  ebm_set_error("miz: nx=%d > 256 not supported by the register-resident kernel", a.nx);
  return EBM_ERR_UNSUPPORTED;
}

int ebm_launch_miz(const MizKArgs& a, int strict, cudaStream_t stream) {
  return strict ? ebm_launch_miz_strict(a, stream) : ebm_launch_miz_fast(a, stream);
}

// step!(Val(:MIZ), ...) for one member (src/miz.jl:150-196) with the literal-order kernel: the ten stored
// variables of the step go to vars_out [EBM_MIZ_NVAR][nx]; state and the closure warm start are updated in place.
int ebm_launch_miz_single_step(const EbmGridTables& g, const double* par22, int ti, double f, double tol, int maxit,
                               double* Ei, double* Ew, double* h, double* D, double* phi, double* T0,
                               double* vars_out, long long* iters, cudaStream_t stream) {
  MizKArgs a;
  memset(&a, 0, sizeof(a));
  a.nx = g.nx; a.nt = g.nt; a.dur = 1; a.nmem = 1; a.year0 = 0; a.nyears = 1;
  a.winter_inx = -1; a.summer_inx = -1; a.lastonly = 1; a.field_stride = 1;
  a.maxit = maxit; a.tol = tol; a.single_ti = ti; a.single_f = f;
  a.g = g; a.par = par22; a.forc = nullptr;
  a.Ei = Ei; a.Ew = Ew; a.h = h; a.D = D; a.phi = phi; a.T0 = T0;
  a.raw = vars_out; a.newton_iters = iters;
  return ebm_launch_miz_strict(a, stream);
}
