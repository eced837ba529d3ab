// classic_uniform.cu -- the classic (Wagner-Eisenman) EBM ensemble kernel for grids up to 208 cells.
//
// TAB = true integrates the 32-member groups whose table-building parameters (D, cg, tau, S0, S2, a0, a2) agree --
// forcing sweeps, hysteresis runs, sweeps over A, B, cw, S1, ai, Fb, k, Lf; TAB = false the groups where they differ
// (coefficients applied per member, no precomputed pivots).  UPAR = true (with TAB) takes a launch in which every
// member has the same 15 parameters (the C4 forcing sweep).  Five instances: TAB, !TAB and UPAR with 8 bands for
// nx <= 104, TAB and !TAB with 16 bands (255 registers, 1 CTA per SM) for 104 < nx <= 208.
//
// Mapping (B200 facts measured with scripts/microbench/fp64_lat.cu: DFMA latency 8.8 cycles, one warp can issue
// a DFMA every 2.4 cycles, the 64 KB register file of an SM sub-partition holds 3 warps at <=168 registers):
//   * lane = member, warp = 2 latitude bands of K = 13 cells for 16 members; CTA = 16 members x WB = 8 bands =
//     4 warps, one per SM sub-partition; 3 CTAs per SM (168 registers; 74.9 KB of shared memory per CTA).
//     E and Tg of every cell stay in registers for the whole launch.  (Measured and rejected: all bands of a
//     member in one warp, 4 bands per warp, 16 bands of 7 cells -- band-homogeneous warps win, DESIGN.md 4.1.)
//   * every latitude-dependent coefficient (S0-S2x^2, x, a0-a2x^2, kappa) is a CTA-wide table in shared memory,
//     read with broadcast 128-bit loads.
//   * physics per cell with selects; the one branch is per thread: "all my cells are open water" (9 FP64
//     instructions per cell) or not.  1/(M - kLf/E) of every cell is carried from step to step.
//   * implicit ghost-layer solve (classic.jl:55-63; symmetric tridiagonal, diagonal depends on the member's
//     ice mask): partitioned.  Rows whose diagonal is the constant kappa_jj -- open water, or ice with a melting
//     surface, i.e. mask (T0<0)&(E<0) false -- have member-independent pivots: a band without masked rows uses
//     elimination tables precomputed once per launch (5 FP64 instructions per row); a band with masked rows
//     eliminates in full with determinant-form pivots (one dependent DFMA per row, independent reciprocals).
//     The WB x WB interface system is solved by warp 0 from both ends at once, entirely in registers.
//     Two CTA barriers per step.
//   * what survives from elimination to back substitution (pivots, spikes), the carried reciprocals and the
//     per-cell annual sums of E live in thread-private shared memory [row][thread] (conflict free).
//   * the hot step carries no sampling code; steps that store output and CTAs that own a member with field
//     output take a second instantiation.  Annual mean of T: one scalar per thread (hemispheric mean is linear);
//     per-cell sums of T and h only in CTAs that write fields.
// Citations: src/classic.jl:43-65 (step), src/infrastructure.jl:549-591 (savesol!), SURVEY.md Appendix A.
#include "ebm_internal.cuh"

#ifdef EBM_PHASE_TIMING
// dev instrumentation: cycles spent by each warp of CTA 0 between the marks of a step, summed over the launch
__device__ unsigned long long g_phase_cycles[8][8];
#define PHASE_MARK(k)                                                                         \
  do {                                                                                        \
    const long long _now = clock64();                                                         \
    if (blockIdx.x == 0 && (threadIdx.x & 31) == 0)                                           \
      atomicAdd(&g_phase_cycles[k][threadIdx.x >> 5], (unsigned long long)(_now - phase_t));  \
    phase_t = _now;                                                                           \
  } while (0)
#define PHASE_BEGIN() long long phase_t = clock64()
#else
#define PHASE_MARK(k) do { } while (0)
#define PHASE_BEGIN() do { } while (0)
#endif

namespace {

// sign test on the high word (integer pipe, not the FP64 pipe).  The state never holds -0.0: it is normalised when
// loaded, and E + dt*(...) cannot produce it (an exact cancellation rounds to +0.0).
__device__ __forceinline__ bool is_neg(double v) { return __double2hiint(v) < 0; }
// (miz_kernel.cu's is_zero, the same predicate in another form, changes the code of every instance: -46 to -168 instructions)
__device__ __forceinline__ bool is_zero(double v) { return ((__double2hiint(v) << 1) | __double2loint(v)) == 0; }

struct __align__(16) PhysTab { double S0x, S1x, aw, wts; };      // per cell
struct __align__(16) ElimTab { double iw, tq, q, s; };           // per row: band-local no-mask elimination
struct __align__(16) CoefTab { double kjj, aoff, coff, ac; };    // per cell, masked path: ac = aoff_j * coff_{j-1} (0 on a band's first row)

// rows of the band system that survive from the elimination to the back substitution, in thread-private shared
// memory [3K][threads] (conflict free), which frees 6K registers for more resident CTAs (DESIGN.md 4.1)
template <int K>
struct RowStore {
  double* base;
  int stride;
  // r(i) = E_i / (M E_i - kLf) = 1/(M - kLf/E_i) of the cell's CURRENT enthalpy, carried from step to step: this
  // step's T0 = C/(M - kLf/E) (classic.jl:50) is C*r of the previous step's update (:56-62 computes it anyway)
  __device__ __forceinline__ double& r(int i) { return base[(2 * K + i) * stride]; }
  __device__ __forceinline__ double& q(int i) { return base[(2 * i) * stride]; }
  __device__ __forceinline__ double& s(int i) { return base[(2 * i + 1) * stride]; }
};

template <int K, int WB, int MW, bool TAB, bool UPAR>
struct Ctx {
  static constexpr int NXP = K * WB;
  // tables / scratch in shared memory
  const PhysTab* phys; const ElimTab* elim; const CoefTab* coef; const double* bandc;
  double *iface, *zs, *red, *sumT, *sumH;
  // TAB = false (groups whose table-building parameters differ between members): the shared tables hold geometry
  // only and every thread applies its own member's S0, S2, a0, a2 and fac = dt*D/cg on the fly; all rows take the
  // general elimination (no precomputed pivots)
  double S0m, S2m, a0m, a2m, facm, fac2m, one_dttaum;
  __device__ __forceinline__ PhysTab phys_at(int j) const {
    PhysTab p = phys[j];
    if constexpr (!TAB) { p.S0x = fma(-S2m, p.S0x, S0m); p.aw = fma(-a2m, p.aw, a0m); }   // the table holds x^2 in both slots
    return p;
  }
  __device__ __forceinline__ CoefTab coef_at(int j) const {
    CoefTab c = coef[j];
    if constexpr (!TAB) {   // the table holds lam_lo + lam_hi, lam_lo, lam_hi, lam_lo_j * lam_hi_{j-1}
      c.kjj = fma(facm, c.kjj, one_dttaum); c.aoff = -facm * c.aoff; c.coff = -facm * c.coff; c.ac = fac2m * c.ac;
    }
    return c;
  }
  // member constants
  // (UPAR: every member of the launch has the same 15 parameters -- the constants below are then read from the kernel
  // argument block, i.e. they are constant-bank operands of the FP64 instructions instead of 26 live registers)
  double A_, Fb_, ai_, cg_tau_, M_, kLf_, inv_cw_, dt_, dt_tau_, dttau_cw_, dc_, inv_nt_, inv_Lf_;
#define EBM_MEMBER_CONSTS(a)                                                                                        \
  const double A = UPAR ? (a).u.A : A_, Fb = UPAR ? (a).u.Fb : Fb_, ai = UPAR ? (a).u.ai : ai_,                     \
               cg_tau = UPAR ? (a).u.cg_tau : cg_tau_, M = UPAR ? (a).u.M : M_, kLf = UPAR ? (a).u.kLf : kLf_,      \
               inv_cw = UPAR ? (a).u.inv_cw : inv_cw_, dt = UPAR ? (a).u.dt : dt_,                                  \
               dt_tau = UPAR ? (a).u.dt_tau : dt_tau_, dttau_cw = UPAR ? (a).u.dttau_cw : dttau_cw_,                \
               dc = UPAR ? (a).u.dc : dc_, inv_nt = UPAR ? (a).u.inv_nt : inv_nt_,                                  \
               inv_Lf = UPAR ? (a).u.inv_Lf : inv_Lf_;                                                              \
  (void)A; (void)Fb; (void)ai; (void)cg_tau; (void)M; (void)kLf; (void)inv_cw; (void)dt; (void)dt_tau;              \
  (void)dttau_cw; (void)dc; (void)inv_nt; (void)inv_Lf
  // thread identity
  int band, mi, j0;
  // index of cell i of this thread in the per-cell shared arrays (annual sums): [cell][member]
  __device__ __forceinline__ int cidx(int i) const { return (j0 + i) * MW + mi; }
  bool active, sel, cta_fields;
  bool solver;   // this warp solves the CTA's interface systems (the warp that owns band pair 1: never the polar pair)
  // original member index of this thread's member (output rows, field selection): recomputed where it is needed (the
  // three sampling steps of a year) instead of being kept in registers through the hot loop
  __device__ __forceinline__ long long member_orig(const ClassicKArgs& a) const {
    long long m = ((long long)(blockIdx.x + (unsigned)a.block0)) * MW + mi;
    if (m >= a.nmem) m = a.nmem - 1;
    return a.orig != nullptr ? a.orig[m] : m;
  }
  // state
  double E[K], Tg[K], accT;
  RowStore<K> rs;
  double* sumE;   // [NXP][MW] running annual sum of E per cell (shared memory: keeps 2K registers free)

  // annual sums and (SLOW only) sampled output of cell i after its update: savesol! (infrastructure.jl:549-591)
  template <bool SLOW>
  __device__ __forceinline__ void sample(const ClassicKArgs& a, const int i, const double wj, const double En,
                                         const double T, const int season, const int ti, const int year,
                                         double& se, double& dgT, double& dgE, double& dgA, double& dgX) {
    EBM_MEMBER_CONSTS(a);
    se += En;                                   // running annual sum of E of this cell (caller loads / stores it)
    const double sEi = se;
    accT = fma(wj, T, accT);
    if (SLOW) {
      const int nx = a.nx, nt = a.nt;
      const int j = j0 + i;
      const int sidx = cidx(i);
      const double Eneg = is_neg(En) ? En : 0.0;
      if (cta_fields) { sumT[sidx] += T; sumH[sidx] += Eneg; }
      const bool rawstep = sel && a.raw != nullptr && (!a.lastonly || year == a.dur - 1);   // not ebm_raw_year: -93 to +84 instr.
      if (rawstep && j < nx) {
        const long long nraw = ebm_nraw(nt, a.dur, a.lastonly);   // (this order of loads keeps the code)
        const long long slot = ebm_raw_slot(year, ti, nt, a.lastonly);
        const long long msel = ebm_field_row(a, member_orig(a));
        double* o = a.raw + ebm_raw_offset(msel, nraw, slot, EBM_CLASSIC_NVAR, nx) + j;
        o[0] = En; o[nx] = T; o[2 * nx] = -Eneg * inv_Lf;          // h = -E/Lf*(E<0)  (classic.jl:65)
      }
      if (season >= 0) {
        double vT = T, vE = En, vN = Eneg;
        if (season == 2) {                                          // annual mean (infrastructure.jl:583-588)
          vE = sEi * inv_nt;
          if (cta_fields) { vT = sumT[sidx] * inv_nt; vN = sumH[sidx] * inv_nt; }
        }
        dgT = fma(wj, vT, dgT);
        dgE = fma(wj, vE, dgE);
        if (vE < 0.0 && j < nx) { dgA += wj; dgX = fmin(dgX, phys[j].S1x); }
        if (sel && a.seasonal != nullptr && j < nx) {
          const long long msel = ebm_field_row(a, member_orig(a));
          double* o = a.seasonal + ebm_seasonal_offset(msel, a.dur, year, season, EBM_CLASSIC_NVAR, nx) + j;
          o[0] = vE; o[nx] = vT; o[2 * nx] = -vN * inv_Lf;
        }
      }
      if (ti == nt) {
        se = 0.0;
        if (cta_fields) { sumT[sidx] = 0.0; sumH[sidx] = 0.0; }
      }
    }
  }

  // Pad cells (a band's cells beyond nx; decoupled rows of weight 0) follow the band's real cells: ice when every one
  // of them is ice at the turn of the year, open water otherwise -- so that they do not decide which code path the band takes (a snowball's polar band
  // would otherwise run the mixed ice / water code for its pad cells alone and hold the CTA's other warps at the
  // barrier).  Their tables (TAB) make both states self-sustaining over a year.  Called at launch and at the end of every
  // year, and it resets the pad cells unconditionally: their state, hence the code path of every step, is a function of
  // the real cells' state at the last year boundary -- launches split at year boundaries stay bit-identical.
  __device__ __forceinline__ void set_pads(const ClassicKArgs& a) {
    EBM_MEMBER_CONSTS(a);
    const int nv = a.nx - j0;
    if (TAB && nv < K && nv > 0) {
      int hand = -1;
#pragma unroll
      for (int i = 0; i < K; ++i) if (i < nv) hand &= __double2hiint(E[i]);
      const bool wantice = hand < 0;
#pragma unroll
      for (int i = 0; i < K; ++i) {
        if (i >= nv) {
          E[i] = wantice ? -10.0 : 100.0; Tg[i] = wantice ? -10.0 : 10.0;
          rs.r(i) = E[i] * ebm_rcp(fma(M, E[i], -kLf));
        }
      }
    }
  }

  static constexpr int GI = UPAR ? 5 : 3;    // cells per statement-major group: all-ice path
  static constexpr int GIM = UPAR ? 4 : 3;   // mixed ice / water path
  template <int I0, bool MIXED, bool SLOW>
  __device__ __forceinline__ void ice_group(const ClassicKArgs& a, const double fmA, const double S1c0, const double S1c1,
                                            const int season, const int ti, const int year, bool& anymask,
                                            double& dgT, double& dgE, double& dgA, double& dgX) {
    EBM_MEMBER_CONSTS(a);
    constexpr int GG = MIXED ? GIM : GI;
    constexpr int N = (I0 + GG <= K) ? GG : K - I0;
    PhysTab p[N]; double rv[N], se[N];
#pragma unroll
    for (int g = 0; g < N; ++g) { p[g] = phys_at(j0 + I0 + g); rv[g] = rs.r(I0 + g); se[g] = sumE[cidx(I0 + g)]; }
    double S[N], C[N], T[N], En[N], r[N], um[N], G[N];
    int ice[N], tneg[N];   // 0 / -1
#pragma unroll
    for (int g = 0; g < N; ++g) S[g] = fma(-S1c0, p[g].S1x, p[g].S0x);                       // S[j,i]
#pragma unroll
    for (int g = 0; g < N; ++g) C[g] = fma(cg_tau, Tg[I0 + g], fmA);
#pragma unroll
    for (int g = 0; g < N; ++g) {
      if constexpr (MIXED) {
        ice[g] = __double2hiint(E[I0 + g]) >> 31;
        const double al = ice[g] ? ai : (is_zero(E[I0 + g]) ? 0.0 : p[g].aw);               // alpha                  :47
        C[g] = fma(al, S[g], C[g]);                                                         //                        :48
      } else {   // every cell of the band is ice (same bits as the general code)
        C[g] = fma(ai, S[g], C[g]);
      }
    }
#pragma unroll
    for (int g = 0; g < N; ++g) G[g] = fma(-S1c1, p[g].S1x, p[g].S0x);                       // S[j,i+1]
#pragma unroll
    for (int g = 0; g < N; ++g) T[g] = C[g] * rv[g];                                          // T0 = C/(M - kLf/E)     :50
#pragma unroll
    for (int g = 0; g < N; ++g) G[g] = fma(ai, G[g], fmA);
#pragma unroll
    for (int g = 0; g < N; ++g) {
      const int cneg = __double2hiint(C[g]) >> 31;              // for E < 0: M - kLf/E > 0, so T0 < 0 <=> C < 0
      if constexpr (MIXED) {
        // T = E/cw [E >= 0] + T0 [E < 0 and T0 < 0]                                              :51
        // (the sign of T0 of a water cell matters only if the cell freezes in this step: fix-up below)
        tneg[g] = ice[g] & cneg;
        const double Tw = E[I0 + g] * inv_cw;
        T[g] = __hiloint2double((__double2hiint(T[g]) & tneg[g]) | (__double2hiint(Tw) & ~ice[g]),
                                (__double2loint(T[g]) & tneg[g]) | (__double2loint(Tw) & ~ice[g]));
      } else {
        tneg[g] = cneg;
        T[g] = __hiloint2double(__double2hiint(T[g]) & cneg, __double2loint(T[g]) & cneg);
      }
    }
#pragma unroll
    for (int g = 0; g < N; ++g) En[g] = fma(-M, T[g], C[g]);
#pragma unroll
    for (int g = 0; g < N; ++g) En[g] = En[g] + Fb;
#pragma unroll
    for (int g = 0; g < N; ++g) En[g] = fma(dt, En[g], E[I0 + g]);                           //                        :53
#pragma unroll
    for (int g = 0; g < N; ++g) r[g] = fma(M, En[g], -kLf);
    {
      double x[N], e[N];
#pragma unroll
      for (int g = 0; g < N; ++g) asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x[g]) : "d"(r[g]));
#pragma unroll
      for (int g = 0; g < N; ++g) e[g] = fma(-r[g], x[g], 1.0);
#pragma unroll
      for (int g = 0; g < N; ++g) e[g] = fma(e[g], e[g], e[g]);
#pragma unroll
      for (int g = 0; g < N; ++g) x[g] = fma(x[g], e[g], x[g]);
#pragma unroll
      for (int g = 0; g < N; ++g) r[g] = En[g] * x[g];                                        // 1/(M - kLf/E), E updated
    }
#pragma unroll
    for (int g = 0; g < N; ++g) um[g] = dt_tau * r[g];
#pragma unroll
    for (int g = 0; g < N; ++g) {
      const int mk = tneg[g] & (__double2hiint(En[g]) >> 31);                                 // (T0<0) & (E<0)      :56,61
      anymask = anymask || (mk != 0);
      um[g] = __hiloint2double(__double2hiint(um[g]) & mk, __double2loint(um[g]) & mk);
    }
#pragma unroll
    for (int g = 0; g < N; ++g) {
      const int pm = ~(__double2hiint(En[g]) >> 31);
      const double Ep = __hiloint2double(__double2hiint(En[g]) & pm, __double2loint(En[g]) & pm);   // E [E >= 0]   :59
      S[g] = fma(dttau_cw, Ep, Tg[I0 + g]);
    }
#pragma unroll
    for (int g = 0; g < N; ++g) Tg[I0 + g] = fma(um[g], G[g], S[g]);                          // right-hand side     :58-62
    if constexpr (MIXED) {
      // a water cell that froze in this step (rare): its row is masked if T0 = C/(M - kLf/E) of the OLD enthalpy E > 0
      // was negative, i.e. C != 0 and sign(C) != sign(M E - kLf)                                :50,56,61
      int frz = 0;
#pragma unroll
      for (int g = 0; g < N; ++g) frz |= ~ice[g] & __double2hiint(En[g]);
      if (frz < 0) {
#pragma unroll
        for (int g = 0; g < N; ++g) {
          const double Eo = E[I0 + g];
          if (!ice[g] && is_neg(En[g]) && !is_zero(Eo) && C[g] != 0.0 && (is_neg(C[g]) != is_neg(fma(M, Eo, -kLf)))) {
            um[g] = dt_tau * r[g];
            Tg[I0 + g] = fma(um[g], G[g], S[g]);
            anymask = true;
          }
        }
      }
    }
#pragma unroll
    for (int g = 0; g < N; ++g) {
      sample<SLOW>(a, I0 + g, p[g].wts, En[g], T[g], season, ti, year, se[g], dgT, dgE, dgA, dgX);
      E[I0 + g] = En[g];
    }
#pragma unroll
    for (int g = 0; g < N; ++g) {
      rs.r(I0 + g) = r[g]; rs.q(I0 + g) = um[g];                // dt_tau/(M - kLf/E) [masked]; times cg_tau in the pivots :56
      sumE[cidx(I0 + g)] = se[g];
    }
  }
  template <int I0, bool MIXED, bool SLOW>
  __device__ __forceinline__ void ice_groups(const ClassicKArgs& a, const double fmA, const double S1c0, const double S1c1,
                                             const int season, const int ti, const int year, bool& anymask,
                                             double& dgT, double& dgE, double& dgA, double& dgX) {
    if constexpr (I0 < K) {
      ice_group<I0, MIXED, SLOW>(a, fmA, S1c0, S1c1, season, ti, year, anymask, dgT, dgE, dgA, dgX);
      ice_groups<I0 + (MIXED ? GIM : GI), MIXED, SLOW>(a, fmA, S1c0, S1c1, season, ti, year, anymask, dgT, dgE, dgA, dgX);
    }
  }

  template <bool SLOW>
  __device__ __forceinline__ void step(const ClassicKArgs& a, const double f, const double S1c0, const double S1c1,
                                       const int ti, const int year) {
    EBM_MEMBER_CONSTS(a);
    const int tid = threadIdx.x;
    const int nx = a.nx, nt = a.nt;
    const double fmA = f - A;
    const double fmAFb = fmA + Fb;
    const int season = SLOW ? ebm_season(a, ti, nt) : -1;
    // rs.q(i): dt_tau/(M - kLf/E) of a masked row (else 0): the diagonal decrement over cg_tau; later the pivots / spikes
    bool anymask = !TAB;   // without precomputed pivots every band eliminates in full
    PHASE_BEGIN();
    double dgT = 0.0, dgE = 0.0, dgA = 0.0, dgX = 2.0;

    // ---- physics (classic.jl:47-53) and the rows of the implicit system (:55-63)
    // One code path per warp (a warp whose lanes disagree would run both, one after the other): the open-water code
    // below only if no lane holds an ice cell or a cell about to freeze (E < 512 dt, a.hthr: signed compare of the high
    // words -- |dE| per step is ~dt * 300), else the ice code for every lane.  Both give the same bits for an open-water cell
    // that stays open water, so the result does not depend on which members share a warp.
    int hmin = 0x7fffffff;
#pragma unroll
    for (int i = 0; i < K; ++i) hmin = min(hmin, __double2hiint(E[i]));
    const bool has_ice = __any_sync(0xffffffffu, hmin < a.hthr);
    if (!has_ice) {
      bool crossed = false;
      double se[K];                                         // annual sums: loaded up front, stored after the loop, so
#pragma unroll                                              // that the K cells overlap instead of serialising on smem
      for (int i = 0; i < K; ++i) se[i] = sumE[cidx(i)];
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const PhysTab p = phys_at(j0 + i);
        const double S = fma(-S1c0, p.S1x, p.S0x);          // S[j,i]; S1x holds x_j, S0x = S0 - S2 x_j^2
        const double Eo = E[i], Tgo = Tg[i];
        const double alpha = is_zero(Eo) ? 0.0 : p.aw;      // alpha = aw, or 0 at E == 0                 :47
        const double C = fma(alpha, S, fma(cg_tau, Tgo, fmA));                                    //     :48
        const double T = Eo * inv_cw;                                                             //     :51
        const double En = fma(dt, fma(-M, T, C) + Fb, Eo);          // (operation order of ice_group)   :53
        E[i] = En;
        Tg[i] = fma(dttau_cw, En, Tgo);
        if constexpr (!TAB) rs.q(i) = 0.0;
        crossed = crossed || is_neg(En);
        sample<SLOW>(a, i, p.wts, En, T, season, ti, year, se[i], dgT, dgE, dgA, dgX);
      }
#pragma unroll
      for (int i = 0; i < K; ++i) sumE[cidx(i)] = se[i];
      if (crossed) {   // freeze-up of a cell with E >= 512 dt inside one step (a tendency beyond 512 W/m^2: safety net): literal mask
#pragma unroll
        for (int i = 0; i < K; ++i) rs.q(i) = 0.0;
#pragma unroll
        for (int i = 0; i < K; ++i) {
          const double En = E[i];
          if (is_neg(En)) {
            // recover the old state of this cell from the update formulas (only the sign of T0 is needed)
            const PhysTab p = phys_at(j0 + i);
            const double Tgo = fma(-dttau_cw, En, Tg[i]);
            const double Cb = fma(p.aw, fma(-S1c0, p.S1x, p.S0x), fma(cg_tau, Tgo, fmAFb));
            const double Eo = fma(-dt, Cb, En) / fma(-dt * M, inv_cw, 1.0);
            const double C = Cb - Fb;
            const double T0 = C / (M - kLf / Eo);                                                 //     :50
            const double r = En * ebm_rcp(fma(M, En, -kLf));
            rs.r(i) = r;
            if (T0 < 0.0) {
              rs.q(i) = dt_tau * r; anymask = true;
              Tg[i] = fma(dt_tau * r, fma(ai, fma(-S1c1, p.S1x, p.S0x), fmA), Tgo);
            } else {
              Tg[i] = Tgo;
            }
          }
        }
      }
    } else {
      // ptxas keeps the source order to a large extent and a warp issues in order: written cell after cell, the
      // cells' dependent chains (C -> T0 -> E' -> reciprocal -> right-hand side, ~16 FP64 instructions deep) run one
      // after the other.  Statement-major over groups of 4 cells gives the warp 4 independent chains; the masks of
      // classic.jl:47-61 are bit masks / selects on operands, no branches.
      // all-ice specialisation (no alpha / T selects) when no thread of the warp needs the general code; both give
      // the same bits for an all-ice band, so the vote does not influence any result
      bool allice = true;
#pragma unroll
      for (int i = 0; i < K; ++i) allice = allice && is_neg(E[i]);
      if (__all_sync(__activemask(), allice)) ice_groups<0, false, SLOW>(a, fmA, S1c0, S1c1, season, ti, year, anymask, dgT, dgE, dgA, dgX);
      else ice_groups<0, true, SLOW>(a, fmA, S1c0, S1c1, season, ti, year, anymask, dgT, dgE, dgA, dgX);
    }
    if (SLOW && season == 2) dgT = accT * inv_nt;   // mean over the year of the hemispheric mean (linear)
    if (SLOW && ti == nt) accT = 0.0;

    PHASE_MARK(0);   // physics
    // ---- local elimination  x_i + q_i x_{i+1} + s_i xL = y_i  and reduction of row 0 to (al, be, ga)
    double i_sl, i_ql, i_yl, i_al, i_be, i_ga;   // this band's interface row (last row + row 0 reduced)
    if (!anymask) {
      // member-independent pivots (precomputed): only the right-hand side is eliminated
      double yprev = 0.0;
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const ElimTab e = elim[j0 + i];
        const double yi = fma(-e.tq, yprev, Tg[i] * e.iw);
        Tg[i] = yi; yprev = yi;
      }
      double al = Tg[K - 2];
#pragma unroll
      for (int i = K - 3; i >= 0; --i) al = fma(-elim[j0 + i].q, al, Tg[i]);
      const ElimTab el = elim[j0 + K - 1];
      i_sl = el.s; i_ql = el.q; i_yl = Tg[K - 1];
      i_al = al; i_be = bandc[2 * band]; i_ga = bandc[2 * band + 1];
    } else {
      // pivots in determinant form: P_i = w_0 ... w_i obeys P_i = d_i P_{i-1} - (a_i c_{i-1}) P_{i-2}, one dependent FMA
      // per row; the K reciprocals 1/w_i = P_{i-1}/P_i are then independent of each other (|w| ~ 50..250: no overflow)
      double Pm2 = 1.0, Pm1 = 1.0;
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const CoefTab cf = coef_at(j0 + i);
        const double diag = fma(-cg_tau, rs.q(i), cf.kjj);      // kappa_jj - dc/(M - kLf/E) [masked]   :56
        const double P = (i == 0) ? diag : fma(diag, Pm1, -(cf.ac * Pm2));
        rs.s(i) = Pm1 * ebm_rcp(P);            // 1 / w_i
        Pm2 = Pm1; Pm1 = P;
      }
      double yprev = 0.0, sprev = 0.0;
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const CoefTab cf = coef_at(j0 + i);
        const double iw = rs.s(i);
        const double tq = cf.aoff * iw;
        const double yi = (i == 0) ? Tg[i] * iw : fma(-tq, yprev, Tg[i] * iw);
        const double si = (i == 0) ? tq : -tq * sprev;
        rs.q(i) = cf.coff * iw; rs.s(i) = si; Tg[i] = yi;
        yprev = yi; sprev = si;
      }
      double al = Tg[K - 2], be = rs.s(K - 2), ga = rs.q(K - 2);
#pragma unroll
      for (int i = K - 3; i >= 0; --i) {
        al = fma(-rs.q(i), al, Tg[i]);
        be = fma(-rs.q(i), be, rs.s(i));
        ga = -rs.q(i) * ga;
      }
      i_sl = rs.s(K - 1); i_ql = rs.q(K - 1); i_yl = Tg[K - 1];
      i_al = al; i_be = be; i_ga = ga;
    }
    {
      double* f6 = iface + (band * 6) * MW + mi;
      f6[0 * MW] = i_sl; f6[1 * MW] = i_ql; f6[2 * MW] = i_yl; f6[3 * MW] = i_al; f6[4 * MW] = i_be; f6[5 * MW] = i_ga;
    }
    if (SLOW && season >= 0) {
      double* r4 = red + (band * 4) * MW + mi;
      r4[0 * MW] = dgT; r4[1 * MW] = dgE; r4[2 * MW] = dgA; r4[3 * MW] = dgX;
    }
    PHASE_MARK(1);   // elimination + reduction
    __syncthreads();
    PHASE_MARK(2);   // barrier 1 wait
    // ---- interface system: WB unknowns per member.  One warp solves it with two lanes per member working from
    // both ends towards the middle ("burn at both ends"), pivots carried as determinants D_k so that the
    // only dependent chain is one DFMA per row; all reciprocals are independent of each other.
    if (solver) {
      constexpr int H = WB / 2;
      const int half = (tid & 31) / MW;                      // 0: rows 0..H-1 downwards, 1: rows WB-1..H upwards
      double a_[H], d_[H], c_[H], r_[H];
#pragma unroll
      for (int k = 0; k < H; ++k) {
        const int b = half ? (WB - 1 - k) : k;
        const double* g6 = iface + (b * 6) * MW + mi;
        const double* n6 = g6 + 6 * MW;                      // band b+1 (a zero band follows the last one)
        const double sl = g6[0 * MW], ql = g6[1 * MW], yl = g6[2 * MW];
        const double dg = fma(-ql, n6[4 * MW], 1.0), sup = -ql * n6[5 * MW];
        r_[k] = fma(-ql, n6[3 * MW], yl);
        d_[k] = dg;
        a_[k] = half ? sup : sl;                             // coupling to the previously eliminated row
        c_[k] = half ? sl : sup;                             // coupling to the next row in sweep order
      }
      double Dm[H + 1];                                      // Dm[k+1] = D_k, Dm[0] = D_{-1} = 1
      Dm[0] = 1.0; Dm[1] = d_[0];
#pragma unroll
      for (int k = 1; k < H; ++k) Dm[k + 1] = fma(d_[k], Dm[k], -(a_[k] * c_[k - 1]) * Dm[k - 1]);
      double cq[H], cy[H];
#pragma unroll
      for (int k = 0; k < H; ++k) {
        const double iw = Dm[k] * ebm_rcp(Dm[k + 1]);
        cq[k] = c_[k] * iw;
        const double g = a_[k] * iw, ri = r_[k] * iw;
        cy[k] = (k == 0) ? ri : fma(-g, cy[k - 1], ri);
      }
      // the two sweeps meet between rows H-1 and H:  x_own = cy_own - cq_own * x_other
      const double ocq = __shfl_xor_sync(0xffffffffu, cq[H - 1], MW);
      const double ocy = __shfl_xor_sync(0xffffffffu, cy[H - 1], MW);
      double x = fma(-cq[H - 1], ocy, cy[H - 1]) * ebm_rcp(fma(-cq[H - 1], ocq, 1.0));
      zs[(half ? (WB - H) : (H - 1)) * MW + mi] = x;
#pragma unroll
      for (int k = H - 2; k >= 0; --k) {
        x = fma(-cq[k], x, cy[k]);
        zs[(half ? (WB - 1 - k) : k) * MW + mi] = x;
      }
      if (SLOW && season >= 0 && a.diag != nullptr && active && half == 0) {
        double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 2.0;
        for (int b = 0; b < WB; ++b) {
          const double* r4 = red + (b * 4) * MW + mi;
          t1 += r4[1 * MW]; t2 += r4[2 * MW]; t3 = fmin(t3, r4[3 * MW]);
          t0 += r4[0 * MW];
        }
        ebm_store_diag(a.diag, member_orig(a), a.dur, year, season, t0, t1, t2, t3);
      }
    }
    PHASE_MARK(3);   // interface solve (warp 0) / nothing
    __syncthreads();
    PHASE_MARK(4);   // barrier 2 wait
    // ---- back substitution with the true neighbours
    const double xL = (band > 0) ? zs[(band - 1) * MW + mi] : 0.0;
    double xn = zs[band * MW + mi];
    Tg[K - 1] = xn;
    if (!anymask) {
#pragma unroll
      for (int i = K - 2; i >= 0; --i) {
        const ElimTab e = elim[j0 + i];
        xn = fma(-e.q, xn, fma(-e.s, xL, Tg[i]));
        Tg[i] = xn;
      }
    } else {
#pragma unroll
      for (int i = K - 2; i >= 0; --i) {
        xn = fma(-rs.q(i), xn, fma(-rs.s(i), xL, Tg[i]));
        Tg[i] = xn;
      }
    }
    PHASE_MARK(5);   // back substitution
    if (SLOW && ti == nt) set_pads(a);
  }
};

template <int K, int WB, int MW>
constexpr size_t uniform_smem_bytes(bool fields) {
  return (size_t)K * WB * (sizeof(PhysTab) + sizeof(ElimTab) + sizeof(CoefTab)) +
         sizeof(double) * ((size_t)2 * WB + (size_t)(WB + 1) * 6 * MW + (size_t)WB * MW * (1 + 4) + 10 * MW +
                           (size_t)K * WB * MW + (fields ? (size_t)2 * K * WB * MW : 0) + (size_t)3 * K * WB * MW);
}

template <int K, int WB, int MW, int MAXR, bool TAB, bool UPAR>
__global__ void __maxnreg__(MAXR) classic_uniform_kernel(const __grid_constant__ ClassicKArgs a) {
  static_assert(!UPAR || TAB, "launch-uniform parameters imply uniform tables");
  static_assert(MW == 16, "warp 0 = two lanes per member (full-warp shuffles)");
  static_assert(WB % 2 == 0 && (WB * MW) % 32 == 0, "whole warps, even band count");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int BPW = 32 / MW;
  constexpr int NXP = K * WB;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  // warp = BPW bands x MW members (interface through shared memory and two CTA barriers)
  const int mi = lane & (MW - 1);
  // which band pair a warp owns rotates with the CTA index: in a partially ice-covered member only the polar bands
  // take the expensive path, and without the rotation every resident CTA puts that warp on the same SM sub-partition
  constexpr int NWARP = WB * MW / 32;
  const unsigned bid = blockIdx.x + (unsigned)a.block0;   // 16-member group of this CTA
  const int wrot = (a.dbg & 4) ? warp : (int)((warp + bid) % NWARP);
  const int band = wrot * BPW + lane / MW;
  const long long nmem = a.nmem;
  const long long m_first = (long long)bid * MW;
  const long long m_raw = m_first + mi;
  const bool active = m_raw < nmem;
  const long long m = active ? m_raw : nmem - 1;
  const int nx = a.nx, nt = a.nt;

  // the TAB instance integrates the 32-member groups whose table-building parameters agree, the !TAB instance the rest
  if constexpr (!UPAR) {
    if (ebm_classic_group_uniform<MW>(a.par, nmem, m_first, mi) != TAB) return;
  }
  double par[EBM_CLASSIC_NPAR];
#pragma unroll
  for (int k = 0; k < EBM_CLASSIC_NPAR; ++k) par[k] = UPAR ? a.u.par[k] : a.par[(long long)k * nmem + m];

  // ---- shared memory carve-up
  PhysTab* phys = reinterpret_cast<PhysTab*>(smem_raw);          // [NXP]
  ElimTab* elim = reinterpret_cast<ElimTab*>(phys + NXP);        // [NXP]
  CoefTab* coef = reinterpret_cast<CoefTab*>(elim + NXP);        // [NXP]
  double* bandc = reinterpret_cast<double*>(coef + NXP);         // [WB][2]  (be, ga) of a band without masked rows
  double* iface = bandc + 2 * WB;                                // [WB+1][6][MW], last band = zeros
  double* zs = iface + (WB + 1) * 6 * MW;                        // [WB][MW]
  double* red = zs + WB * MW;                                    // [WB][4][MW]
  double* fr = red + WB * 4 * MW;                                // [10][MW]
  double* sumE = fr + 10 * MW;                                   // [NXP][MW]
  double* qsm = sumE + NXP * MW;                                 // [3K][threads] band rows q, s, r
  double* sumT = qsm + 3 * NXP * MW;                             // [NXP][MW], only if the launch writes fields
  double* sumH = sumT + NXP * MW;

  const double pD = par[0], pA = par[1], pB = par[2], pcw = par[3], pS0 = par[4], pS1 = par[5], pS2 = par[6];
  const double pa0 = par[7], pa2 = par[8], pai = par[9], pFb = par[10], pk = par[11], pLf = par[12], pcg = par[13];
  const double ptau = par[14];
  const double dt = 1.0 / nt;
  const double cg_tau = pcg / ptau, dt_tau = dt / ptau;
  const double fac = dt * pD / pcg;          // kappa = (1+dt_tau) I - fac*diffop        classic.jl:21
  const double one_dttau = 1.0 + dt_tau;

  for (int j = tid; j < NXP; j += blockDim.x) {
    const bool v = j < nx;
    const double xj = v ? a.g.x[j] : 0.0, x2 = v ? a.g.x2[j] : 0.0;
    const double ll = v ? a.g.lam_lo[j] : 0.0, lh = v ? a.g.lam_hi[j] : 0.0;
    PhysTab p; CoefTab c;
    const double lhm = (j % K == 0 || !v) ? 0.0 : a.g.lam_hi[j - 1];
    if constexpr (TAB) {
      // pad cells: as open water they absorb aw S = 1000 W/m^2 and stay warm, as ice ai S ~ 0 and they stay frozen
      p.S0x = v ? fma(-pS2, x2, pS0) : 1e-3; p.aw = v ? fma(-pa2, x2, pa0) : 1e6;
      c.kjj = fma(fac, ll + lh, one_dttau); c.aoff = -fac * ll; c.coff = -fac * lh; c.ac = c.aoff * (-fac * lhm);
    } else {   // geometry only: Ctx::phys_at / coef_at apply the member's parameters
      p.S0x = x2; p.aw = x2;
      c.kjj = ll + lh; c.aoff = ll; c.coff = lh; c.ac = ll * lhm;
    }
    p.S1x = xj; p.wts = v ? a.g.wts[j] : 0.0;
    phys[j] = p;
    coef[j] = c;
  }
  for (int qd = tid; qd < 6 * MW; qd += blockDim.x) iface[WB * 6 * MW + qd] = 0.0;
  for (int qd = tid; qd < 10 * MW; qd += blockDim.x) {
    const int r = qd / MW, mm = qd % MW;
    long long gm = m_first + mm;
    if (gm >= nmem) gm = nmem - 1;
    fr[qd] = a.forc[(long long)r * nmem + gm];
  }
  __syncthreads();
  // band-local elimination of the constant matrix kappa (no masked rows)
  if (TAB && tid < WB) {
    const int b = tid;
    double qprev = 0.0, sprev = 0.0;
    for (int i = 0; i < K; ++i) {
      const CoefTab c = coef[b * K + i];
      const double w = (i == 0) ? c.kjj : c.kjj - c.aoff * qprev;
      ElimTab e; e.iw = 1.0 / w; e.tq = c.aoff * e.iw; e.q = c.coff * e.iw; e.s = (i == 0) ? e.tq : -e.tq * sprev;
      elim[b * K + i] = e;
      qprev = e.q; sprev = e.s;
    }
    double be = elim[b * K + K - 2].s, ga = elim[b * K + K - 2].q;
    for (int i = K - 3; i >= 0; --i) {
      const ElimTab e = elim[b * K + i];
      be = e.s - e.q * be;
      ga = -e.q * ga;
    }
    bandc[2 * b] = be; bandc[2 * b + 1] = ga;
  }

  Ctx<K, WB, MW, TAB, UPAR> cx;
  cx.S0m = pS0; cx.S2m = pS2; cx.a0m = pa0; cx.a2m = pa2; cx.facm = fac; cx.fac2m = fac * fac; cx.one_dttaum = one_dttau;
  cx.rs.base = qsm + tid;
  cx.rs.stride = WB * MW;
  cx.phys = phys; cx.elim = elim; cx.coef = coef; cx.bandc = bandc;
  cx.iface = iface; cx.zs = zs; cx.red = red; cx.sumE = sumE; cx.sumT = sumT; cx.sumH = sumH;
  cx.A_ = pA; cx.Fb_ = pFb; cx.ai_ = pai; cx.cg_tau_ = cg_tau; cx.M_ = pB + cg_tau; cx.kLf_ = pk * pLf;
  cx.inv_cw_ = 1.0 / pcw; cx.dt_ = dt; cx.dt_tau_ = dt_tau; cx.dttau_cw_ = dt_tau * cx.inv_cw_; cx.dc_ = dt_tau * cg_tau;
  cx.inv_nt_ = 1.0 / nt; cx.inv_Lf_ = 1.0 / pLf;
  const double cM = UPAR ? a.u.M : cx.M_, ckLf = UPAR ? a.u.kLf : cx.kLf_;
  cx.band = band; cx.mi = mi; cx.j0 = band * K;
  cx.solver = (a.dbg & 8) ? warp == 0 : (wrot == (NWARP > 1 ? 1 : 0));
  cx.active = active;
  const long long mo = a.orig != nullptr ? a.orig[m] : m;   // ebm_classic_device_args_t.member_index
  cx.sel = active && ebm_field_selected(a, mo);
  cx.cta_fields = __syncthreads_or(cx.sel && (a.seasonal != nullptr)) != 0;
  cx.accT = 0.0;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = cx.j0 + i;
    const bool v = j < nx;
    // -0.0 -> +0.0: classic.jl:47's masks are E>0 / E<0 (alpha = 0 at either zero), the sign-bit tests below would
    // take -0.0 for ice; an FMA result is -0.0 only if both addends are, so the state never produces one itself
    cx.E[i] = (v ? a.E[(long long)j * nmem + m] : 1.0) + 0.0;     // pad cells: decoupled open-water rows
    cx.Tg[i] = v ? a.Tg[(long long)j * nmem + m] : 0.0;
    sumE[cx.cidx(i)] = 0.0;
    cx.rs.r(i) = cx.E[i] * ebm_rcp(fma(cM, cx.E[i], -ckLf));   // same expression as in the step: r is a pure function of E
    if (cx.cta_fields) { sumT[cx.cidx(i)] = 0.0; sumH[cx.cidx(i)] = 0.0; }
  }
  cx.set_pads(a);
  const auto frow = [&](int r) { return fr[r * MW + mi]; };
  const double fbase = frow(0);
  const bool constf = __syncthreads_and(ebm_forcing_const(frow)) != 0;
  const bool has_raw = __syncthreads_or(cx.sel && (a.raw != nullptr)) != 0;

  const double cS1 = UPAR ? a.u.par[5] : pS1;
  double S1c_next = cS1 * __ldg(a.g.ctab);   // S1*cos(2*pi*t_1); ctab[nt] == ctab[0] closes the year (classic.jl:25)
  for (int year = a.year0; year < a.year0 + a.nyears; ++year) {
    const bool raw_year = has_raw && (!a.lastonly || year == a.dur - 1);   // not ebm_raw_year: -3 instructions each instance
#pragma unroll 1
    for (int ti = 1; ti <= nt; ++ti) {
      // The loop carries `ti` and `year` only: an opaque copy of the index keeps ptxas from expanding it into 64-bit
      // induction variables (table pointer, global step number), which it then spilled -- 8 local-memory instructions in a
      // dependent chain at the end of every step.
      int tix = ti;
      asm volatile("" : "+r"(tix));
      // column i+1 of this step is column i of the next: one table load per step, consumed late in the step
      const double S1c0 = S1c_next, S1c1 = cS1 * __ldg(a.g.ctab + tix);
      S1c_next = S1c1;
      double f = fbase;
      if (!constf) {
        const long long tinx = (long long)(year + a.start_year) * nt + tix;
        f = ebm_forcing_at(frow, tinx, nt);
      }
      const bool slow = cx.cta_fields || raw_year || ti == a.winter_inx || ti == a.summer_inx || ti == nt;
      if (slow) cx.template step<true>(a, f, S1c0, S1c1, ti, year);
      else cx.template step<false>(a, f, S1c0, S1c1, ti, year);
    }
  }

  bool bad = false;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = cx.j0 + i;
    if (j < nx && active) {
      a.E[(long long)j * nmem + m] = cx.E[i];
      a.Tg[(long long)j * nmem + m] = cx.Tg[i];
      bad = bad || ebm_state_bad(cx.E[i]) || ebm_state_bad(cx.Tg[i]);
    }
  }
  if (bad && a.flags != nullptr) atomicOr(a.flags + mo, 1);
}

template <int K, int WB, int MW, int MAXR, bool TAB = true, bool UPAR = false>
int launch_uniform(const ClassicKArgs& a, cudaStream_t stream) {
  if (a.nx > K * WB) {
    ebm_set_error("classic_uniform: nx=%d exceeds %d bands of %d cells", a.nx, WB, K);
    return EBM_ERR_UNSUPPORTED;
  }
  const bool fields = a.seasonal != nullptr && a.field_stride > 0;
  const size_t smem = uniform_smem_bytes<K, WB, MW>(fields);
  auto kern = classic_uniform_kernel<K, WB, MW, MAXR, TAB, UPAR>;
  EBM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // leave room for several CTAs per SM: ask for the largest shared-memory carve-out (L1 is hardly used)
  EBM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  const long long blocks = a.nblocks > 0 ? a.nblocks : (a.nmem + MW - 1) / MW - a.block0;
  if (blocks <= 0) return EBM_OK;
  kern<<<(unsigned)blocks, WB * MW, smem, stream>>>(a);
  EBM_CUDA_TRY(cudaGetLastError());
  ebm_count_launch();
  return EBM_OK;
}

}  // namespace

// resident CTAs of the production instantiation (nx <= kClassic8BandMaxNx) on the current device
int ebm_classic_uniform_slots() {
  int dev = 0, sms = 0, per_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) { cudaGetLastError(); return 0; }
  auto kern = classic_uniform_kernel<13, 8, 16, 168, true, false>;
  const size_t smem = uniform_smem_bytes<13, 8, 16>(false);
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 8 * 16, smem) != cudaSuccess) { cudaGetLastError(); return 0; }
  return sms * per_sm;
}

// <K cells per thread, WB bands, MW members per CTA, max registers per thread>.  Up to kClassic8BandMaxNx: band rows
// (pivots / spikes / carried reciprocals) in thread-private shared memory, 168 registers, 3 CTAs (12 warps) per SM;
// larger grids: 16 bands, 8 warps per CTA, 1 CTA per SM.  The mappings measured and rejected are in DESIGN.md 4.1.
int ebm_launch_classic_uniform(const ClassicKArgs& a, cudaStream_t stream) {
  if (a.nx > kClassic8BandMaxNx) return launch_uniform<13, 16, 16, 255>(a, stream);
  if (a.upar) return launch_uniform<13, 8, 16, 168, true, true>(a, stream);
  return launch_uniform<13, 8, 16, 168>(a, stream);
}

// groups whose table-building parameters differ between members (e.g. a sweep over D): same mapping, coefficients
// applied per member, every band eliminated in full
int ebm_launch_classic_general(const ClassicKArgs& a, cudaStream_t stream) {
  if (a.upar) return EBM_OK;   // the launch-uniform instance integrated every group
  if (a.nx > kClassic8BandMaxNx) return launch_uniform<13, 16, 16, 255, false>(a, stream);
  return launch_uniform<13, 8, 16, 168, false>(a, stream);
}

// dev: read and reset the phase counters (zeros unless built with -DEBM_PHASE_TIMING)
extern "C" int ebm_debug_phase_cycles(unsigned long long* out64) {
#ifdef EBM_PHASE_TIMING
  if (cudaMemcpyFromSymbol(out64, g_phase_cycles, sizeof(unsigned long long) * 64) != cudaSuccess) return -2;
  unsigned long long z[64] = {0};
  cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z));
  return 0;
#else
  for (int i = 0; i < 64; ++i) out64[i] = 0;
  return 1;
#endif
}
