// classic_bands.cu -- band kernel of the classic (Wagner-Eisenman) EBM ensemble: the first fast kernel of this
// library, now the kernel for grids with 208 < nx <= 256; classic_uniform.cu integrates everything up to 208 cells
// 2-3x faster.
//
// Replaces, for a whole ensemble and many years per launch, the reference's
//   integrate loop           src/infrastructure.jl:630-634
//   step!(::Val{:Classic})   src/classic.jl:43-65   (arithmetic spec: SURVEY.md Appendix A)
//   savesol! / annual_mean   src/infrastructure.jl:536-591
//
// Mapping (B200: 148 SMs, 64 FP64 lanes/SM, 64K regs/SM, no tensor-core work in this path):
//   * lane  = ensemble member  -> every latitude-dependent constant is warp-uniform (shared-memory
//             broadcast), per-member parameters live in registers, global I/O is coalesced over members,
//             and the ice / no-ice branch diverges only between members, never between latitudes.
//   * warp  = latitude band of K cells; a CTA = MW members x W bands.  Each member's E and Tg stay in
//             registers for the whole launch (years); nothing but sampled output touches HBM.
//   * the implicit ghost-layer solve (a symmetric tridiagonal system whose diagonal depends on the
//             member's current ice mask, classic.jl:55-63) is a partitioned solve: every band eliminates
//             its K rows locally carrying a left spike, one half-warp solves the W x W interface system,
//             and every band back-substitutes.  Two CTA barriers per time step.
//   * insolation is computed on the fly from a per-step cos(2*pi*t) table (1 value per step).
//   * annual means are running sums in shared memory; diagnostics are reduced across bands in shared
//     memory and written once per season.
//
// Arithmetic here is NOT the literal association order of the reference (reciprocal multiplies, merged
// divisions, FMA contraction): results agree with the oracle to ~1e-12 relative, the stated tolerance is
// 1e-9 (tests/test_classic_gpu.py).  The literal-order kernel is classic_strict.cu.
#include "ebm_internal.cuh"

namespace {

// reciprocal for well-scaled operands (pivots of a diagonally dominant matrix, 1 <= |w| < 1e4): MUFU.RCP64H seed +
// two Newton steps, ~1 ulp, no denormal/overflow slow path.  Not ebm_rcp: its one cubic step gives other bits.
__device__ __forceinline__ double rcp_newton2(double w) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(w));
  double e = fma(-w, x, 1.0);
  x = fma(x, e, x);
  e = fma(-w, x, 1.0);
  x = fma(x, e, x);
  return x;
}

template <int K, int MW, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) classic_bands_kernel(const ClassicKArgs a) {
  extern __shared__ double smem[];
  constexpr int BPW = 32 / MW;  // bands per warp
  const int W = a.W;
  const int NXP = W * K;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int mi = lane & (MW - 1);
  const int band_raw = warp * BPW + lane / MW;
  const int band = band_raw < W ? band_raw : W - 1;   // (the launcher rounds W up to whole warps: band_raw < W always)
  const long long m_raw = (long long)blockIdx.x * MW + mi;
  const bool active = m_raw < a.nmem && band_raw < W;
  const long long m = active ? m_raw : a.nmem - 1;
  const long long nmem = a.nmem;
  const int nx = a.nx, nt = a.nt;
  const int j0 = band * K;

  // ---- shared memory carve-up
  double* xs = smem;               // [NXP]
  double* x2s = xs + NXP;          // [NXP]
  double* lamlo = x2s + NXP;       // [NXP]  lambda between j-1 and j
  double* lamhi = lamlo + NXP;     // [NXP]  lambda between j and j+1
  double* wts = lamhi + NXP;       // [NXP]
  double* sumE = wts + NXP;        // [NXP][MW] running annual sums
  double* sumT = sumE + NXP * MW;
  double* sumH = sumT + NXP * MW;  // sum of min(E,0)
  double* iface = sumH + NXP * MW; // [W][6][MW]
  double* zs = iface + W * 6 * MW; // [W][MW] interface solution
  double* cqs = zs + W * MW;       // [W][MW]
  double* cys = cqs + W * MW;      // [W][MW]
  double* red = cys + W * MW;      // [W][4][MW] diagnostic partials
  double* fr = red + W * 4 * MW;   // [10][MW] forcing rows

  for (int j = tid; j < NXP; j += blockDim.x) {
    const bool v = j < nx;
    xs[j] = v ? a.g.x[j] : 0.0;
    x2s[j] = v ? a.g.x2[j] : 0.0;
    lamlo[j] = v ? a.g.lam_lo[j] : 0.0;
    lamhi[j] = v ? a.g.lam_hi[j] : 0.0;
    wts[j] = v ? a.g.wts[j] : 0.0;
  }
  for (int q = tid; q < 10 * MW; q += blockDim.x) {
    const int r = q / MW, mm = q % MW;
    long long gm = (long long)blockIdx.x * MW + mm;
    if (gm >= nmem) gm = nmem - 1;
    fr[q] = a.forc[(long long)r * nmem + gm];
  }

  // ---- per-member constants (get_statics, classic.jl:18-29)
  const double pD = a.par[0 * nmem + m], pA = a.par[1 * nmem + m], pB = a.par[2 * nmem + m];
  const double pcw = a.par[3 * nmem + m], pS0 = a.par[4 * nmem + m], pS1 = a.par[5 * nmem + m];
  const double pS2 = a.par[6 * nmem + m], pa0 = a.par[7 * nmem + m], pa2 = a.par[8 * nmem + m];
  const double pai = a.par[9 * nmem + m], pFb = a.par[10 * nmem + m], pk = a.par[11 * nmem + m];
  const double pLf = a.par[12 * nmem + m], pcg = a.par[13 * nmem + m], ptau = a.par[14 * nmem + m];
  const double dt = 1.0 / nt;
  const double cg_tau = pcg / ptau;
  const double dt_tau = dt / ptau;
  const double dc = dt_tau * cg_tau;
  const double M = pB + cg_tau;
  const double kLf = pk * pLf;
  const double inv_cw = 1.0 / pcw;
  const double dttau_cw = dt_tau * inv_cw;
  const double fac = dt * pD / pcg;  // kappa = (1+dt_tau) I - fac * diffop
  const double one_dttau = 1.0 + dt_tau;
  const double inv_nt = 1.0 / nt;
  const double inv_Lf = 1.0 / pLf;

  // ---- state in registers
  double E[K], Tg[K];
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = j0 + i;
    const bool v = j < nx;
    E[i] = v ? a.E[(long long)j * nmem + m] : 0.0;
    Tg[i] = v ? a.Tg[(long long)j * nmem + m] : 0.0;
  }
#pragma unroll
  for (int i = 0; i < K; ++i) {
    sumE[(j0 + i) * MW + mi] = 0.0;
    sumT[(j0 + i) * MW + mi] = 0.0;
    sumH[(j0 + i) * MW + mi] = 0.0;
  }
  __syncthreads();

  const long long mo = a.orig != nullptr ? a.orig[m] : m;   // original member index: output rows
  const bool sel = active && ebm_field_selected(a, mo);
  const long long msel = sel ? ebm_field_row(a, mo) : 0;
  const long long nraw = ebm_nraw(nt, a.dur, a.lastonly);
  // Forcing{true}: the call is `base`.  Not ebm_forcing_const / _at: +5 instructions (-6 with a by-value accessor)
  const double fbase = fr[0 * MW + mi];
  const bool myconst = fr[1 * MW + mi] == fbase && fr[2 * MW + mi] == fbase && fr[6 * MW + mi] == 0.0 &&
                       fr[7 * MW + mi] == 0.0 && fr[8 * MW + mi] == 0.0 && fr[9 * MW + mi] == 0.0;
  const bool constf = __syncthreads_and(myconst) != 0;

  for (int year = a.year0; year < a.year0 + a.nyears; ++year) {
    for (int ti = 1; ti <= nt; ++ti) {
      // ---- per-step scalars
      const double c0 = __ldg(a.g.ctab + (ti - 1)), c1 = __ldg(a.g.ctab + ti);
      const double S1c0 = pS1 * c0, S1c1 = pS1 * c1;
      double f = fbase;
      if (!constf) {
        const long long tinx = (long long)(year + a.start_year) * nt + ti;
        f = ebm_forcing_eval(fr[0 * MW + mi], fr[1 * MW + mi], fr[2 * MW + mi], fr[3 * MW + mi], fr[4 * MW + mi],
                             fr[6 * MW + mi], fr[7 * MW + mi], fr[8 * MW + mi], fr[9 * MW + mi],
                             ebm_global_time(tinx, nt));
      }
      const double fmA = f - pA;
      const int season = ebm_season(a, ti, nt);
      const bool rawstep = sel && a.raw != nullptr && ebm_raw_year(year, a.dur, a.lastonly);
      const long long rawidx = ebm_raw_slot(year, ti, nt, a.lastonly);

      double q[K], s[K];  // Tg[] is reused for rhs -> y -> solution
      double dgT = 0.0, dgE = 0.0, dgA = 0.0, dgX = 2.0;  // diagnostic partials (edge: 2.0 = none)

      // ---- phase A: physics + local forward elimination with left spike
      double qprev = 0.0, yprev = 0.0, sprev = 0.0;
#pragma unroll
      for (int i = 0; i < K; ++i) {
        const int j = j0 + i;
        const double xj = xs[j], x2j = x2s[j];
        const double S0x = fma(-pS2, x2j, pS0);
        const double S = fma(-S1c0, xj, S0x);               // S[j,i]   (classic.jl:23-24)
        const double Eo = E[i], Tgo = Tg[i];
        const double base = fma(cg_tau, Tgo, fmA);           // cg_tau*Tg - A + f
        double C, T;
        bool T0neg;
        if (Eo >= 0.0) {
          const double alpha = (Eo > 0.0) ? fma(-pa2, x2j, pa0) : 0.0;  // :47 (alpha = 0 at E == 0)
          C = fma(alpha, S, base);                                      // :48
          T = Eo * inv_cw;                                              // :51
          // sign of T0 = C/(M - kLf/E) is only needed if this step crosses into E < 0 (rare): literal then
          T0neg = false;
        } else {
          C = fma(pai, S, base);
          const double T0 = (C * Eo) / fma(M, Eo, -kLf);                // :50, C/(M - kLf/E) with one division
          T0neg = T0 < 0.0;
          T = T0neg ? T0 : 0.0;                                         // :51
        }
        double En = fma(dt, fma(-M, T, C) + pFb, Eo);                   // :53
        if (j >= nx) En = 0.0;
        if (Eo >= 0.0 && En < 0.0) {  // freeze-up crossing: evaluate the reference's mask literally
          const double T0 = C / (M - kLf / Eo);
          T0neg = T0 < 0.0;
        }
        E[i] = En;
        // running annual sums (annusol.raw -> crossmean, infrastructure.jl:556-559, utilities.jl:390-395)
        const int sidx = j * MW + mi;
        const double Eneg = En < 0.0 ? En : 0.0;
        sumE[sidx] += En;
        sumT[sidx] += T;
        sumH[sidx] += Eneg;
        // sampled output of this step's fields
        if (season >= 0) {
          double vT = T, vE = En, vN = Eneg;
          if (season == 2) {  // annual mean fields
            vT = sumT[sidx] * inv_nt; vE = sumE[sidx] * inv_nt; vN = sumH[sidx] * inv_nt;
          }
          const double wj = wts[j];
          dgT = fma(wj, vT, dgT);
          dgE = fma(wj, vE, dgE);
          if (vE < 0.0 && j < nx) { dgA += wj; dgX = fmin(dgX, xj); }
          if (sel && a.seasonal != nullptr && j < nx) {
            double* o = a.seasonal + ebm_seasonal_offset(msel, a.dur, year, season, EBM_CLASSIC_NVAR, nx) + j;
            o[0] = vE; o[nx] = vT; o[2 * nx] = -vN * inv_Lf;
          }
        }
        if (rawstep && j < nx) {
          double* o = a.raw + ebm_raw_offset(msel, nraw, rawidx, EBM_CLASSIC_NVAR, nx) + j;
          o[0] = En; o[nx] = T; o[2 * nx] = -Eneg * inv_Lf;   // h = -E/Lf*(E<0)  (:65)
        }
        if (ti == nt) { sumE[sidx] = 0.0; sumT[sidx] = 0.0; sumH[sidx] = 0.0; }

        // implicit ghost-layer row (classic.jl:55-63): masks use T0 of the OLD E and the UPDATED E
        const double kjj = fma(fac, lamlo[j] + lamhi[j], one_dttau);
        double diag, rhs;
        if (En >= 0.0) {
          diag = kjj;
          rhs = fma(dttau_cw, En, Tgo);
        } else if (T0neg) {
          const double r = En / fma(M, En, -kLf);                       // 1/(M - kLf/E)
          diag = fma(-dc, r, kjj);
          const double Sn = fma(-S1c1, xj, S0x);                        // S[j,i+1]
          rhs = fma(dt_tau * r, fma(pai, Sn, fmA), Tgo);
        } else {
          diag = kjj;
          rhs = Tgo;
        }
        // forward elimination:  x_i + q_i x_{i+1} + s_i xL = y_i
        const double ai_ = -fac * lamlo[j];
        const double ci_ = -fac * lamhi[j];
        const double w = (i == 0) ? diag : fma(-ai_, qprev, diag);
        const double iw = rcp_newton2(w);
        const double tq = ai_ * iw;
        q[i] = ci_ * iw;
        const double yi = (i == 0) ? rhs * iw : fma(-tq, yprev, rhs * iw);
        const double si = (i == 0) ? tq : -tq * sprev;
        s[i] = si; Tg[i] = yi;
        qprev = q[i]; yprev = yi; sprev = si;
      }
      // ---- local backward reduction: x_0 = al - be*xL - ga*z  (z = this band's last unknown)
      {
        double al = Tg[K - 2], be = s[K - 2], ga = q[K - 2];
#pragma unroll
        for (int i = K - 3; i >= 0; --i) {
          al = fma(-q[i], al, Tg[i]);
          be = fma(-q[i], be, s[i]);
          ga = -q[i] * ga;
        }
        double* f6 = iface + (band * 6) * MW + mi;
        f6[0 * MW] = s[K - 1]; f6[1 * MW] = q[K - 1]; f6[2 * MW] = Tg[K - 1];
        f6[3 * MW] = al; f6[4 * MW] = be; f6[5 * MW] = ga;
        if (season >= 0) {
          double* r4 = red + (band * 4) * MW + mi;
          r4[0 * MW] = dgT; r4[1 * MW] = dgE; r4[2 * MW] = dgA; r4[3 * MW] = dgX;
        }
      }
      __syncthreads();
      // ---- phase B: interface system (W unknowns per member), one lane group
      if (tid < MW) {
        double cq = 0.0, cy = 0.0;
        for (int b = 0; b < W; ++b) {
          const double* f6 = iface + (b * 6) * MW + mi;
          const double sl = f6[0 * MW], ql = f6[1 * MW], yl = f6[2 * MW];
          double dg = 1.0, sup = 0.0, rh = yl;
          if (b < W - 1) {
            const double* n6 = iface + ((b + 1) * 6) * MW + mi;
            dg = fma(-ql, n6[4 * MW], 1.0);
            sup = -ql * n6[5 * MW];
            rh = fma(-ql, n6[3 * MW], yl);
          }
          const double w = (b == 0) ? dg : fma(-sl, cq, dg);
          const double iw = rcp_newton2(w);
          cy = (b == 0) ? rh * iw : fma(-sl, cy, rh) * iw;
          cq = sup * iw;
          cqs[b * MW + mi] = cq; cys[b * MW + mi] = cy;
        }
        double z = cy;
        zs[(W - 1) * MW + mi] = z;
        for (int b = W - 2; b >= 0; --b) {
          z = fma(-cqs[b * MW + mi], z, cys[b * MW + mi]);
          zs[b * MW + mi] = z;
        }
        if (season >= 0 && a.diag != nullptr && active) {
          double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 2.0;
          for (int b = 0; b < W; ++b) {
            const double* r4 = red + (b * 4) * MW + mi;
            t0 += r4[0 * MW]; t1 += r4[1 * MW]; t2 += r4[2 * MW]; t3 = fmin(t3, r4[3 * MW]);
          }
          ebm_store_diag(a.diag, mo, a.dur, year, season, t0, t1, t2, t3);
        }
      }
      __syncthreads();
      // ---- phase C: back substitution with the true neighbours
      {
        const double xL = (band > 0) ? zs[(band - 1) * MW + mi] : 0.0;
        double xn = zs[band * MW + mi];
        Tg[K - 1] = xn;
#pragma unroll
        for (int i = K - 2; i >= 0; --i) {
          xn = fma(-q[i], xn, fma(-s[i], xL, Tg[i]));
          Tg[i] = xn;
        }
      }
    }
  }

  // ---- write back the final state
  bool bad = false;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int j = j0 + i;
    if (j < nx && active) {
      a.E[(long long)j * nmem + m] = E[i];
      a.Tg[(long long)j * nmem + m] = Tg[i];
      bad = bad || ebm_state_bad(E[i]) || ebm_state_bad(Tg[i]);
    }
  }
  if (bad && a.flags != nullptr) atomicOr(a.flags + mo, 1);
}

template <int K, int MW, int MAXT, int MINB>
int launch_variant(const ClassicKArgs& a0, cudaStream_t stream) {
  ClassicKArgs a = a0;
  // whole warps only: with MW = 16 an odd band count gets one more band of pad cells (decoupled rows), so that no
  // thread has to shadow another thread's band (two threads updating the same shared-memory slots)
  constexpr int BPW = 32 / MW;
  a.W = (a.nx + K - 1) / K;
  a.W = (a.W + BPW - 1) / BPW * BPW;
  if (a.W < 1 || a.W * MW > MAXT) {
    ebm_set_error("classic_bands: nx=%d needs %d bands of %d cells (> %d threads)", a.nx, a.W, K, MAXT);
    return EBM_ERR_UNSUPPORTED;
  }
  const int threads = ((a.W * MW + 31) / 32) * 32;
  const int NXP = a.W * K;
  const size_t smem = sizeof(double) * ((size_t)5 * NXP + (size_t)3 * NXP * MW + (size_t)a.W * MW * (6 + 3 + 4) + 10 * MW);
  auto kern = classic_bands_kernel<K, MW, MAXT, MINB>;
  EBM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long blocks = (a.nmem + MW - 1) / MW;
  kern<<<(unsigned)blocks, threads, smem, stream>>>(a);
  EBM_CUDA_TRY(cudaGetLastError());
  ebm_count_launch();
  return EBM_OK;
}

}  // namespace

int ebm_launch_classic_bands(const ClassicKArgs& a, cudaStream_t stream) {
  // up to 16 bands of 16 cells, 16 members per CTA
  if (a.nx <= 2) { ebm_set_error("classic_bands: nx must be > 2"); return EBM_ERR_INVALID; }
  if (a.nx <= 256) return launch_variant<16, 16, 256, 1>(a, stream);
  ebm_set_error("classic_bands: nx=%d > 256 not supported by the register-resident kernel", a.nx);
  return EBM_ERR_UNSUPPORTED;
}
