// ebm_internal.cuh -- shared declarations of libebm_cuda.so (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "ebm_cuda.h"

// ----------------------------------------------------------------------------- error plumbing
void ebm_set_error(const char* fmt, ...);
void ebm_count_launch(int n = 1);

#define EBM_CUDA_TRY(expr)                                                                        \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) {                                                                      \
      ebm_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);  \
      return (_e == cudaErrorMemoryAllocation) ? EBM_ERR_OOM : EBM_ERR_CUDA;                      \
    }                                                                                             \
  } while (0)
#define EBM_TRY(expr) do { int _rc = (expr); if (_rc != EBM_OK) return _rc; } while (0)

// ----------------------------------------------------------------------------- host-buffer runs (ebm_capi.cu)
// One call of ebm_classic_run or ebm_miz_run, described by the arrays its model carries.  Host arrays are
// [nmem][...]; an output pointer may be NULL (not wanted).
struct EbmHostRun {
  int npar, nvar, nstate;                 // nstate: classic 2 (E, Tg); MIZ 6 (Ei, Ew, h, D, phi, T0)
  const double* par; const double* forc;  // [nmem][npar], [nmem][EBM_NFORCING]
  const double* init[6];                  // [nmem][nx]; NULL uploads zeros (MIZ T0guess only)
  double* diag; double* seasonal; double* raw;
  double* fin[6];                         // final state planes
  int64_t* newton_iters; int64_t* nonconv; int32_t* flags;
  // The model's device entry point, called with a copy of this description whose arrays are on the device ([...][nmem];
  // the state planes, updated in place, are `fin`).  member_index: NULL or the permutation `order` returned.
  int (*run_device)(const ebm_grid_t* grid, long long nmem, const EbmHostRun& dev, const long long* member_index,
                    const ebm_options_t& opt, cudaStream_t stream);
  // NULL, or the order in which the members go to the device: perm[slot] = original index; empty = the caller's order
  std::vector<long long> (*order)(const ebm_grid_t* grid, long long nmem, const EbmHostRun& run, const ebm_options_t& opt);
};
EbmHostRun ebm_classic_host_run(const ebm_classic_params_t* par, const ebm_forcing_t* forc, const double* E0,
                                const double* Tg0, const ebm_classic_outputs_t* out);
EbmHostRun ebm_miz_host_run(const ebm_miz_params_t* par, const ebm_forcing_t* forc, const double* Ei0, const double* Ew0,
                            const double* h0, const double* D0, const double* phi0, const double* T0guess,
                            const ebm_miz_outputs_t* out);
// Receives the device-resident diagnostics of a host run instead of a copy to run.diag: ebm_*_run_multi sends them
// to another GPU over NCCL.
struct EbmDiagHook {
  virtual int consume(const double* ddiag, size_t count, cudaStream_t stream) = 0;   // EBM_* status
  virtual ~EbmDiagHook() {}
};
// Uploads, integrates on a private stream of opt->device and downloads; diag_hook (may be NULL) takes the diagnostics.
int ebm_run_host(const ebm_grid_t* grid, long long nmem, const EbmHostRun& run, const ebm_options_t* opt,
                 EbmDiagHook* diag_hook);
ebm_options_t default_options();   // device -1, lastonly 1, everything else 0
// Classic regime of one member's state E [nx]: 0 ice free, 1 partial cover, 2 every cell ice.
int ebm_classic_regime(const double* E, int nx);

// ----------------------------------------------------------------------------- multi-device (ebm_multi.cu)
int ebm_launch_scatter_rows(const double* src, double* dst, long long nrows, long long rowlen, const long long* idx,
                            cudaStream_t stream);   // dst[idx[r]][:] = src[r][:]
void ebm_multi_shutdown();   // destroys the NCCL communicators of ebm_multi.cu

// ----------------------------------------------------------------------------- device grid tables
// Everything that depends only on SpaceTime (x, t, nx, nt), computed once on the host in IEEE
// double with the reference's association order, cached per device (ebm_capi.cu).
struct EbmGridTables {
  int nx, nt, kind;
  const double* x;       // [nx]      st.x
  const double* x2;      // [nx]      x*x
  const double* lam_lo;  // [nx]      get_diffop lambda between j-1 and j (0 at j=0)        infrastructure.jl:482-488
  const double* lam_hi;  // [nx]      lambda between j and j+1 (0 at j=nx-1)
  const double* wts;     // [nx]      hemispheric_mean trapezoid weight of cell j            utilities.jl:397-403
  const double* ctab;    // [nt+1]    cos(2*pi*t_i), entry nt := entry 0                      classic.jl:24-25
  // generic flux-form stencil (infrastructure.jl:509-519)
  const double* diffx;   // [nx+1]
  const double* mxxph;   // [nx]
  const double* mxxmh;   // [nx]
  const double* phmmh;   // [nx]
  // the same stencil as matrix coefficients (classic on non-uniform grids, ebm_options_t.classic_stencil)
  const double* glam_lo; // [nx]      mxxmh / (diffx[j] * phmmh),   0 at j = 0
  const double* glam_hi; // [nx]      mxxph / (diffx[j+1] * phmmh), 0 at j = nx-1
};

// ----------------------------------------------------------------------------- kernel argument blocks
// Classic member constants of a launch in which every member has the same 15 parameters (the C4 forcing sweep):
// derived on the host with the same IEEE expressions the kernels use per member, read as constant-bank operands.
struct ClassicUPar {
  double par[EBM_CLASSIC_NPAR];
  double A, Fb, ai, cg_tau, M, kLf, inv_cw, dt, dt_tau, dttau_cw, dc, inv_nt, inv_Lf;
};

struct ClassicKArgs {
  int nx, nt, dur, W;
  long long nmem;
  int year0, nyears;             // integrate years [year0, year0+nyears), 0-based
  int start_year;                // years already simulated before this run: added to the time passed to Forcing
  int winter_inx, summer_inx, lastonly, field_stride, all_const_forcing;
  int reserved;                  // unused: keeps the argument-block layout, and with it the measured code of the classic kernels
  EbmGridTables g;
  const double* par;             // [15][nmem]
  const double* forc;            // [10][nmem]
  double* E; double* Tg;         // [nx][nmem]
  double* diag; double* seasonal; double* raw; int* flags;
  const long long* orig;         // NULL or [nmem]: original member index of slot m (output rows, field selection)
  int dbg;                       // development switches (env EBM_DBG): 4 no band-pair rotation, 8 warp 0 solves the interface
  int hthr;                      // high word of 512/nt: an open-water cell with E above it cannot freeze within one step
  int upar;                      // 1: u is valid (every member of the launch shares all 15 parameters)
  ClassicUPar u;
  long long block0, nblocks;     // classic_uniform.cu: this launch covers the 16-member groups [block0, block0 + nblocks); nblocks 0 = all
};

struct MizKArgs {
  int nx, nt, dur;
  long long nmem;
  int year0, nyears;
  int winter_inx, summer_inx, lastonly, field_stride, all_const_forcing;
  int maxit; double tol;
  int start_year;                  // years already simulated before this run (Forcing time offset)
  int step_limit;                  // > 0: stop after this many steps of the run (partial last year)
  int single_ti; double single_f;  // > 0: exactly one step at year-index single_ti with forcing single_f (ebm_miz_step)
  EbmGridTables g;
  const double* par;             // [22][nmem]
  const double* forc;            // [10][nmem]
  double *Ei, *Ew, *h, *D, *phi, *T0;   // [nx][nmem]
  double* diag; double* seasonal; double* raw;
  long long* newton_iters; long long* nonconv; int* flags;
};

// launchers (each returns an EBM_* status; kernels are enqueued on `stream`)
// classic_uniform.cu integrates grids of up to 16 bands of 13 cells; up to 8 bands it runs 3 CTAs per SM and has
// the launch-uniform-parameter instance.  Larger grids take classic_bands.cu.
constexpr int kClassic8BandMaxNx = 13 * 8;
constexpr int kClassicUniformMaxNx = 13 * 16;
int ebm_launch_classic_bands(const ClassicKArgs& a, cudaStream_t stream);
int ebm_launch_classic_uniform(const ClassicKArgs& a, cudaStream_t stream);
int ebm_launch_classic_general(const ClassicKArgs& a, cudaStream_t stream);
int ebm_classic_uniform_slots();   // resident CTAs of the production kernel on the current device (wave balancing)
int ebm_launch_classic_strict(const ClassicKArgs& a, cudaStream_t stream);
int ebm_launch_classic_single_step(const EbmGridTables& g, const double* par15, int ti, double f,
                                   double* E, double* Tg, double* T, double* h, cudaStream_t stream,
                                   int dbg_which = 0, double* dbg = nullptr);   // dbg: device [nx] or NULL (EBM_DEBUG_*)
int ebm_launch_miz(const MizKArgs& a, int strict, cudaStream_t stream);
int ebm_launch_miz_fast(const MizKArgs& a, cudaStream_t stream);     // miz_kernel.cu
int ebm_launch_miz_strict(const MizKArgs& a, cudaStream_t stream);   // miz_strict.cu (-fmad=false)
int ebm_launch_miz_single_step(const EbmGridTables& g, const double* par22, int ti, double f, double tol, int maxit,
                               double* Ei, double* Ew, double* h, double* D, double* phi, double* T0,
                               double* vars_out, long long* iters, cudaStream_t stream);
int ebm_launch_transpose(const double* src, double* dst, long long rows, long long cols, cudaStream_t stream);
int ebm_launch_fill(double* dst, long long n, double v, cudaStream_t stream);
// head[k] = par[k][0] (k < npar); *differs = 1 if some member's parameters are not bit-identical to member 0's
int ebm_launch_par_uniform(const double* par, int npar, long long nmem, double* head, int* differs, cudaStream_t stream);
// dst[c][r] = src[idx[r]][c] (rows x cols -> cols x rows with a row gather); inverse: dst[idx[r]][c] = src[c][r]
int ebm_launch_gather_transpose(const double* src, double* dst, long long rows, long long cols, const long long* idx,
                                int inverse, cudaStream_t stream);
int ebm_run_fp64_peak(int device, double* tflops, double* mhz);

// ----------------------------------------------------------------------------- small device helpers
// Forcing call (src/infrastructure.jl:294-307).  fr = base, peak, cool, rate_up, rate_down, d1..d5.
__device__ __forceinline__ double ebm_forcing_eval(double base, double peak, double cool, double rup, double rdown,
                                                   double d2, double d3, double d4, double d5, double T) {
  if (T < d2) return base;
  if (T < d3) return base + rup * (T - d2);
  if (T < d4) return peak;
  if (T < d5) return peak + rdown * (T - d4);
  return cool;
}

// SpaceTime.T[tinx] (1-based): correctly rounded (2*tinx-1)/(2*nt)  (infrastructure.jl:130, TwicePrecision range)
__device__ __forceinline__ double ebm_global_time(long long tinx, int nt) {
  return __ddiv_rn((double)(2 * tinx - 1), (double)(2LL * nt));
}

// The classic parameters that feed the CTA-wide tables of classic_uniform.cu: D, cg, tau (the matrix kappa,
// classic.jl:21) and S0, S2, a0, a2 (insolation / albedo profiles, :23-28); A, B, cw, S1, ai, Fb, k, Lf are
// per-member registers.
constexpr int kClassicNTablePar = 7;
__host__ __device__ constexpr int ebm_classic_table_par(int q) {
  constexpr int k[kClassicNTablePar] = {0, 4, 6, 7, 8, 13, 14};
  return k[q];
}

// Do the members of the 32-aligned group that contains this CTA's members share the table-building classic
// parameters bit for bit?  Called by every thread of the CTA (contains a barrier); mi = member slot of the thread, MW = members per
// CTA (a divisor of 32).  The uniform and the general kernel use this same rule to split an ensemble between them.
template <int MW>
__device__ __forceinline__ bool ebm_classic_group_uniform(const double* __restrict__ par, long long nmem,
                                                          long long m_first, int mi) {
  const long long g0 = (m_first / 32) * 32;
  bool same = true;
#pragma unroll 1
  for (int r = 0; r < 32 / MW; ++r) {
    long long mm = g0 + mi + (long long)r * MW;
    if (mm >= nmem) mm = nmem - 1;
    for (int q = 0; q < kClassicNTablePar; ++q) {
      const int k = ebm_classic_table_par(q);
      same = same && (par[(long long)k * nmem + mm] == par[(long long)k * nmem + g0]);
    }
  }
  return __syncthreads_and(same) != 0;
}
