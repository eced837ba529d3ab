// ebm_capi.cu -- the C ABI of libebm_cuda.so (include/ebm_cuda.h): argument checking, the cached
// device tables that depend only on SpaceTime, host<->device marshalling, launch orchestration.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <map>
#include <mutex>
#include <vector>

#include "ebm_internal.cuh"

// ----------------------------------------------------------------------------- errors / counters
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void ebm_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void ebm_count_launch(int n) { g_launches += n; }

extern "C" const char* ebm_version(void) { return "ebm_cuda 0.1.0 (sm_100a)"; }
extern "C" const char* ebm_last_error(void) { return g_err; }
extern "C" int64_t ebm_launch_count(void) { return g_launches.load(); }
extern "C" int32_t ebm_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// ----------------------------------------------------------------------------- grid table cache
namespace {

struct GridCacheEntry {
  int device, nx, nt, kind;
  unsigned long long hash;
  double* dev;  // one allocation holding every table
  EbmGridTables tabs;
};
std::mutex g_cache_mu;
std::vector<GridCacheEntry> g_cache;          // least recently used first
constexpr size_t kMaxGridCache = 16;

unsigned long long fnv1a(const void* p, size_t n, unsigned long long h = 1469598103934665603ULL) {
  const unsigned char* b = (const unsigned char*)p;
  for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ULL; }
  return h;
}

int check_grid(const ebm_grid_t* g) {
  if (!g || !g->x || !g->t) { ebm_set_error("grid, grid->x and grid->t must be non-NULL"); return EBM_ERR_INVALID; }
  if (g->nx < 3 || g->nt < 1 || g->dur < 1) { ebm_set_error("need nx >= 3, nt >= 1, dur >= 1 (got %d, %d, %d)", g->nx, g->nt, g->dur); return EBM_ERR_INVALID; }
  if (g->grid_kind != 0 && g->grid_kind != 1) { ebm_set_error("grid_kind must be 0 (identity) or 1 (generic)"); return EBM_ERR_INVALID; }
  return EBM_OK;
}

// Build (or fetch) the device tables for this SpaceTime on the current device.
int get_tables(const ebm_grid_t* g, EbmGridTables* out, cudaStream_t stream) {
  int dev = 0;
  EBM_CUDA_TRY(cudaGetDevice(&dev));
  unsigned long long h = fnv1a(g->x, sizeof(double) * g->nx);
  h = fnv1a(g->t, sizeof(double) * g->nt, h);
  std::lock_guard<std::mutex> lk(g_cache_mu);
  for (size_t k = 0; k < g_cache.size(); ++k) {
    auto& e = g_cache[k];
    if (e.device == dev && e.nx == g->nx && e.nt == g->nt && e.kind == g->grid_kind && e.hash == h) {
      *out = e.tabs;
      if (k + 1 != g_cache.size()) { GridCacheEntry hit = e; g_cache.erase(g_cache.begin() + k); g_cache.push_back(hit); }   // most recent last
      return EBM_OK;
    }
  }
  const int nx = g->nx, nt = g->nt;
  // layout: x, x2, lam_lo, lam_hi, wts [nx each]; ctab [nt+1]; diffx [nx+1]; mxxph, mxxmh, phmmh, glam_lo, glam_hi [nx each]
  const size_t n = (size_t)5 * nx + (nt + 1) + (nx + 1) + (size_t)5 * nx;
  std::vector<double> hbuf(n, 0.0);
  double* x = hbuf.data(); double* x2 = x + nx; double* lam_lo = x2 + nx; double* lam_hi = lam_lo + nx;
  double* wts = lam_hi + nx; double* ctab = wts + nx; double* diffx = ctab + nt + 1;
  double* mxxph = diffx + nx + 1; double* mxxmh = mxxph + nx; double* phmmh = mxxmh + nx;
  double* glo = phmmh + nx; double* ghi = glo + nx;
  const double dx = 1.0 / nx;
  for (int j = 0; j < nx; ++j) { x[j] = g->x[j]; x2[j] = g->x[j] * g->x[j]; }
  // get_diffop (src/infrastructure.jl:482-484): xb = dx:dx:1-dx (== j/nx), lambda = (1 - xb^2)/dx^2
  for (int b = 1; b <= nx - 1; ++b) {
    const double xb = (double)b / (double)nx;
    const double lam = (1 - xb * xb) / (dx * dx);
    lam_lo[b] = lam;      // boundary between cell b-1 and b, seen from cell b
    lam_hi[b - 1] = lam;  // ... seen from cell b-1
  }
  // hemispheric_mean (src/utilities.jl:397-403) as per-cell trapezoid weights
  for (int j = 0; j < nx; ++j) {
    double w = 0.0;
    if (j < nx - 1) w += (g->x[j + 1] - g->x[j]) / 2.0;
    if (j > 0) w += (g->x[j] - g->x[j - 1]) / 2.0;
    wts[j] = w;
  }
  for (int i = 0; i < nt; ++i) ctab[i] = cos(2.0 * kPi * g->t[i]);  // classic.jl:24, miz.jl:11
  ctab[nt] = ctab[0];                                               // classic.jl:25
  {  // generic stencil caches, src/infrastructure.jl:510-518
    std::vector<double> xe(nx + 2);
    xe[0] = -g->x[0];
    for (int j = 0; j < nx; ++j) xe[j + 1] = g->x[j];
    xe[nx + 1] = 2 - g->x[nx - 1];
    for (int q = 0; q < nx + 1; ++q) diffx[q] = xe[q + 1] - xe[q];
    for (int j = 0; j < nx; ++j) {
      const int i = j + 1;
      const double xxph = (xe[i + 1] + xe[i]) / 2.0, xxmh = (xe[i] + xe[i - 1]) / 2.0;
      mxxph[j] = 1.0 - xxph * xxph; mxxmh[j] = 1.0 - xxmh * xxmh; phmmh[j] = xxph - xxmh;
      glo[j] = j > 0 ? mxxmh[j] / (diffx[j] * phmmh[j]) : 0.0;            // zero flux at both ends (:520-521)
      ghi[j] = j < nx - 1 ? mxxph[j] / (diffx[j + 1] * phmmh[j]) : 0.0;
    }
  }
  double* dbuf = nullptr;
  EBM_CUDA_TRY(cudaMalloc(&dbuf, sizeof(double) * n));
  EBM_CUDA_TRY(cudaMemcpyAsync(dbuf, hbuf.data(), sizeof(double) * n, cudaMemcpyHostToDevice, stream));
  EBM_CUDA_TRY(cudaStreamSynchronize(stream));  // hbuf goes out of scope
  GridCacheEntry e;
  e.device = dev; e.nx = nx; e.nt = nt; e.kind = g->grid_kind; e.hash = h; e.dev = dbuf;
  e.tabs.nx = nx; e.tabs.nt = nt; e.tabs.kind = g->grid_kind;
  e.tabs.x = dbuf; e.tabs.x2 = dbuf + nx; e.tabs.lam_lo = dbuf + 2 * nx; e.tabs.lam_hi = dbuf + 3 * nx;
  e.tabs.wts = dbuf + 4 * nx; e.tabs.ctab = dbuf + 5 * nx; e.tabs.diffx = e.tabs.ctab + nt + 1;
  e.tabs.mxxph = e.tabs.diffx + nx + 1; e.tabs.mxxmh = e.tabs.mxxph + nx; e.tabs.phmmh = e.tabs.mxxmh + nx;
  e.tabs.glam_lo = e.tabs.phmmh + nx; e.tabs.glam_hi = e.tabs.glam_lo + nx;
  // bounded: the least recently used entry goes when the cache is full.  Its tables may still be read by kernels in
  // flight on other streams, so the block is released only after the device has drained.
  if (g_cache.size() >= kMaxGridCache) {
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(g_cache.front().device);
    cudaDeviceSynchronize();
    cudaFree(g_cache.front().dev);
    cudaSetDevice(cur);
    g_cache.erase(g_cache.begin());
  }
  g_cache.push_back(e);
  *out = e.tabs;
  return EBM_OK;
}

// Restores the caller's current CUDA device when an entry point returns (select_device may change it).
struct DeviceRestore {
  int prev = -1;
  DeviceRestore() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
  ~DeviceRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

int select_device(const ebm_options_t& o) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    ebm_set_error("no CUDA device available (%s); libebm_cuda has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return EBM_ERR_CUDA;
  }
  if (o.device >= n) { ebm_set_error("device %d out of range (%d devices)", o.device, n); return EBM_ERR_INVALID; }
  if (o.device >= 0) EBM_CUDA_TRY(cudaSetDevice(o.device));
  return EBM_OK;
}

// Device workspace of the host entry points.  cudaMalloc / cudaFree of the GB-sized staging and output buffers cost
// up to hundreds of milliseconds per call, so freed blocks are kept per device and reused by the next call
// (released by ebm_shutdown, or when an allocation fails).
struct WsBlock { int device; void* ptr; size_t bytes; bool in_use; };
std::mutex g_ws_mu;
std::vector<WsBlock> g_ws;

void ws_release_free_blocks(int device) {   // caller holds g_ws_mu
  for (size_t i = 0; i < g_ws.size();) {
    if (!g_ws[i].in_use && (device < 0 || g_ws[i].device == device)) {
      cudaFree(g_ws[i].ptr);
      g_ws[i] = g_ws.back(); g_ws.pop_back();
    } else ++i;
  }
}

struct DevBufs {
  std::vector<void*> ptrs;
  ~DevBufs() {
    std::lock_guard<std::mutex> lk(g_ws_mu);
    for (void* p : ptrs)
      for (auto& b : g_ws) if (b.ptr == p) b.in_use = false;
  }
  template <typename T>
  int alloc(T** out, size_t count) {
    const size_t bytes = sizeof(T) * (count ? count : 1);
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(g_ws_mu);
    WsBlock* best = nullptr;
    for (auto& b : g_ws)
      if (!b.in_use && b.device == dev && b.bytes >= bytes && b.bytes <= 2 * bytes + 4096 && (!best || b.bytes < best->bytes)) best = &b;
    if (best) { best->in_use = true; ptrs.push_back(best->ptr); *out = (T*)best->ptr; return EBM_OK; }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {   // give cached blocks back and retry once
      cudaGetLastError();
      ws_release_free_blocks(dev);
      e = cudaMalloc(&p, bytes);
    }
    if (e != cudaSuccess) { cudaGetLastError(); ebm_set_error("cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e)); return EBM_ERR_OOM; }
    g_ws.push_back(WsBlock{dev, p, bytes, true});
    ptrs.push_back(p);
    *out = (T*)p;
    return EBM_OK;
  }
};

// Owns the private stream of a host entry point.  Its destructor drains the stream before destroying it: an error
// path must not hand the workspace blocks back (DevBufs, destroyed afterwards) while kernels or copies still use them.
struct StreamGuard {
  cudaStream_t s;
  ~StreamGuard() { cudaStreamSynchronize(s); cudaStreamDestroy(s); cudaGetLastError(); }
};

// host [rows][cols] -> device [cols][rows] via a staging buffer
int upload_transposed(const double* host, double* stage, double* dst, long long rows, long long cols, cudaStream_t s) {
  EBM_CUDA_TRY(cudaMemcpyAsync(stage, host, sizeof(double) * rows * cols, cudaMemcpyHostToDevice, s));
  return ebm_launch_transpose(stage, dst, rows, cols, s);
}
int download_transposed(double* host, double* stage, const double* src, long long rows_src, long long cols_src, cudaStream_t s) {
  EBM_TRY(ebm_launch_transpose(src, stage, rows_src, cols_src, s));
  EBM_CUDA_TRY(cudaMemcpyAsync(host, stage, sizeof(double) * rows_src * cols_src, cudaMemcpyDeviceToHost, s));
  return EBM_OK;
}

// The classic kernels: the literal-order one on request; up to kClassicUniformMaxNx cells the table-driven kernel
// (the 32-member groups whose table-building parameters agree) and its per-member-coefficient instance (the other
// groups); larger grids the band kernel.
int launch_classic(const ClassicKArgs& a, bool strict, cudaStream_t stream) {
  if (strict) return ebm_launch_classic_strict(a, stream);
  if (a.nx > kClassicUniformMaxNx) return ebm_launch_classic_bands(a, stream);
  EBM_TRY(ebm_launch_classic_uniform(a, stream));
  return ebm_launch_classic_general(a, stream);
}

// The opening steps of ebm_classic_run_device and ebm_miz_run_device after their pointer checks: device, the
// field-output check, the grid tables and the argument-block fields both models name alike.  The caller holds the
// DeviceRestore.
template <typename KArgs, typename DeviceArgs>
int device_prologue(const ebm_grid_t* grid, const DeviceArgs* args, const ebm_options_t& opt, KArgs* a,
                    cudaStream_t stream) {
  if (args->nmem < 1) { ebm_set_error("nmem must be >= 1"); return EBM_ERR_INVALID; }
  EBM_TRY(select_device(opt));
  if ((args->seasonal || args->raw) && opt.field_stride <= 0) { ebm_set_error("seasonal/raw output requested but field_stride == 0"); return EBM_ERR_INVALID; }
  memset(a, 0, sizeof(*a));
  EBM_TRY(get_tables(grid, &a->g, stream));
  a->nx = grid->nx; a->nt = grid->nt; a->dur = grid->dur; a->nmem = args->nmem;
  a->winter_inx = grid->winter_inx; a->summer_inx = grid->summer_inx;
  a->lastonly = opt.lastonly; a->field_stride = opt.field_stride;
  a->start_year = opt.start_year > 0 ? opt.start_year : 0;
  return EBM_OK;
}

// the run in launches of opt.years_per_launch years
template <typename KArgs, typename Launch>
int launch_years(KArgs a, const ebm_grid_t* grid, const ebm_options_t& opt, Launch launch) {
  const int ypl = opt.years_per_launch > 0 ? opt.years_per_launch : grid->dur;
  for (int y0 = 0; y0 < grid->dur; y0 += ypl) {
    a.year0 = y0;
    a.nyears = (y0 + ypl <= grid->dur) ? ypl : grid->dur - y0;
    EBM_TRY(launch(a));
  }
  return EBM_OK;
}

// Lanes of a warp are members: members in different regimes (snowball next to ice free) make every warp take both code
// paths.  Sort the members by the regime of their initial state (stable: the caller's order survives within a regime);
// the kernels write every output row at the member's original index (member_index).
std::vector<long long> classic_member_order(const ebm_grid_t* grid, long long nmem, const EbmHostRun& run,
                                            const ebm_options_t& opt) {
  std::vector<long long> perm;
  if (opt.strict || nmem <= 32) return perm;
  // primary key: the set of table-building parameters (D, S0, S2, a0, a2, cg, tau -- the table-driven kernel needs
  // them uniform over 32-member groups), numbered in order of first appearance; secondary: regime of the initial
  // state.  Ensembles made of many distinct parameter sets (a pure sweep over D) are left in the caller's order
  // within each regime.
  const int nx = grid->nx;
  std::map<std::array<double, kClassicNTablePar>, int> sets;
  std::vector<int> key((size_t)nmem);
  bool many_sets = false;
  for (long long m = 0; m < nmem; ++m) {
    int sid = 0;
    if (!many_sets) {
      std::array<double, kClassicNTablePar> tp;
      for (int q = 0; q < kClassicNTablePar; ++q) tp[q] = run.par[m * EBM_CLASSIC_NPAR + ebm_classic_table_par(q)];
      auto it = sets.find(tp);
      if (it == sets.end()) it = sets.emplace(tp, (int)sets.size()).first;
      sid = it->second;
      if ((long long)sets.size() * 32 > nmem) many_sets = true;   // groups cannot be made uniform anyway
    }
    key[m] = sid * 4 + ebm_classic_regime(run.init[0] + m * nx, nx);
  }
  if (many_sets) for (long long m = 0; m < nmem; ++m) key[m] &= 3;
  if (std::is_sorted(key.begin(), key.end())) return perm;
  perm.resize((size_t)nmem);
  for (long long m = 0; m < nmem; ++m) perm[m] = m;
  std::stable_sort(perm.begin(), perm.end(), [&](long long a, long long b) { return key[a] < key[b]; });
  return perm;
}

// The per-model step of a host run: the public device entry point on the run's device arrays.
int call_classic_device(const ebm_grid_t* grid, long long nmem, const EbmHostRun& dev, const long long* member_index,
                        const ebm_options_t& opt, cudaStream_t stream) {
  const ebm_classic_device_args_t da = {nmem, dev.par, dev.forc, dev.fin[0], dev.fin[1], dev.diag, dev.seasonal, dev.raw,
                                        dev.flags, (const int64_t*)member_index};
  return ebm_classic_run_device(grid, &da, &opt, stream);
}

int call_miz_device(const ebm_grid_t* grid, long long nmem, const EbmHostRun& dev, const long long*,
                    const ebm_options_t& opt, cudaStream_t stream) {
  const ebm_miz_device_args_t da = {nmem, dev.par, dev.forc, dev.fin[0], dev.fin[1], dev.fin[2], dev.fin[3], dev.fin[4],
                                    dev.fin[5], dev.diag, dev.seasonal, dev.raw, dev.newton_iters, dev.nonconv, dev.flags};
  return ebm_miz_run_device(grid, &da, &opt, stream);
}

}  // namespace

// ----------------------------------------------------------------------------- host-buffer runs
ebm_options_t default_options() {
  ebm_options_t o;
  memset(&o, 0, sizeof(o));
  o.device = -1; o.lastonly = 1;
  return o;
}

int ebm_classic_regime(const double* E, int nx) {
  int ice = 0;
  for (int j = 0; j < nx; ++j) ice += E[j] < 0.0;
  return ice == 0 ? 0 : (ice == nx ? 2 : 1);
}

int ebm_run_host(const ebm_grid_t* grid, long long nmem, const EbmHostRun& run, const ebm_options_t* opt_in,
                 EbmDiagHook* diag_hook) {
  EBM_TRY(check_grid(grid));
  ebm_options_t opt = opt_in ? *opt_in : default_options();
  DeviceRestore _dr;
  EBM_TRY(select_device(opt));
  if ((run.seasonal || run.raw) && opt.field_stride <= 0) { ebm_set_error("seasonal/raw output requested but field_stride == 0"); return EBM_ERR_INVALID; }
  const int nx = grid->nx, nt = grid->nt, dur = grid->dur;
  const long long nsel = ebm_nsel(opt, nmem), nraw = ebm_nraw(nt, dur, opt.lastonly);
  const std::vector<long long> perm = run.order ? run.order(grid, nmem, run, opt) : std::vector<long long>();
  cudaStream_t s;
  EBM_CUDA_TRY(cudaStreamCreate(&s));
  DevBufs B;                 // declared first: destroyed last
  StreamGuard sg{s};         // ... after the stream has drained (error paths return without a synchronise of their own)
  double *stage, *dpar, *dforc;
  long long* dperm = nullptr;
  EBM_TRY(B.alloc(&stage, (size_t)nmem * std::max(nx, run.npar)));
  if (!perm.empty()) {
    EBM_TRY(B.alloc(&dperm, (size_t)nmem));
    EBM_CUDA_TRY(cudaMemcpyAsync(dperm, perm.data(), sizeof(long long) * nmem, cudaMemcpyHostToDevice, s));
  }
  auto upload = [&](const double* host, double* dst, long long cols) -> int {   // host [nmem][cols] -> device [cols][slots]
    if (!dperm) return upload_transposed(host, stage, dst, nmem, cols, s);
    EBM_CUDA_TRY(cudaMemcpyAsync(stage, host, sizeof(double) * nmem * cols, cudaMemcpyHostToDevice, s));
    return ebm_launch_gather_transpose(stage, dst, nmem, cols, dperm, 0, s);
  };
  auto download = [&](double* host, const double* src) -> int {      // device [nx][slots] -> host [nmem][nx], original order
    if (!dperm) return download_transposed(host, stage, src, nx, nmem, s);
    EBM_TRY(ebm_launch_gather_transpose(src, stage, nmem, nx, dperm, 1, s));
    EBM_CUDA_TRY(cudaMemcpyAsync(host, stage, sizeof(double) * nmem * nx, cudaMemcpyDeviceToHost, s));
    return EBM_OK;
  };
  EbmHostRun dev = run;   // the same run on device arrays
  EBM_TRY(B.alloc(&dpar, (size_t)nmem * run.npar));
  EBM_TRY(B.alloc(&dforc, (size_t)nmem * EBM_NFORCING));
  EBM_TRY(upload(run.par, dpar, run.npar));
  EBM_TRY(upload(run.forc, dforc, EBM_NFORCING));
  dev.par = dpar; dev.forc = dforc;
  for (int q = 0; q < run.nstate; ++q) {
    EBM_TRY(B.alloc(&dev.fin[q], (size_t)nmem * nx));
    if (run.init[q]) EBM_TRY(upload(run.init[q], dev.fin[q], nx));
    else EBM_CUDA_TRY(cudaMemsetAsync(dev.fin[q], 0, sizeof(double) * nmem * nx, s));
    dev.init[q] = dev.fin[q];
  }
  // outputs: allocated when wanted; fields and diagnostics NaN (what the reference leaves undef), counters zero
  const size_t ndiag = ebm_diag_offset(nmem, dur, 0, 0);
  const size_t nseas = ebm_seasonal_offset(nsel, dur, 0, 0, run.nvar, nx);
  const size_t nrawn = ebm_raw_offset(nsel, nraw, 0, run.nvar, nx);
  auto nan_filled = [&](double** d, bool wanted, size_t n) -> int {
    *d = nullptr;
    if (!wanted) return EBM_OK;
    EBM_TRY(B.alloc(d, n));
    return ebm_launch_fill(*d, (long long)n, NAN, s);
  };
  auto zeroed = [&](auto** d, bool wanted) -> int {
    *d = nullptr;
    if (!wanted) return EBM_OK;
    EBM_TRY(B.alloc(d, (size_t)nmem));
    EBM_CUDA_TRY(cudaMemsetAsync(*d, 0, sizeof(**d) * nmem, s));
    return EBM_OK;
  };
  EBM_TRY(nan_filled(&dev.diag, run.diag || diag_hook, ndiag));
  EBM_TRY(nan_filled(&dev.seasonal, run.seasonal, nseas));
  EBM_TRY(nan_filled(&dev.raw, run.raw, nrawn));
  EBM_TRY(zeroed(&dev.newton_iters, run.newton_iters));
  EBM_TRY(zeroed(&dev.nonconv, run.nonconv));
  EBM_TRY(zeroed(&dev.flags, run.flags));
  EBM_TRY(run.run_device(grid, nmem, dev, dperm, opt, s));
  auto fetch = [&](auto* host, const auto* d, size_t n) -> int {
    if (host) EBM_CUDA_TRY(cudaMemcpyAsync(host, d, sizeof(*host) * n, cudaMemcpyDeviceToHost, s));
    return EBM_OK;
  };
  if (diag_hook) EBM_TRY(diag_hook->consume(dev.diag, ndiag, s));
  else EBM_TRY(fetch(run.diag, dev.diag, ndiag));
  EBM_TRY(fetch(run.seasonal, dev.seasonal, nseas));
  EBM_TRY(fetch(run.raw, dev.raw, nrawn));
  EBM_TRY(fetch(run.newton_iters, dev.newton_iters, (size_t)nmem));
  EBM_TRY(fetch(run.nonconv, dev.nonconv, (size_t)nmem));
  EBM_TRY(fetch(run.flags, dev.flags, (size_t)nmem));
  for (int q = 0; q < run.nstate; ++q)
    if (run.fin[q]) EBM_TRY(download(run.fin[q], dev.fin[q]));
  EBM_CUDA_TRY(cudaStreamSynchronize(s));   // the copies above share the stream: one wait covers them all
  return EBM_OK;
}

EbmHostRun ebm_classic_host_run(const ebm_classic_params_t* par, const ebm_forcing_t* forc, const double* E0,
                                const double* Tg0, const ebm_classic_outputs_t* out) {
  return {EBM_CLASSIC_NPAR, EBM_CLASSIC_NVAR, 2, (const double*)par, (const double*)forc, {E0, Tg0},
          out->diag, out->seasonal, out->raw, {out->E_final, out->Tg_final}, nullptr, nullptr, out->flags,
          call_classic_device, classic_member_order};
}

EbmHostRun ebm_miz_host_run(const ebm_miz_params_t* par, const ebm_forcing_t* forc, const double* Ei0, const double* Ew0,
                            const double* h0, const double* D0, const double* phi0, const double* T0guess,
                            const ebm_miz_outputs_t* out) {
  return {EBM_MIZ_NPAR, EBM_MIZ_NVAR, 6, (const double*)par, (const double*)forc, {Ei0, Ew0, h0, D0, phi0, T0guess},
          out->diag, out->seasonal, out->raw,
          {out->Ei_final, out->Ew_final, out->h_final, out->D_final, out->phi_final, out->T0_final},
          out->newton_iters, out->nonconv, out->flags, call_miz_device, nullptr};
}

extern "C" int32_t ebm_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_cache_mu);
  int cur = 0;
  cudaGetDevice(&cur);
  for (auto& e : g_cache) { cudaSetDevice(e.device); cudaFree(e.dev); }
  g_cache.clear();
  {
    std::lock_guard<std::mutex> lk2(g_ws_mu);
    ws_release_free_blocks(-1);
  }
  cudaSetDevice(cur);
  cudaGetLastError();
  ebm_multi_shutdown();
  return EBM_OK;
}

extern "C" int32_t ebm_transpose_device(const double* src, double* dst, int64_t rows, int64_t cols, void* stream) {
  if (!src || !dst || rows < 0 || cols < 0) { ebm_set_error("transpose: bad arguments"); return EBM_ERR_INVALID; }
  return ebm_launch_transpose(src, dst, rows, cols, (cudaStream_t)stream);
}

extern "C" int32_t ebm_fp64_peak(int32_t device, double* tflops, double* sm_clock_mhz_est) {
  ebm_options_t o = default_options();
  o.device = device;
  DeviceRestore _dr;
  EBM_TRY(select_device(o));
  return ebm_run_fp64_peak(-1, tflops, sm_clock_mhz_est);
}

// ----------------------------------------------------------------------------- classic
extern "C" int32_t ebm_classic_run_device(const ebm_grid_t* grid, const ebm_classic_device_args_t* args,
                                          const ebm_options_t* opt_in, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  EBM_TRY(check_grid(grid));
  if (!args || !args->par || !args->forc || !args->E || !args->Tg) { ebm_set_error("classic_run_device: par, forc, E, Tg must be non-NULL"); return EBM_ERR_INVALID; }
  const ebm_options_t opt = opt_in ? *opt_in : default_options();
  DeviceRestore _dr;
  ClassicKArgs a;
  EBM_TRY(device_prologue(grid, args, opt, &a, stream));
  if (opt.step_limit > 0) { ebm_set_error("step_limit is only supported by the MIZ path"); return EBM_ERR_UNSUPPORTED; }
  if (opt.classic_stencil == 1) {   // classic on non-uniform grids: the generic flux-form stencil in kappa
    a.g.lam_lo = a.g.glam_lo; a.g.lam_hi = a.g.glam_hi;
  } else if (opt.classic_stencil != 0) {
    ebm_set_error("classic_stencil must be 0 (get_diffop, as the reference) or 1 (generic flux-form stencil)");
    return EBM_ERR_INVALID;
  }
  a.par = args->par; a.forc = args->forc; a.E = args->E; a.Tg = args->Tg;
  a.diag = args->diag; a.seasonal = args->seasonal; a.raw = args->raw; a.flags = args->flags;
  a.orig = (const long long*)args->member_index;
  a.dbg = getenv("EBM_DBG") ? atoi(getenv("EBM_DBG")) : 0;
  {   // |dE| per step <= dt * |alpha S - A + f - B T + Fb| ~ dt * 300: cells above 512 dt stay open water for a step
    const double ethr = 512.0 / (double)grid->nt;
    long long bits; memcpy(&bits, &ethr, sizeof(bits));
    a.hthr = (int)(bits >> 32);
  }
  // ---- launch-uniform parameters (a forcing sweep such as C4: members differ in forcing and initial state only).  The
  // member constants then travel in the kernel argument block and are constant-bank operands of the FP64 instructions;
  // the 26 registers they otherwise occupy go to instruction-level parallelism (classic_uniform.cu, UPAR).  The host
  // derives them with the same IEEE expressions the kernels evaluate per member, so the results are bit-identical.
  DevBufs upar_bufs;
  if (!opt.strict && a.nx <= kClassic8BandMaxNx && !getenv("EBM_NO_UPAR")) {
    double* dhead = nullptr; int* ddiff = nullptr;
    EBM_TRY(upar_bufs.alloc(&dhead, EBM_CLASSIC_NPAR));
    EBM_TRY(upar_bufs.alloc(&ddiff, 1));
    EBM_TRY(ebm_launch_par_uniform(a.par, EBM_CLASSIC_NPAR, a.nmem, dhead, ddiff, stream));
    int differs = 1;
    EBM_CUDA_TRY(cudaMemcpyAsync(&differs, ddiff, sizeof(int), cudaMemcpyDeviceToHost, stream));
    EBM_CUDA_TRY(cudaMemcpyAsync(a.u.par, dhead, sizeof(double) * EBM_CLASSIC_NPAR, cudaMemcpyDeviceToHost, stream));
    EBM_CUDA_TRY(cudaStreamSynchronize(stream));
    if (!differs) {
      const double* p = a.u.par;   // D A B cw S0 S1 S2 a0 a2 ai Fb k Lf cg tau
      ClassicUPar& u = a.u;
      u.dt = 1.0 / a.nt;
      u.cg_tau = p[13] / p[14]; u.dt_tau = u.dt / p[14];
      u.A = p[1]; u.Fb = p[10]; u.ai = p[9]; u.M = p[2] + u.cg_tau; u.kLf = p[11] * p[12];
      u.inv_cw = 1.0 / p[3]; u.dttau_cw = u.dt_tau * u.inv_cw; u.dc = u.dt_tau * u.cg_tau;
      u.inv_nt = 1.0 / a.nt; u.inv_Lf = 1.0 / p[12];
      a.upar = 1;
    }
  }
  // ---- wave balancing.  A CTA integrates 16 members for the whole run; the device holds `slots` CTAs at a time.
  // 8192 members (the 8-GPU share of the 65 536-member sweep) are 512 CTAs on 444 slots: one launch runs them as
  // two waves, the second 15 % full.  Cut instead into 8 ranges of CTAs on 8 streams, each advancing in chunks of
  // years: whenever a range finishes a chunk its slots go to whichever range is waiting, and the makespan
  // approaches work / slots.  Results are bit-identical (a CTA's arithmetic does not depend on the launch shape).
  if (!opt.strict && a.nx <= kClassic8BandMaxNx && !getenv("EBM_NO_WAVE_BALANCE")) {
    const long long blocks = (a.nmem + 15) / 16;
    const long long slots = ebm_classic_uniform_slots();
    const long long waves = slots > 0 ? (blocks + slots - 1) / slots : 0;
    if (slots > 0 && blocks > slots && blocks <= 12 * slots && grid->dur >= 8 &&
        (double)(waves * slots) > 1.08 * (double)blocks) {
      constexpr int S = 8, nchunk = 16;   // measured flat between 4 x 20 and 16 x 40 (DESIGN.md)
      const int chunk = std::min(opt.years_per_launch > 0 ? opt.years_per_launch : grid->dur, std::max(1, grid->dur / nchunk));
      cudaEvent_t fork;
      EBM_CUDA_TRY(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
      EBM_CUDA_TRY(cudaEventRecord(fork, stream));
      int rc = EBM_OK;
      cudaStream_t aux[S];
      cudaEvent_t done[S];
      int made = 0;
      for (; made < S && rc == EBM_OK; ++made) {
        if (cudaStreamCreateWithFlags(&aux[made], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&done[made], cudaEventDisableTiming) != cudaSuccess) { rc = EBM_ERR_CUDA; ebm_set_error("wave balancing: stream creation failed"); break; }
        if (cudaStreamWaitEvent(aux[made], fork, 0) != cudaSuccess) rc = EBM_ERR_CUDA;
      }
      for (int y0 = 0; y0 < grid->dur && rc == EBM_OK; y0 += chunk) {
        for (int q = 0; q < made && rc == EBM_OK; ++q) {
          ClassicKArgs b = a;
          b.year0 = y0;
          b.nyears = std::min(chunk, grid->dur - y0);
          b.block0 = blocks * q / made;
          b.nblocks = blocks * (q + 1) / made - b.block0;
          if (b.nblocks <= 0) continue;
          rc = launch_classic(b, false, aux[q]);
        }
      }
      for (int q = 0; q < made; ++q) {   // join (and release: destruction is deferred until the work has drained)
        cudaEventRecord(done[q], aux[q]);
        cudaStreamWaitEvent(stream, done[q], 0);
        cudaEventDestroy(done[q]);
        cudaStreamDestroy(aux[q]);
      }
      cudaEventDestroy(fork);
      return rc;
    }
  }
  return launch_years(a, grid, opt, [&](const ClassicKArgs& b) { return launch_classic(b, opt.strict != 0, stream); });
}

extern "C" int32_t ebm_classic_run(const ebm_grid_t* grid, int64_t nmem, const ebm_classic_params_t* par,
                                   const ebm_forcing_t* forc, const double* E0, const double* Tg0,
                                   const ebm_options_t* opt_in, ebm_classic_outputs_t* out) {
  EBM_TRY(check_grid(grid));
  if (nmem < 1 || !par || !forc || !E0 || !Tg0 || !out) { ebm_set_error("classic_run: nmem >= 1 and par, forc, E0, Tg0, out must be non-NULL"); return EBM_ERR_INVALID; }
  return ebm_run_host(grid, nmem, ebm_classic_host_run(par, forc, E0, Tg0, out), opt_in, nullptr);
}

extern "C" int32_t ebm_classic_step_debug(const ebm_grid_t* grid, const ebm_classic_params_t* par, int32_t ti, double f,
                                          double* E, double* Tg, double* T, double* h, int32_t which, double* debug_out) {
  EBM_TRY(check_grid(grid));
  if (!par || !E || !Tg || !T || !h) { ebm_set_error("classic_step: NULL argument"); return EBM_ERR_INVALID; }
  if (ti < 1 || ti > grid->nt) { ebm_set_error("classic_step: ti=%d outside 1..nt", ti); return EBM_ERR_INVALID; }
  if (which < EBM_DEBUG_NONE || which > EBM_DEBUG_MASK || (which != EBM_DEBUG_NONE && !debug_out)) {
    ebm_set_error("classic_step_debug: `which` must be one of EBM_DEBUG_* (the device cannot evaluate a debug::Expr) and debug_out non-NULL");
    return which < EBM_DEBUG_NONE || which > EBM_DEBUG_MASK ? EBM_ERR_UNSUPPORTED : EBM_ERR_INVALID;
  }
  ebm_options_t opt = default_options();
  DeviceRestore _dr;
  EBM_TRY(select_device(opt));
  const int nx = grid->nx;
  EbmGridTables tabs;
  EBM_TRY(get_tables(grid, &tabs, 0));
  DevBufs B;
  double* d = nullptr;
  EBM_TRY(B.alloc(&d, (size_t)EBM_CLASSIC_NPAR + 5 * nx));
  double *dpar = d, *dE = d + EBM_CLASSIC_NPAR, *dTg = dE + nx, *dT = dTg + nx, *dh = dT + nx, *ddbg = dh + nx;
  EBM_CUDA_TRY(cudaMemcpy(dpar, par, sizeof(double) * EBM_CLASSIC_NPAR, cudaMemcpyHostToDevice));
  EBM_CUDA_TRY(cudaMemcpy(dE, E, sizeof(double) * nx, cudaMemcpyHostToDevice));
  EBM_CUDA_TRY(cudaMemcpy(dTg, Tg, sizeof(double) * nx, cudaMemcpyHostToDevice));
  EBM_TRY(ebm_launch_classic_single_step(tabs, dpar, ti, f, dE, dTg, dT, dh, 0, which, which != EBM_DEBUG_NONE ? ddbg : nullptr));
  EBM_CUDA_TRY(cudaMemcpy(E, dE, sizeof(double) * nx, cudaMemcpyDeviceToHost));
  EBM_CUDA_TRY(cudaMemcpy(Tg, dTg, sizeof(double) * nx, cudaMemcpyDeviceToHost));
  EBM_CUDA_TRY(cudaMemcpy(T, dT, sizeof(double) * nx, cudaMemcpyDeviceToHost));
  EBM_CUDA_TRY(cudaMemcpy(h, dh, sizeof(double) * nx, cudaMemcpyDeviceToHost));
  if (which != EBM_DEBUG_NONE) EBM_CUDA_TRY(cudaMemcpy(debug_out, ddbg, sizeof(double) * nx, cudaMemcpyDeviceToHost));
  return EBM_OK;
}

extern "C" int32_t ebm_classic_step(const ebm_grid_t* grid, const ebm_classic_params_t* par, int32_t ti, double f,
                                    double* E, double* Tg, double* T, double* h) {
  return ebm_classic_step_debug(grid, par, ti, f, E, Tg, T, h, EBM_DEBUG_NONE, nullptr);
}

// ----------------------------------------------------------------------------- MIZ
extern "C" int32_t ebm_miz_run_device(const ebm_grid_t* grid, const ebm_miz_device_args_t* args,
                                      const ebm_options_t* opt_in, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  EBM_TRY(check_grid(grid));
  if (!args || !args->par || !args->forc || !args->Ei || !args->Ew || !args->h || !args->D || !args->phi || !args->T0) {
    ebm_set_error("miz_run_device: par, forc and the six state arrays must be non-NULL");
    return EBM_ERR_INVALID;
  }
  const ebm_options_t opt = opt_in ? *opt_in : default_options();
  DeviceRestore _dr;
  MizKArgs a;
  EBM_TRY(device_prologue(grid, args, opt, &a, stream));
  a.maxit = opt.newton_maxit > 0 ? opt.newton_maxit : 100;
  a.tol = opt.newton_tol > 0.0 ? opt.newton_tol : 1e-8;
  a.step_limit = opt.step_limit > 0 ? opt.step_limit : 0;
  a.par = args->par; a.forc = args->forc;
  a.Ei = args->Ei; a.Ew = args->Ew; a.h = args->h; a.D = args->D; a.phi = args->phi; a.T0 = args->T0;
  a.diag = args->diag; a.seasonal = args->seasonal; a.raw = args->raw;
  a.newton_iters = (long long*)args->newton_iters; a.nonconv = (long long*)args->nonconv; a.flags = args->flags;
  return launch_years(a, grid, opt, [&](const MizKArgs& b) { return ebm_launch_miz(b, opt.strict, stream); });
}

extern "C" int32_t ebm_miz_run(const ebm_grid_t* grid, int64_t nmem, const ebm_miz_params_t* par,
                               const ebm_forcing_t* forc, const double* Ei0, const double* Ew0, const double* h0,
                               const double* D0, const double* phi0, const double* T0guess,
                               const ebm_options_t* opt_in, ebm_miz_outputs_t* out) {
  EBM_TRY(check_grid(grid));
  if (nmem < 1 || !par || !forc || !Ei0 || !Ew0 || !h0 || !D0 || !phi0 || !out) { ebm_set_error("miz_run: NULL argument or nmem < 1"); return EBM_ERR_INVALID; }
  return ebm_run_host(grid, nmem, ebm_miz_host_run(par, forc, Ei0, Ew0, h0, D0, phi0, T0guess, out), opt_in, nullptr);
}

extern "C" int32_t ebm_miz_step(const ebm_grid_t* grid, const ebm_miz_params_t* par, int32_t ti, double f,
                                double* Ei, double* Ew, double* h, double* D, double* phi, double* T0,
                                double* vars_out, int32_t* newton_iters) {
  EBM_TRY(check_grid(grid));
  if (!par || !Ei || !Ew || !h || !D || !phi || !T0 || !vars_out) { ebm_set_error("miz_step: NULL argument"); return EBM_ERR_INVALID; }
  if (ti < 1 || ti > grid->nt) { ebm_set_error("miz_step: ti=%d outside 1..nt", ti); return EBM_ERR_INVALID; }
  ebm_options_t opt = default_options();
  DeviceRestore _dr;
  EBM_TRY(select_device(opt));
  const int nx = grid->nx;
  EbmGridTables tabs;
  EBM_TRY(get_tables(grid, &tabs, 0));
  DevBufs B;
  double* d = nullptr; long long* dit = nullptr;
  EBM_TRY(B.alloc(&d, (size_t)EBM_MIZ_NPAR + (6 + EBM_MIZ_NVAR) * (size_t)nx));
  EBM_TRY(B.alloc(&dit, 1));
  double* dpar = d; double* st6 = d + EBM_MIZ_NPAR; double* dvars = st6 + 6 * nx;
  double* host6[6] = {Ei, Ew, h, D, phi, T0};
  EBM_CUDA_TRY(cudaMemcpy(dpar, par, sizeof(double) * EBM_MIZ_NPAR, cudaMemcpyHostToDevice));
  for (int q = 0; q < 6; ++q) EBM_CUDA_TRY(cudaMemcpy(st6 + q * nx, host6[q], sizeof(double) * nx, cudaMemcpyHostToDevice));
  EBM_CUDA_TRY(cudaMemset(dit, 0, sizeof(long long)));
  EBM_TRY(ebm_launch_miz_single_step(tabs, dpar, ti, f, 1e-8, 100, st6, st6 + nx, st6 + 2 * nx, st6 + 3 * nx, st6 + 4 * nx,
                                     st6 + 5 * nx, dvars, dit, 0));
  for (int q = 0; q < 6; ++q) EBM_CUDA_TRY(cudaMemcpy(host6[q], st6 + q * nx, sizeof(double) * nx, cudaMemcpyDeviceToHost));
  EBM_CUDA_TRY(cudaMemcpy(vars_out, dvars, sizeof(double) * EBM_MIZ_NVAR * nx, cudaMemcpyDeviceToHost));
  long long hit = 0;
  EBM_CUDA_TRY(cudaMemcpy(&hit, dit, sizeof(long long), cudaMemcpyDeviceToHost));
  if (newton_iters) *newton_iters = (int32_t)hit;
  return EBM_OK;
}
