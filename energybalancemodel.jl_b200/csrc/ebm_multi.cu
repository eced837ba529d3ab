// ebm_multi.cu -- one call, several GPUs: ebm_classic_run_multi / ebm_miz_run_multi (include/ebm_cuda.h).
//
// Members of an ensemble are independent (no reference code path couples them: src/infrastructure.jl:615-636 runs one
// member), so the time-stepping path shards with no data-path collective.  Single process, one host thread and one
// stream per GPU (SURVEY.md 8b "Threading"):
//   * members are dealt to the GPUs in packets of 32 after a stable sort by what they cost (classic: the regime of the
//     initial state) -- a contiguous cut of an ensemble ordered by a physical parameter hands one GPU all the expensive
//     members (round-1 VERDICT: the rank holding F = -20... set the step time);
//   * every thread runs the host run of ebm_classic_run / ebm_miz_run (ebm_run_host) on its members and scatters the
//     rows it gets back to the caller's arrays at the members' original indices;
//   * diagnostics: with multi->diag_device < 0 every GPU copies its own rows to the caller's host buffer; with
//     diag_device >= 0 the caller's `diag` is DEVICE memory on that GPU and the other GPUs send their rows there over
//     NVLink: each thread passes its host run a GatherHook, which takes the device-resident rows and runs ncclSend /
//     ncclRecv on communicators this library owns (ncclCommInitAll, created lazily per device set, destroyed by
//     ebm_shutdown).  NCCL is bound with dlopen("libnccl.so.2") at first use, so the library has no link-time
//     dependency on it and shares the copy a host process (e.g. torch) has already loaded;
//   * field outputs (seasonal / raw): each GPU integrates its field-selected members once more (FieldSel).
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "ebm_internal.cuh"

namespace {

// ----------------------------------------------------------------------------- NCCL, bound at run time
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  bool ok = false;
};
std::mutex g_nccl_mu;
NcclApi g_nccl;
std::map<std::vector<int>, std::vector<ncclComm_t>> g_comms;   // device list -> one communicator per device

bool load_nccl(std::string* why) {   // caller holds g_nccl_mu
  if (g_nccl.ok) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    g_nccl.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.handle) break;
  }
  if (!g_nccl.handle) { *why = std::string("dlopen(libnccl.so.2) failed: ") + dlerror(); return false; }
#define EBM_SYM(field, name) \
  *(void**)(&g_nccl.field) = dlsym(g_nccl.handle, name); \
  if (!g_nccl.field) { *why = std::string("libnccl lacks ") + name; return false; }
  EBM_SYM(CommInitAll, "ncclCommInitAll")
  EBM_SYM(CommDestroy, "ncclCommDestroy")
  EBM_SYM(GetErrorString, "ncclGetErrorString")
  EBM_SYM(Send, "ncclSend")
  EBM_SYM(Recv, "ncclRecv")
  EBM_SYM(GroupStart, "ncclGroupStart")
  EBM_SYM(GroupEnd, "ncclGroupEnd")
#undef EBM_SYM
  g_nccl.ok = true;
  return true;
}

int get_comms(const std::vector<int>& devs, std::vector<ncclComm_t>* out) {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  std::string why;
  if (!load_nccl(&why)) { ebm_set_error("NCCL is not available: %s", why.c_str()); return EBM_ERR_UNSUPPORTED; }
  auto it = g_comms.find(devs);
  if (it == g_comms.end()) {
    std::vector<ncclComm_t> comms(devs.size());
    const ncclResult_t r = g_nccl.CommInitAll(comms.data(), (int)devs.size(), devs.data());
    if (r != ncclSuccess) { ebm_set_error("ncclCommInitAll failed: %s", g_nccl.GetErrorString(r)); return EBM_ERR_CUDA; }
    it = g_comms.emplace(devs, comms).first;
  }
  *out = it->second;
  return EBM_OK;
}

// ----------------------------------------------------------------------------- dealing
// packets of `packet` members, round-robin over the devices, after a stable sort by `key` (may be empty)
std::vector<std::vector<long long>> deal(long long nmem, int ndev, const std::vector<int>& key, int packet) {
  std::vector<long long> order((size_t)nmem);
  std::iota(order.begin(), order.end(), 0LL);
  if (!key.empty()) std::stable_sort(order.begin(), order.end(), [&](long long a, long long b) { return key[a] < key[b]; });
  std::vector<std::vector<long long>> idx((size_t)ndev);
  const long long npk = (nmem + packet - 1) / packet;
  for (long long g = 0; g < npk; ++g) {
    auto& v = idx[(size_t)(g % ndev)];
    for (long long q = g * packet; q < std::min(nmem, (g + 1) * packet); ++q) v.push_back(order[(size_t)q]);
  }
  return idx;
}

template <typename T>
std::vector<T> take_rows(const T* src, const std::vector<long long>& idx, size_t rowlen) {
  std::vector<T> out(idx.size() * rowlen);
  for (size_t r = 0; r < idx.size(); ++r) memcpy(&out[r * rowlen], src + (size_t)idx[r] * rowlen, sizeof(T) * rowlen);
  return out;
}
template <typename T>
void put_rows(T* dst, const std::vector<T>& src, const std::vector<long long>& idx, size_t rowlen) {
  if (!dst) return;
  for (size_t r = 0; r < idx.size(); ++r) memcpy(dst + (size_t)idx[r] * rowlen, &src[r * rowlen], sizeof(T) * rowlen);
}

int resolve_devices(const ebm_multi_t* multi, std::vector<int>* devs) {
  const int avail = ebm_device_count();
  if (avail < 1) { ebm_set_error("no CUDA device available; libebm_cuda has no CPU fallback"); return EBM_ERR_CUDA; }
  int n = multi ? multi->ndevices : 0;
  if (n <= 0) n = avail;
  for (int q = 0; q < n; ++q) {
    const int d = (multi && multi->devices) ? multi->devices[q] : q;
    if (d < 0 || d >= avail) { ebm_set_error("multi: device %d out of range (%d devices)", d, avail); return EBM_ERR_INVALID; }
    if (std::find(devs->begin(), devs->end(), d) != devs->end()) { ebm_set_error("multi: device %d listed twice", d); return EBM_ERR_INVALID; }
    devs->push_back(d);
  }
  return EBM_OK;
}

// ----------------------------------------------------------------------------- diagnostics over NCCL
// Shared by the threads of one call: the root posts one ncclRecv per peer into a packed device buffer and scatters
// the rows to their final place in the caller's device array; the peers ncclSend their packed rows.
struct NcclGather {
  std::vector<ncclComm_t> comms;
  std::vector<std::vector<long long>> idx;   // members of every device
  int root = 0;                              // rank (position in the device list) that owns the caller's diag
  double* dst = nullptr;                     // caller's device array [nmem][rowlen] on the root device
  size_t rowlen = 0;
};

struct GatherHook : EbmDiagHook {
  NcclGather* g; int rank;
  GatherHook(NcclGather* g_, int rank_) : g(g_), rank(rank_) {}
  int consume(const double* ddiag, size_t count, cudaStream_t stream) override {
    const size_t mine = g->idx[(size_t)rank].size() * g->rowlen;
    if (count != mine) { ebm_set_error("multi: diagnostics of rank %d hold %zu values, expected %zu", rank, count, mine); return EBM_ERR_INVALID; }
    if (rank != g->root) {
      ncclResult_t r = g_nccl.GroupStart();
      if (r == ncclSuccess && mine) r = g_nccl.Send(ddiag, mine, ncclDouble, g->root, g->comms[(size_t)rank], stream);
      const ncclResult_t r2 = g_nccl.GroupEnd();
      if (r != ncclSuccess || r2 != ncclSuccess) { ebm_set_error("ncclSend failed: %s", g_nccl.GetErrorString(r != ncclSuccess ? r : r2)); return EBM_ERR_CUDA; }
      return EBM_OK;
    }
    // root: receive every peer's packed rows, then scatter (own rows included) by member index
    const int ndev = (int)g->idx.size();
    std::vector<double*> rbuf((size_t)ndev, nullptr);
    std::vector<long long*> ribuf((size_t)ndev, nullptr);
    int rc = EBM_OK;
    for (int p = 0; p < ndev && rc == EBM_OK; ++p) {
      const size_t n = g->idx[(size_t)p].size();
      if (!n) continue;
      if (p != rank && cudaMallocAsync(&rbuf[(size_t)p], sizeof(double) * n * g->rowlen, stream) != cudaSuccess) rc = EBM_ERR_OOM;
      if (rc == EBM_OK && cudaMallocAsync(&ribuf[(size_t)p], sizeof(long long) * n, stream) != cudaSuccess) rc = EBM_ERR_OOM;
      if (rc == EBM_OK && cudaMemcpyAsync(ribuf[(size_t)p], g->idx[(size_t)p].data(), sizeof(long long) * n, cudaMemcpyHostToDevice, stream) != cudaSuccess) rc = EBM_ERR_CUDA;
    }
    if (rc != EBM_OK) { cudaGetLastError(); ebm_set_error("multi: allocating the receive buffers failed"); }
    if (rc == EBM_OK) {
      ncclResult_t r = g_nccl.GroupStart();
      for (int p = 0; p < ndev && r == ncclSuccess; ++p)
        if (p != rank && rbuf[(size_t)p]) r = g_nccl.Recv(rbuf[(size_t)p], g->idx[(size_t)p].size() * g->rowlen, ncclDouble, p, g->comms[(size_t)rank], stream);
      const ncclResult_t r2 = g_nccl.GroupEnd();
      if (r != ncclSuccess || r2 != ncclSuccess) { ebm_set_error("ncclRecv failed: %s", g_nccl.GetErrorString(r != ncclSuccess ? r : r2)); rc = EBM_ERR_CUDA; }
    }
    for (int p = 0; p < ndev && rc == EBM_OK; ++p) {
      const size_t n = g->idx[(size_t)p].size();
      if (!n) continue;
      rc = ebm_launch_scatter_rows(p == rank ? ddiag : rbuf[(size_t)p], g->dst, (long long)n, (long long)g->rowlen, ribuf[(size_t)p], stream);
    }
    for (int p = 0; p < ndev; ++p) {
      if (rbuf[(size_t)p]) cudaFreeAsync(rbuf[(size_t)p], stream);
      if (ribuf[(size_t)p]) cudaFreeAsync(ribuf[(size_t)p], stream);
    }
    return rc;
  }
};

// Field outputs (seasonal / raw) of the members a device holds: the selected ones (global index % field_stride == 0) are
// integrated once more as a small sub-ensemble with field_stride = 1 -- a member's arithmetic does not depend on its
// neighbours, so the fields belong bit for bit to the run that produced the diagnostics -- and their rows land at
// global index / field_stride in the caller's arrays.
struct FieldSel {
  std::vector<long long> member, slot;   // the member's index, its row in the caller's field arrays
  FieldSel(const std::vector<long long>& ix, const ebm_options_t& opt, bool wanted) {
    if (!wanted) return;
    for (long long m : ix)
      if (ebm_field_selected(opt, m)) { member.push_back(m); slot.push_back(ebm_field_row(opt, m)); }
  }
  bool any() const { return !member.empty(); }
};

struct ThreadResult { int rc = EBM_OK; std::string err; };

// runs `work(rank)` on one thread per device; returns the first failure
template <typename F>
int run_threads(int ndev, F work) {
  std::vector<ThreadResult> res((size_t)ndev);
  std::vector<std::thread> th;
  for (int q = 0; q < ndev; ++q)
    th.emplace_back([&, q] {
      res[(size_t)q].rc = work(q);
      if (res[(size_t)q].rc != EBM_OK) res[(size_t)q].err = ebm_last_error();
    });
  for (auto& t : th) t.join();
  for (int q = 0; q < ndev; ++q)
    if (res[(size_t)q].rc != EBM_OK) { ebm_set_error("device thread %d: %s", q, res[(size_t)q].err.c_str()); return res[(size_t)q].rc; }
  return EBM_OK;
}

int setup_gather(const ebm_multi_t* multi, const std::vector<int>& devs, NcclGather* g, double* diag, size_t rowlen) {
  const int dd = multi ? multi->diag_device : -1;
  if (dd < 0 || !diag) return 0;   // host diagnostics
  const auto it = std::find(devs.begin(), devs.end(), dd);
  if (it == devs.end()) { ebm_set_error("multi: diag_device %d is not one of the devices of this call", dd); return EBM_ERR_INVALID; }
  g->root = (int)(it - devs.begin());
  g->dst = diag;
  g->rowlen = rowlen;
  const int rc = get_comms(devs, &g->comms);
  return rc == EBM_OK ? 1 : rc;
}

}  // namespace

void ebm_multi_shutdown() {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  if (g_nccl.ok)
    for (auto& kv : g_comms)
      for (ncclComm_t c : kv.second) g_nccl.CommDestroy(c);
  g_comms.clear();
}

namespace {

// The members `ix` of `run`: their input rows, copied into `rows`, and no output wanted.
struct MemberRows { std::vector<double> par, forc, init[6]; };
EbmHostRun members(const EbmHostRun& run, const std::vector<long long>& ix, int nx, MemberRows* rows) {
  EbmHostRun r = run;
  rows->par = take_rows(run.par, ix, (size_t)run.npar);
  rows->forc = take_rows(run.forc, ix, EBM_NFORCING);
  r.par = rows->par.data(); r.forc = rows->forc.data();
  for (int k = 0; k < run.nstate; ++k) {
    if (run.init[k]) rows->init[k] = take_rows(run.init[k], ix, (size_t)nx);
    r.init[k] = run.init[k] ? rows->init[k].data() : nullptr;
    r.fin[k] = nullptr;
  }
  r.diag = r.seasonal = r.raw = nullptr;
  r.newton_iters = r.nonconv = nullptr;
  r.flags = nullptr;
  return r;
}

// The per-device body of both models: every thread runs the host run of its members, puts their rows back at the
// members' original indices and reruns its field-selected members with field_stride = 1.  key: deal key (may be empty).
int run_multi(const ebm_grid_t* grid, long long nmem, const EbmHostRun& run, const std::vector<int>& key,
              const ebm_options_t* opt_in, const ebm_multi_t* multi) {
  std::vector<int> devs;
  int rc = resolve_devices(multi, &devs);
  if (rc != EBM_OK) return rc;
  const int ndev = (int)devs.size(), nx = grid->nx;
  const size_t rowlen = ebm_diag_offset(1, grid->dur, 0, 0);
  NcclGather g;
  g.idx = deal(nmem, ndev, key, (multi && multi->packet > 0) ? multi->packet : 32);
  const int nccl = setup_gather(multi, devs, &g, run.diag, rowlen);
  if (nccl < 0) return nccl;
  return run_threads(ndev, [&](int q) -> int {
    const auto& ix = g.idx[(size_t)q];
    const size_t n = ix.size();
    GatherHook hook(&g, q);
    if (n == 0) {   // no member for this GPU (fewer packets than devices): it still takes part in the exchange
      if (!nccl) return EBM_OK;
      EBM_CUDA_TRY(cudaSetDevice(devs[(size_t)q]));
      const int r0 = hook.consume(nullptr, 0, 0);
      EBM_CUDA_TRY(cudaStreamSynchronize(0));
      return r0;
    }
    MemberRows in;
    EbmHostRun r = members(run, ix, nx, &in);
    std::vector<double> fin[6], dg(run.diag && !nccl ? n * rowlen : 0);
    for (int k = 0; k < run.nstate; ++k) {
      if (run.fin[k]) fin[k].resize(n * nx);
      r.fin[k] = run.fin[k] ? fin[k].data() : nullptr;
    }
    std::vector<int64_t> it(run.newton_iters ? n : 0), nc(run.nonconv ? n : 0);
    std::vector<int32_t> fl(run.flags ? n : 0);
    r.diag = run.diag && !nccl ? dg.data() : nullptr;
    r.newton_iters = run.newton_iters ? it.data() : nullptr;
    r.nonconv = run.nonconv ? nc.data() : nullptr;
    r.flags = run.flags ? fl.data() : nullptr;
    ebm_options_t op = opt_in ? *opt_in : default_options();
    op.device = devs[(size_t)q];
    op.field_stride = 0;
    EBM_TRY(ebm_run_host(grid, (long long)n, r, &op, nccl ? &hook : nullptr));
    if (!nccl) put_rows(run.diag, dg, ix, rowlen);
    for (int k = 0; k < run.nstate; ++k) put_rows(run.fin[k], fin[k], ix, (size_t)nx);
    put_rows(run.newton_iters, it, ix, 1);
    put_rows(run.nonconv, nc, ix, 1);
    put_rows(run.flags, fl, ix, 1);
    const FieldSel fs(ix, opt_in ? *opt_in : default_options(), run.seasonal || run.raw);
    if (fs.any()) {
      const size_t ns = fs.member.size();
      const size_t lenS = ebm_seasonal_offset(1, grid->dur, 0, 0, run.nvar, nx);
      const size_t lenR = ebm_raw_offset(1, ebm_nraw(grid->nt, grid->dur, op.lastonly), 0, run.nvar, nx);
      MemberRows in2;
      EbmHostRun r2 = members(run, fs.member, nx, &in2);
      std::vector<double> se(run.seasonal ? ns * lenS : 0), rw(run.raw ? ns * lenR : 0);
      r2.seasonal = run.seasonal ? se.data() : nullptr;
      r2.raw = run.raw ? rw.data() : nullptr;
      op.field_stride = 1;
      EBM_TRY(ebm_run_host(grid, (long long)ns, r2, &op, nullptr));
      put_rows(run.seasonal, se, fs.slot, lenS);
      put_rows(run.raw, rw, fs.slot, lenR);
    }
    return EBM_OK;
  });
}

}  // namespace

extern "C" int32_t ebm_classic_run_multi(const ebm_grid_t* grid, int64_t nmem, const ebm_classic_params_t* par,
                                         const ebm_forcing_t* forc, const double* E0, const double* Tg0,
                                         const ebm_options_t* opt_in, const ebm_multi_t* multi, ebm_classic_outputs_t* out) {
  if (!grid || nmem < 1 || !par || !forc || !E0 || !Tg0 || !out) { ebm_set_error("classic_run_multi: NULL argument or nmem < 1"); return EBM_ERR_INVALID; }
  std::vector<int> key((size_t)nmem);
  for (long long m = 0; m < nmem; ++m) key[(size_t)m] = ebm_classic_regime(E0 + m * grid->nx, grid->nx);
  return run_multi(grid, nmem, ebm_classic_host_run(par, forc, E0, Tg0, out), key, opt_in, multi);
}

extern "C" int32_t ebm_miz_run_multi(const ebm_grid_t* grid, int64_t nmem, const ebm_miz_params_t* par,
                                     const ebm_forcing_t* forc, const double* Ei0, const double* Ew0, const double* h0,
                                     const double* D0, const double* phi0, const double* T0guess,
                                     const ebm_options_t* opt_in, const ebm_multi_t* multi, ebm_miz_outputs_t* out) {
  if (!grid || nmem < 1 || !par || !forc || !Ei0 || !Ew0 || !h0 || !D0 || !phi0 || !out) { ebm_set_error("miz_run_multi: NULL argument or nmem < 1"); return EBM_ERR_INVALID; }
  return run_multi(grid, nmem, ebm_miz_host_run(par, forc, Ei0, Ew0, h0, D0, phi0, T0guess, out), std::vector<int>(), opt_in,
                   multi);
}
