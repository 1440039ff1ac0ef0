// C ABI (include/tssplat_b200.h) over the plan builder and the sm_100a kernels.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/tssplat_b200.h"
#include "tsb_kernels.cuh"
#include "tsb_plan.h"

struct tsb_handle_s {
  int device = 0;
  tsb::KParams kp{};
  tsb::LaunchConfig lc{};
  // tsb_energy_grad_host: calls alternate between two internal streams, each running upload -> kernel ->
  // download on its own staging buffers; only the kernels are ordered across the two (ev_run), so call
  // i+1's upload overlaps call i's kernel and download.  (Measured on the pool's B200 hosts: 31.6 us per call
  // for 0.64 MB each way; a third stream for the downloads, or one stream per stage, costs 2.5x the CPU time
  // per call in the driver and ends up slower: 46-49 us.)
  float *stage_x[2] = {nullptr, nullptr}, *stage_grad[2] = {nullptr, nullptr}, *stage_energy[2] = {nullptr, nullptr};
  cudaStream_t s_pipe[2] = {nullptr, nullptr};
  cudaEvent_t ev_run[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
  unsigned host_calls = 0;
  bool amips = false;
  tsb_info_t info{};
  std::vector<void *> allocs;
  std::string err;
};

namespace {

thread_local std::string g_create_err;

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int d) : dev(d) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  int dev;
  ~DeviceGuard() { if (prev >= 0 && prev != dev) cudaSetDevice(prev); }
};

// device that owns a device pointer (falls back to the current device)
int device_of(const void *p) {
  cudaPointerAttributes a{};
  if (p && cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeDevice) return a.device;
  cudaGetLastError();
  int d = 0;
  cudaGetDevice(&d);
  return d;
}

int fail(tsb_handle_t h, int code, const std::string &msg) {
  if (h) h->err = msg; else g_create_err = msg;
  return code;
}

template <class T>
int upload(tsb_handle_t h, const T *src, size_t count, const T **out, size_t min_elems = 1) {
  const size_t bytes = std::max(count, min_elems) * sizeof(T);
  void *d = nullptr;
  cudaError_t e = cudaMalloc(&d, bytes);
  if (e != cudaSuccess) return fail(h, TSB_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  h->allocs.push_back(d);
  h->info.device_bytes += int64_t(bytes);
  if (count) {
    e = cudaMemcpy(d, src, count * sizeof(T), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("cudaMemcpy: ") + cudaGetErrorString(e));
  }
  *out = static_cast<const T *>(d);
  return TSB_OK;
}

template <class T>
int alloc_zero(tsb_handle_t h, size_t elems, T **out) {
  const size_t bytes = std::max<size_t>(elems, 1) * sizeof(T);
  void *d = nullptr;
  cudaError_t e = cudaMalloc(&d, bytes);
  if (e != cudaSuccess) return fail(h, TSB_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  h->allocs.push_back(d);
  h->info.device_bytes += int64_t(bytes);
  e = cudaMemset(d, 0, bytes);
  if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("cudaMemset: ") + cudaGetErrorString(e));
  *out = static_cast<T *>(d);
  return TSB_OK;
}

int env_int(const char *name, int dflt) {
  const char *e = std::getenv(name);
  return e && *e ? std::atoi(e) : dflt;
}

struct Choice { int nw, ring, smem, ctas, global; };

}  // namespace

extern "C" {

int tsb_create(const float *rest_xyz, const int32_t *tets, int32_t n, int32_t nele, const tsb_options_t *opt,
               int device, tsb_handle_t *out) {
  if (!out) return fail(nullptr, TSB_E_INVALID, "out is null");
  *out = nullptr;
  tsb::PlanConfig pc;
  int nw = env_int("TSSPLAT_B200_WARPS", 16), ring = env_int("TSSPLAT_B200_RING_SLOTS", 2);
  const int cpc = std::max(1, std::min(8, env_int("TSSPLAT_B200_CELLS_PER_CHUNK", 6)));
  int tet_cost_x100 = env_int("TSSPLAT_B200_TET_COST_X100", 0);
  if (opt) {
    if (opt->warps_per_cta != 0) nw = opt->warps_per_cta;
    if (opt->ring_slots != 0) ring = opt->ring_slots;
    if (opt->tet_cost_x100 > 0) tet_cost_x100 = opt->tet_cost_x100;
    pc.laplacian_scale = opt->laplacian_scale ? 1 : 0;
    pc.force_global = opt->force_global ? 1 : 0;
    pc.enable_amips = opt->enable_amips ? 1 : 0;
  }
  if (env_int("TSSPLAT_B200_FORCE_GLOBAL", 0)) pc.force_global = 1;
  pc.max_lanes_per_row = std::max(1, std::min(4, env_int("TSSPLAT_B200_LANES_PER_ROW", pc.max_lanes_per_row)));
  if (env_int("TSSPLAT_B200_TETCELL_COST_X100", 0) > 0) pc.tetcell_cost = float(env_int("TSSPLAT_B200_TETCELL_COST_X100", 0)) / 100.f;
  if (nw != 8 && nw != 16) return fail(nullptr, TSB_E_INVALID, "warps_per_cta must be 8 or 16");
  if (ring < 2 || ring > 8) return fail(nullptr, TSB_E_INVALID, "ring_slots must be in [2, 8]");
  if (tet_cost_x100 > 0) pc.tet_cost = float(tet_cost_x100) / 100.f;
  pc.nw = nw;

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
    cudaGetLastError();
    return fail(nullptr, TSB_E_CUDA, "no CUDA device " + std::to_string(device) + " (tssplat_b200 has no CPU path)");
  }
  DeviceGuard guard(device);
  if (!guard.ok) return fail(nullptr, TSB_E_CUDA, "cannot select CUDA device " + std::to_string(device));
  int sms = 0, smem_optin = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0 ||
      cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess)
    return fail(nullptr, TSB_E_CUDA, "cannot query the CUDA device");
  pc.area_cap = std::min(tsb::kMaxStagedVerts, std::max(0, (smem_optin - tsb::energy_smem_bytes(nw, 2, cpc, 0, false) - 256) / 32));

  // Called by the plan builder once the component sizes are known: pick the ring size that lets the
  // staging area fit, query occupancy, return the persistent grid.
  Choice ch{nw, ring, 0, 0, 0};
  std::string cb_err;
  pc.grid_cb = [&](int /*vh*/, int area_verts, bool &global_mode) -> int {
    if (!global_mode) {
      int r = ring;
      while (r > 2 && tsb::energy_smem_bytes(nw, r, cpc, area_verts, false) > smem_optin) --r;
      if (tsb::energy_smem_bytes(nw, r, cpc, area_verts, false) > smem_optin) global_mode = true;
      else ch.ring = r;
    }
    ch.global = global_mode ? 1 : 0;
    if (global_mode) while (ch.ring > 2 && tsb::energy_smem_bytes(nw, ch.ring, cpc, 0, true) > smem_optin) --ch.ring;
    ch.smem = tsb::energy_smem_bytes(nw, ch.ring, cpc, global_mode ? 0 : area_verts, global_mode);
    int ctas = 0;
    cudaError_t e = tsb::energy_occupancy(nw, ch.smem, global_mode, pc.enable_amips != 0, &ctas);
    if (e != cudaSuccess || ctas < 1) {
      cb_err = std::string("kernel does not fit the device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "occupancy 0");
      return 0;
    }
    const int want = env_int("TSSPLAT_B200_CTAS_PER_SM", nw == 16 ? 1 : 2);
    ch.ctas = std::max(1, std::min(ctas, want));
    return ch.ctas * sms;
  };

  pc.ring_cells = env_int("TSSPLAT_B200_NO_SPLIT", 0) ? 0 : ring * cpc;
  pc.rb_cap_div = std::max(1, env_int("TSSPLAT_B200_RB_CAP_DIV", pc.rb_cap_div));
  if (env_int("TSSPLAT_B200_SEG_OVERHEAD_X100", -1) >= 0) pc.seg_overhead = float(env_int("TSSPLAT_B200_SEG_OVERHEAD_X100", 25)) / 100.f;
  tsb::HostPlan plan;
  std::string err;
  int rc = tsb::build_plan(rest_xyz, tets, n, nele, pc, plan, err);
  if (rc != TSB_OK) return fail(nullptr, cb_err.empty() ? rc : TSB_E_CUDA, cb_err.empty() ? err : cb_err);

  tsb_handle_t h = new tsb_handle_s();
  h->device = device;
  tsb::KParams &kp = h->kp;
#define TSB_TRY(expr) do { rc = (expr); if (rc != TSB_OK) { g_create_err = h->err; tsb_destroy(h); return rc; } } while (0)
  TSB_TRY(upload(h, plan.stream.data(), plan.stream.size(), &kp.stream, 16));
  {
    const float *x4 = nullptr;
    TSB_TRY(upload(h, plan.X4.data(), plan.X4.size(), &x4, 4));
    kp.X4 = reinterpret_cast<const float4 *>(x4);
    const tsb::SegHdr *sg = nullptr;
    TSB_TRY(upload(h, plan.segs.data(), plan.segs.size(), &sg, 1));
    kp.segs = sg;
    const int32_t *cs = nullptr;
    TSB_TRY(upload(h, plan.cta_seg.data(), plan.cta_seg.size(), &cs, 2));
    kp.cta_seg = reinterpret_cast<const int2 *>(cs);
    const uint32_t *wd = nullptr;
    TSB_TRY(upload(h, plan.wdesc.data(), plan.wdesc.size(), &wd, 2));
    kp.wdesc = reinterpret_cast<const uint2 *>(wd);
    const uint16_t *wsg = nullptr;
    TSB_TRY(upload(h, plan.wseg.data(), plan.wseg.size(), &wsg, 2));
    kp.wseg = reinterpret_cast<const ushort2 *>(wsg);
  }
  TSB_TRY(upload(h, plan.vlist.data(), plan.vlist.size(), &kp.vlist, 1));
  TSB_TRY(upload(h, plan.pos16.data(), plan.pos16.size(), &kp.pos16, 2));
  TSB_TRY(upload(h, plan.pos_gid.data(), plan.pos_gid.size(), &kp.pos_gid, 1));
  TSB_TRY(upload(h, plan.orphans.data(), plan.orphans.size(), &kp.orphans, 1));
  if (pc.enable_amips) {
    const float *bt = nullptr;
    TSB_TRY(upload(h, plan.Bt.data(), plan.Bt.size(), &bt, 4));
    kp.Bt = reinterpret_cast<const float4 *>(bt);
    TSB_TRY(upload(h, plan.wtc0.data(), plan.wtc0.size(), &kp.wtc0, 1));
  }
  TSB_TRY(alloc_zero(h, size_t(plan.n_components), &kp.done));
  {
    std::vector<unsigned long long> init(size_t(plan.grid) * 4, tsb::kEnergySentinel);
    const unsigned long long *ce = nullptr;
    TSB_TRY(upload(h, init.data(), init.size(), &ce, 2));
    kp.cta_energy = reinterpret_cast<double *>(const_cast<unsigned long long *>(ce));
  }
#ifdef TSB_TRACE
  TSB_TRY(alloc_zero(h, size_t(plan.grid) * 16, &kp.trace));
#endif
  if (plan.mode_global) {
    TSB_TRY(alloc_zero(h, size_t(plan.n), &kp.u4g));
    TSB_TRY(alloc_zero(h, size_t(plan.n), &kp.x4g));
  }
#undef TSB_TRY
  kp.n_orphans = int32_t(plan.orphans.size());
  kp.n_components = plan.n_components;
  kp.n = plan.n;
  kp.vh = plan.vh;
  kp.ring_bytes = tsb::energy_ring_bytes(ch.ring, cpc, plan.mode_global != 0);
  kp.cells_per_chunk = cpc;
  kp.ring_slots = ch.ring;
  kp.stage_bytes = plan.mode_global ? 0 : plan.area_verts * 32;
  h->lc = tsb::LaunchConfig{nw, plan.grid, ch.smem, plan.mode_global, 0};
  h->amips = pc.enable_amips != 0;

  tsb_info_t &I = h->info;
  I.n = plan.n; I.nele = plan.nele; I.n_components = plan.n_components; I.grid = plan.grid;
  I.warps_per_cta = nw; I.ctas_per_sm = ch.ctas; I.mode_global = plan.mode_global; I.smem_bytes = ch.smem;
  I.ring_slots = ch.ring; I.n_segments = int32_t(plan.segs.size()); I.n_boundary_faces = plan.n_boundary_faces;
  I.max_component_vertices = plan.max_comp_verts; I.nnz = plan.nnz; I.nnz_padded = plan.nnz_padded;
  // bytes one launch requests: the warp streams, rest positions + x per staged component copy, grad
  int64_t staged = 0;
  for (const tsb::SegHdr &s : plan.segs) staged += s.nv;
  I.stream_bytes = int64_t(plan.stream.size()) + (plan.mode_global ? int64_t(plan.n) * (12 + 16 + 64) : staged * (16 + 12 + 2)) +
                   int64_t(plan.n) * 12 + int64_t(plan.segs.size()) * 32 + int64_t(plan.grid) * (16 + 8 * nw);
  *out = h;
  return TSB_OK;
}

void tsb_destroy(tsb_handle_t h) {
  if (!h) return;
  DeviceGuard guard(h->device);
  for (int k = 0; k < 2; ++k) {
    if (h->ev_run[k]) cudaEventDestroy(h->ev_run[k]);
    if (h->ev_done[k]) cudaEventDestroy(h->ev_done[k]);
    if (h->s_pipe[k]) cudaStreamDestroy(h->s_pipe[k]);
  }
  for (void *p : h->allocs) cudaFree(p);
  delete h;
}

const char *tsb_last_error(tsb_handle_t h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int tsb_get_info(tsb_handle_t h, tsb_info_t *info) {
  if (!h || !info) return TSB_E_INVALID;
  *info = h->info;
  return TSB_OK;
}

static int energy_grad_impl(tsb_handle_t h, const float *x_dev, float c1, float c2, float c3, int32_t order, float gradH,
                            const float *gradH_dev, float *energy_out_dev, int energy4, float *grad_out_dev, void *stream) {
  if (!h) return TSB_E_INVALID;
  if (!x_dev || !energy_out_dev) return fail(h, TSB_E_INVALID, "x_dev and energy_out_dev must be non-null");
  if (order != 2 && order != 4)
    return fail(h, TSB_E_INVALID, "order must be 2 or 4 (the reference yields zeros for anything else: tet_spheres_cuda.cu:57-63)");
  if (c3 != 0.f && !h->amips) return fail(h, TSB_E_INVALID, "c3 != 0 needs a handle created with tsb_options_t.enable_amips = 1");
  DeviceGuard guard(h->device);
  if (!guard.ok) return fail(h, TSB_E_CUDA, "cannot select the handle's CUDA device");
  tsb::KParams kp = h->kp;
  kp.x = x_dev; kp.grad = grad_out_dev; kp.energy_out = energy_out_dev; kp.gradH_dev = gradH_dev;
  kp.c1 = c1; kp.c2 = c2; kp.c3 = c3; kp.gradH = gradH; kp.order = order; kp.energy4 = energy4;
  tsb::LaunchConfig lc = h->lc;
  lc.amips = c3 != 0.f ? 1 : 0;          // c3 == 0: the very instantiation tsb_energy_grad always ran
  cudaError_t e = tsb::launch_energy_grad(kp, lc, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("energy_grad launch: ") + cudaGetErrorString(e));
  return TSB_OK;
}

int tsb_energy_grad(tsb_handle_t h, const float *x_dev, float c1, float c2, int32_t order, float gradH,
                    const float *gradH_dev, float *energy_out_dev, float *grad_out_dev, void *stream) {
  return energy_grad_impl(h, x_dev, c1, c2, 0.f, order, gradH, gradH_dev, energy_out_dev, 0, grad_out_dev, stream);
}

int tsb_energy_grad_ex(tsb_handle_t h, const float *x_dev, const tsb_terms_t *terms, float gradH, const float *gradH_dev,
                       float *energy_out_dev, float *grad_out_dev, void *stream) {
  if (!h) return TSB_E_INVALID;
  if (!terms) return fail(h, TSB_E_INVALID, "terms is null");
  return energy_grad_impl(h, x_dev, terms->c1, terms->c2, terms->c3, terms->order, gradH, gradH_dev, energy_out_dev, 1, grad_out_dev, stream);
}

int tsb_energy_grad_host(tsb_handle_t h, const float *x_host, float c1, float c2, int32_t order, float gradH,
                         float *energy_out_host, float *grad_out_host, void *stream) {
  if (!h) return TSB_E_INVALID;
  if (!x_host || !energy_out_host) return fail(h, TSB_E_INVALID, "x_host and energy_out_host must be non-null");
  if (order != 2 && order != 4) return fail(h, TSB_E_INVALID, "order must be 2 or 4");
  DeviceGuard guard(h->device);
  if (!guard.ok) return fail(h, TSB_E_CUDA, "cannot select the handle's CUDA device");
  const size_t nb = size_t(h->info.n) * 3 * sizeof(float);
  if (!h->stage_x[0]) {
    int rc = TSB_OK;
    for (int k = 0; k < 2 && rc == TSB_OK; ++k) {
      rc = alloc_zero(h, size_t(h->info.n) * 3, &h->stage_x[k]);
      if (rc == TSB_OK) rc = alloc_zero(h, size_t(h->info.n) * 3, &h->stage_grad[k]);
      if (rc == TSB_OK) rc = alloc_zero(h, 4, &h->stage_energy[k]);
    }
    if (rc != TSB_OK) return rc;
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) {
      e = cudaStreamCreateWithFlags(&h->s_pipe[k], cudaStreamNonBlocking);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_run[k], cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_done[k], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("pipeline stream setup: ") + cudaGetErrorString(e));
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; }
  const int k = int(h->host_calls & 1u);
  cudaError_t e;
  if (cap != cudaStreamCaptureStatusNone) {      // inside a stream capture: keep it linear on the caller's stream
    e = cudaMemcpyAsync(h->stage_x[k], x_host, nb, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("H2D copy: ") + cudaGetErrorString(e));
    const int rc = tsb_energy_grad(h, h->stage_x[k], c1, c2, order, gradH, nullptr, h->stage_energy[k],
                                   grad_out_host ? h->stage_grad[k] : nullptr, stream);
    if (rc != TSB_OK) return rc;
    e = cudaMemcpyAsync(energy_out_host, h->stage_energy[k], 3 * sizeof(float), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && grad_out_host) e = cudaMemcpyAsync(grad_out_host, h->stage_grad[k], nb, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("D2H copy: ") + cudaGetErrorString(e));
    return TSB_OK;
  }
  ++h->host_calls;
  // stream k: upload (ordered after call i-2's download of the same buffers by stream order) ...
  cudaStream_t sk = h->s_pipe[k];
  e = cudaMemcpyAsync(h->stage_x[k], x_host, nb, cudaMemcpyHostToDevice, sk);
  // ... kernel, after the previous call's kernel on the other stream (the handle's counters are shared) ...
  if (e == cudaSuccess) e = cudaStreamWaitEvent(sk, h->ev_run[k ^ 1], 0);
  if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("H2D copy: ") + cudaGetErrorString(e));
  // pinned + mapped host memory has a device alias (UVA): the kernel stores the 3 floats there itself, one copy
  // less per call (looked up every call: the address may have been freed and reused as pageable memory)
  float *e_alias = nullptr;
  {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, energy_out_host) == cudaSuccess && a.type == cudaMemoryTypeHost && a.devicePointer)
      e_alias = static_cast<float *>(a.devicePointer);
    else
      cudaGetLastError();
  }
  float *e_dst = e_alias ? e_alias : h->stage_energy[k];
  const int rc = tsb_energy_grad(h, h->stage_x[k], c1, c2, order, gradH, nullptr, e_dst,
                                 grad_out_host ? h->stage_grad[k] : nullptr, sk);
  if (rc != TSB_OK) return rc;
  e = cudaEventRecord(h->ev_run[k], sk);
  // ... download; the caller's stream waits for it, so synchronising `stream` completes the call
  if (e == cudaSuccess && !e_alias)
    e = cudaMemcpyAsync(energy_out_host, h->stage_energy[k], 3 * sizeof(float), cudaMemcpyDeviceToHost, sk);
  if (e == cudaSuccess && grad_out_host) e = cudaMemcpyAsync(grad_out_host, h->stage_grad[k], nb, cudaMemcpyDeviceToHost, sk);
  if (e == cudaSuccess) e = cudaEventRecord(h->ev_done[k], sk);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(st, h->ev_done[k], 0);
  if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("D2H copy: ") + cudaGetErrorString(e));
  return TSB_OK;
}

int tsb_scale(const float *g_dev, int64_t count, float gradH, const float *gradH_dev, float *out_dev, void *stream) {
  if (!g_dev || !out_dev || count < 0) return fail(nullptr, TSB_E_INVALID, "tsb_scale: null pointer or negative count");
  if (count == 0) return TSB_OK;
  DeviceGuard guard(device_of(g_dev));
  cudaError_t e = tsb::launch_scale(g_dev, count, gradH, gradH_dev, out_dev, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(nullptr, TSB_E_CUDA, std::string("scale launch: ") + cudaGetErrorString(e));
  return TSB_OK;
}

int tsb_grad_limit(float *grad_dev, int64_t count, float s_threshold, float s, float *work_dev, void *stream) {
  if (!grad_dev || !work_dev || count < 0) return fail(nullptr, TSB_E_INVALID, "tsb_grad_limit: null pointer or negative count");
  if (count == 0) return TSB_OK;
  DeviceGuard guard(device_of(grad_dev));
  cudaError_t e = tsb::launch_grad_limit(grad_dev, count, s_threshold, s, work_dev, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(nullptr, TSB_E_CUDA, std::string("grad_limit launch: ") + cudaGetErrorString(e));
  return TSB_OK;
}

int tsb_adam_uniform_step(float *p_dev, const float *grad_dev, float *g1_dev, float *g2_dev, int64_t count, double lr,
                          double beta1, double beta2, int32_t step, double grad_limit, float *work_dev, void *stream) {
  if (!p_dev || !grad_dev || !g1_dev || !g2_dev || !work_dev || count < 0 || step < 1)
    return fail(nullptr, TSB_E_INVALID, "tsb_adam_uniform_step: null pointer, negative count or step < 1");
  if (count == 0) return TSB_OK;
  DeviceGuard guard(device_of(p_dev));
  cudaError_t e = tsb::launch_adam_uniform(p_dev, grad_dev, g1_dev, g2_dev, count, lr, beta1, beta2, step, grad_limit,
                                           work_dev, static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(nullptr, TSB_E_CUDA, std::string("adam_uniform launch: ") + cudaGetErrorString(e));
  return TSB_OK;
}

int tsb_train_step(tsb_handle_t h, float *x_dev, const float *grad_ext_dev, float c1, float c2, int32_t order,
                   const tsb_train_state_t *st, void *stream) {
  if (!h) return TSB_E_INVALID;
  if (!x_dev || !st) return fail(h, TSB_E_INVALID, "tsb_train_step: x_dev and st must be non-null");
  if (!st->g1 || !st->g2 || !st->grad || !st->energy || !st->schedule || !st->history || !st->step || !st->work)
    return fail(h, TSB_E_INVALID, "tsb_train_step: a state buffer is null");
  if (st->n_steps < 1) return fail(h, TSB_E_INVALID, "tsb_train_step: n_steps must be >= 1");
  if (!(st->beta1 >= 0.0 && st->beta1 < 1.0 && st->beta2 >= 0.0 && st->beta2 < 1.0))
    return fail(h, TSB_E_INVALID, "tsb_train_step: betas must be in [0, 1)");
  // validates order, selects the device and runs the very launch tsb_energy_grad runs with gradH = 1
  int rc = energy_grad_impl(h, x_dev, c1, c2, 0.f, order, 1.f, nullptr, st->energy, 0, st->grad, stream);
  if (rc != TSB_OK) return rc;
  DeviceGuard guard(h->device);
  cudaError_t e = tsb::launch_train_adam(x_dev, st->grad, grad_ext_dev, st->g1, st->g2, int64_t(h->info.n) * 3, st->beta1,
                                         st->beta2, st->schedule, st->energy, st->history, st->step, st->n_steps, st->work,
                                         static_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(h, TSB_E_CUDA, std::string("train_step launch: ") + cudaGetErrorString(e));
  return TSB_OK;
}

#ifdef TSB_TRACE
/* profiling build only: copy the [grid][16] phase stamps of the last launch to the host */
int tsb_trace_read(tsb_handle_t h, unsigned long long *out, int64_t count) {
  if (!h || !out) return TSB_E_INVALID;
  DeviceGuard guard(h->device);
  const int64_t have = int64_t(h->info.grid) * 16;
  return cudaMemcpy(out, h->kp.trace, size_t(std::min(count, have)) * 8, cudaMemcpyDeviceToHost) == cudaSuccess ? TSB_OK : TSB_E_CUDA;
}
#endif

}  // extern "C"
