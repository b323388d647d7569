// ufair_host.cu -- host-buffer pipeline: the call a user with numpy / pinned host arrays makes.
//
// The member axis is cut into chunks; each chunk's rows are copied H2D with one strided
// cudaMemcpy2DAsync per array, integrated by the fused kernel, and copied back D2H, on three
// streams with two device staging buffers so copy-in(c+1), kernel(c) and copy-out(c-1) overlap.
// Scenario-shared inputs go up once.  Statistics accumulate across chunks in the private
// histogram copies and are finalised once at the end; statistics labels (stat_group) are staged per
// chunk next to scen_idx, or not at all when they are scen_idx itself, and member weights
// (ufair_run_host_weighted_*) next to them.
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <new>

#include "../../include/ufair.h"
#include "ufair_internal.h"

namespace ufair {

// switch to `device` for the lifetime of the guard, then back to whatever the caller had current
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != device) err = cudaSetDevice(device);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

// The arrays of one call: the descriptor's, and the statistics weights of ufair_run_host_weighted_*, which are not a
// descriptor field.  The staging table addresses each array by the offset of its pointer in this struct.
struct RunArrays {
  ufair_desc d;
  const uint32_t* weight;  // [n_member], or NULL: unweighted statistics
};

// One array the pipeline stages per chunk: `rows` rows of the chunk's members, `elem` bytes each, in a device buffer
// that takes the place of field `field` in the chunk's arrays.
struct Staged {
  size_t field;      // offsetof(RunArrays, <the array's pointer>)
  size_t rows;       // rows per member
  size_t elem;       // bytes per element
  bool in;           // copied up before the kernel; else written by the kernel
  bool on;           // staged in this call
  bool back;         // copied back to the caller's array after the kernel
  bool flat;         // an [n_member] array without row pitch: one 1-D copy
  size_t alias = 0;  // not staged but the staged array of this field instead (labels that are scen_idx itself)
};
constexpr int kStaged = 15;  // entries of run_chunks' table

struct Stage {
  DevBuf b[kStaged];
  cudaEvent_t in_done = nullptr, run_done = nullptr, out_done = nullptr;
  bool used = false;
};

}  // namespace ufair

struct ufair_workspace {
  int device = 0;
  int64_t chunk = 0;
  cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr;
  ufair::Stage st[2];
  ufair::DevBuf e_scen, fext_scen, hist_private, mom_private, hist_out, mom_out;
};

namespace ufair {

#define CK(call, what)                                    \
  do {                                                    \
    cudaError_t e__ = (call);                             \
    if (e__ != cudaSuccess) return cuda_error(e__, what); \
  } while (0)

// the pointer field at byte offset `field` of a call's arrays (every array field is a plain pointer)
static const void* get_field(const RunArrays& a, size_t field) {
  const void* p;
  memcpy(&p, (const char*)&a + field, sizeof p);
  return p;
}
static void set_field(RunArrays& a, size_t field, const void* p) { memcpy((char*)&a + field, &p, sizeof p); }

// members [c0, c0 + cm) of staged array t, between the caller's array (row pitch ld_member) and its device buffer
// (row pitch chunk)
static int copy_chunk(const Staged& t, const RunArrays& h, void* dev, int64_t c0, int64_t cm, int64_t chunk,
                      cudaMemcpyKind kind, cudaStream_t s) {
  char* host = (char*)get_field(h, t.field) + (size_t)c0 * t.elem;
  const bool up = kind == cudaMemcpyHostToDevice;
  void* dst = up ? dev : (void*)host;
  const void* src = up ? (const void*)host : dev;
  const size_t w = (size_t)cm * t.elem, hp = (size_t)h.d.ld_member * t.elem, dp = (size_t)chunk * t.elem;
  if (t.flat) {
    CK(cudaMemcpyAsync(dst, src, w, kind, s), "cudaMemcpyAsync");
    return UFAIR_OK;
  }
  if (t.rows == 0 || w == 0) return UFAIR_OK;
  CK(cudaMemcpy2DAsync(dst, up ? dp : hp, src, up ? hp : dp, w, t.rows, kind, s), "cudaMemcpy2DAsync");
  return UFAIR_OK;
}

// ha: the caller's host arrays; da: the same with the scenario-shared inputs and statistics buffers on the device
template <typename Real>
static int run_chunks(ufair_workspace* ws, const RunArrays& ha, const RunArrays& da) {
  const ufair_desc* h = &ha.d;
  const size_t es = sizeof(Real), i4 = sizeof(int32_t), os = out_elem(h, es);  // os: C / RF / T (out_type)
  const int G = h->n_gas, n_t = h->n_t, out = h->out_mask;
  const int64_t M = h->n_member;
  const size_t gt = (size_t)G * n_t, srows = UFAIR_STATE_ROWS(G);
  const size_t n_out = (size_t)out_rows(h), go = (size_t)G * n_out;  // output rows: per step or per period
  const bool e_member = h->e_mode == UFAIR_E_MEMBER;
  const bool labels_are_scen = h->stat_group != nullptr && h->stat_group == h->scen_idx;
  auto want = [&](int bit) { return (out & bit) != 0; };
  // Every array staged per chunk, in the order its copies are issued: field, rows per member, element bytes, in, on,
  // back, flat[, alias].  Arrays that are not staged keep their field of `da`: NULL, or the scenario-shared copy
  // run_host put on the device.
#define F(x) offsetof(RunArrays, d.x)
  const Staged table[] = {
      {F(emissions), gt, es, true, e_member, false, false},
      {F(f_ext), (size_t)n_t, es, true, h->fext_mode == UFAIR_FEXT_MEMBER, false, false},
      {F(gas_params), (size_t)G * UFAIR_GP_COUNT, es, true, true, false, false},
      {F(thermal_params), UFAIR_TP_COUNT, es, true, true, false, false},
      {F(state_in), srows, es, true, h->state_in != nullptr, false, false},
      {F(e_scale), (size_t)G, es, true, !e_member && h->e_scale != nullptr, false, false},
      {F(scen_idx), 1, i4, true, h->scen_idx != nullptr, false, true},
      {F(stat_group), 1, i4, true, h->stat_group != nullptr && !labels_are_scen, false, true,
       labels_are_scen ? F(scen_idx) : 0},
      {offsetof(RunArrays, weight), 1, sizeof(uint32_t), true, ha.weight != nullptr, false, true},
      {F(out_C), go, os, false, want(UFAIR_OUT_C), want(UFAIR_OUT_C), false},
      {F(out_RF), go, os, false, want(UFAIR_OUT_RF), want(UFAIR_OUT_RF), false},
      {F(out_T), n_out, os, false, want(UFAIR_OUT_T) || h->stats != 0, want(UFAIR_OUT_T), false},  // stats read T
      {F(out_alpha), gt, es, false, want(UFAIR_OUT_ALPHA), want(UFAIR_OUT_ALPHA), false},
      {F(out_E), gt, es, false, want(UFAIR_OUT_E), want(UFAIR_OUT_E), false},
      {F(state_out), srows, es, false, h->state_out != nullptr, h->state_out != nullptr, false},
  };
#undef F
  static_assert(sizeof(table) / sizeof(table[0]) == kStaged, "one staging buffer per table entry");
  // the workspace's chunk size, cut down for long runs so that the two staging sets stay within
  // kStagingBudget bytes (rows per member grow with the step count; the [n_member] label arrays are not counted)
  size_t member_bytes = 0;
  for (const Staged& t : table)
    if (t.on && !t.flat) member_bytes += t.rows * t.elem;
  constexpr size_t kStagingBudget = (size_t)8 << 30;  // bytes, both staging sets together
  int64_t fit = (int64_t)(kStagingBudget / 2 / member_bytes);
  fit = fit / 256 * 256;
  const int64_t chunk = std::min<int64_t>(ws->chunk, std::max<int64_t>(fit, 256));

  // Chunk schedule: the pipeline's fill time is the first chunk's copy-in (plus, when everything comes back, its
  // kernel), during which nothing else runs -- so the first chunks are short and double up to the workspace's
  // size (chunk/8, chunk/4, chunk/2, chunk, chunk, ...; never below 4096 members, whole 256-member groups).
  // A kernel-bound call (few bytes per member: scenario inputs, statistics out) wants large chunks, which fill
  // the GPU for several waves; with the ramp it no longer pays a large chunk's copy-in up front.
  int64_t next = std::min<int64_t>(chunk, std::max<int64_t>(4096, (chunk / 8 + 255) / 256 * 256));
  int64_t c0 = 0;
  for (int64_t c = 0; c0 < M; ++c) {
    Stage& S = ws->st[c & 1];
    const int64_t cm = std::min(next, M - c0);
    if (S.used) {  // staging of chunk c-2: inputs consumed by its kernel, outputs copied out
      CK(cudaStreamWaitEvent(ws->s_in, S.run_done, 0), "cudaStreamWaitEvent");
      CK(cudaStreamWaitEvent(ws->s_run, S.out_done, 0), "cudaStreamWaitEvent");
    }
    for (int i = 0; i < kStaged; ++i) {
      const size_t bytes = table[i].rows * (size_t)chunk * table[i].elem;
      if (table[i].on && S.b[i].cap < bytes) {
        CK(cudaDeviceSynchronize(), "cudaDeviceSynchronize");  // growing: first call with this shape only
        CK(S.b[i].reserve(bytes), "cudaMalloc(staging)");
      }
    }
    // ---- H2D
    for (int i = 0; i < kStaged; ++i) {
      if (!table[i].on || !table[i].in) continue;
      const int rc = copy_chunk(table[i], ha, S.b[i].p, c0, cm, chunk, cudaMemcpyHostToDevice, ws->s_in);
      if (rc != UFAIR_OK) return rc;
    }
    CK(cudaEventRecord(S.in_done, ws->s_in), "cudaEventRecord");
    // ---- kernel
    CK(cudaStreamWaitEvent(ws->s_run, S.in_done, 0), "cudaStreamWaitEvent");
    RunArrays k = da;
    k.d.n_member = cm;
    k.d.ld_member = chunk;
    for (int i = 0; i < kStaged; ++i) {
      if (table[i].on)
        set_field(k, table[i].field, S.b[i].p);
      else if (table[i].alias)
        set_field(k, table[i].field, get_field(k, table[i].alias));
    }
    int rc = run_device<Real>(&k.d, ws->s_run);
    if (rc == UFAIR_OK && h->stats) rc = run_stats_pass<Real>(&k.d, k.weight, ws->s_run);
    if (rc != UFAIR_OK) return rc;
    CK(cudaEventRecord(S.run_done, ws->s_run), "cudaEventRecord");
    // ---- D2H
    CK(cudaStreamWaitEvent(ws->s_out, S.run_done, 0), "cudaStreamWaitEvent");
    for (int i = 0; i < kStaged; ++i) {
      if (!table[i].back) continue;
      rc = copy_chunk(table[i], ha, S.b[i].p, c0, cm, chunk, cudaMemcpyDeviceToHost, ws->s_out);
      if (rc != UFAIR_OK) return rc;
    }
    CK(cudaEventRecord(S.out_done, ws->s_out), "cudaEventRecord");
    S.used = true;
    c0 += cm;
    next = std::min<int64_t>(chunk, next * 2);
  }
  return UFAIR_OK;
}

// like CK, but first waits for the copies already queued from the caller's host buffers, so that no
// transfer is still reading them when the error is reported
#define CKS(call, what)                      \
  do {                                       \
    cudaError_t e__ = (call);                \
    if (e__ != cudaSuccess) {                \
      cudaStreamSynchronize(ws->s_in);       \
      return cuda_error(e__, what);          \
    }                                        \
  } while (0)

// weighted: ufair_run_host_weighted_*, whose statistics take the member weights `weight`
template <typename Real>
static int run_host(ufair_workspace* ws, const ufair_desc* h, bool weighted, const uint32_t* weight, uint64_t* hist,
                    double* moments) {
  if (!ws) return set_error(UFAIR_ERR_ARG, "workspace is NULL");
  if (weighted && !weight) return set_error(UFAIR_ERR_ARG, "ufair_run_host_weighted: weight is NULL");
  // the device path's run rules; its placement rules apply to the staged chunks (run_device, run_stats_pass)
  const int rc0 = check_run(h, sizeof(Real));
  if (rc0 != UFAIR_OK) return rc0;
  if (h->stats && (!hist || !moments)) return set_error(UFAIR_ERR_ARG, "stats requested but hist/moments NULL");
  if (weighted && !h->stats) return set_error(UFAIR_ERR_ARG, "ufair_run_host_weighted: weights need stats == 1");
  if (h->n_member == 0 || h->n_t == 0) return UFAIR_OK;
  DeviceGuard guard(ws->device);  // the caller's current device is restored on every return path
  if (guard.err != cudaSuccess) return cuda_error(guard.err, "cudaSetDevice");

  const size_t es = sizeof(Real);
  const int G = h->n_gas, n_t = h->n_t;
  const size_t stat_rows = (size_t)stat_groups(h) * out_rows(h);  // statistics rows: [groups][n_out]
  ufair_desc d = *h;
  if (h->e_mode != UFAIR_E_MEMBER) {  // scenario-shared inputs go up once
    const size_t nb = (size_t)G * n_t * h->n_scen * es;
    CK(ws->e_scen.reserve(nb), "cudaMalloc(e_scen)");
    CK(cudaMemcpyAsync(ws->e_scen.p, h->emissions, nb, cudaMemcpyHostToDevice, ws->s_in), "H2D scenario emissions");
    d.emissions = ws->e_scen.p;
  }
  if (h->fext_mode == UFAIR_FEXT_SCENARIO) {
    const size_t nb = (size_t)n_t * h->n_scen * es;
    CKS(ws->fext_scen.reserve(nb), "cudaMalloc(fext_scen)");
    CKS(cudaMemcpyAsync(ws->fext_scen.p, h->f_ext, nb, cudaMemcpyHostToDevice, ws->s_in), "H2D scenario forcing");
    d.f_ext = ws->fext_scen.p;
  }
  if (h->stats) {
    d.hist_copies = h->hist_copies > 0 ? h->hist_copies : 16;
    d.hist_t0 = 0;
    d.hist_rows = out_rows(h);
    const size_t rows = (size_t)d.hist_copies * stat_rows;
    CKS(ws->hist_private.reserve(rows * h->hist_bins * sizeof(uint32_t)), "cudaMalloc(hist_private)");
    CKS(ws->mom_private.reserve(rows * UFAIR_MOM_COUNT * sizeof(double)), "cudaMalloc(mom_private)");
    CKS(ws->hist_out.reserve(stat_rows * h->hist_bins * sizeof(uint64_t)), "cudaMalloc(hist)");
    CKS(ws->mom_out.reserve(stat_rows * UFAIR_MOM_COUNT * sizeof(double)), "cudaMalloc(moments)");
    d.hist_private = (uint32_t*)ws->hist_private.p;
    d.moments_private = (double*)ws->mom_private.p;
    int rc = ufair_stats_reset(&d, ws->s_run);
    if (rc != UFAIR_OK) {
      cudaStreamSynchronize(ws->s_in);
      return rc;
    }
  }
  cudaEvent_t shared_up;
  CKS(cudaEventCreateWithFlags(&shared_up, cudaEventDisableTiming), "cudaEventCreate");
  cudaEventRecord(shared_up, ws->s_in);
  cudaStreamWaitEvent(ws->s_run, shared_up, 0);

  int rc = run_chunks<Real>(ws, RunArrays{*h, weight}, RunArrays{d, nullptr});

  if (rc == UFAIR_OK && h->stats) {
    rc = ufair_stats_finalize(&d, (uint64_t*)ws->hist_out.p, (double*)ws->mom_out.p, ws->s_run);
    if (rc == UFAIR_OK) {
      cudaMemcpyAsync(hist, ws->hist_out.p, stat_rows * h->hist_bins * sizeof(uint64_t), cudaMemcpyDeviceToHost, ws->s_run);
      cudaMemcpyAsync(moments, ws->mom_out.p, stat_rows * UFAIR_MOM_COUNT * sizeof(double), cudaMemcpyDeviceToHost, ws->s_run);
    }
  }
  const cudaError_t e1 = cudaStreamSynchronize(ws->s_in), e2 = cudaStreamSynchronize(ws->s_run),
                    e3 = cudaStreamSynchronize(ws->s_out);
  cudaEventDestroy(shared_up);
  ws->st[0].used = ws->st[1].used = false;
  if (rc != UFAIR_OK) return rc;
  if (e1 != cudaSuccess) return cuda_error(e1, "copy-in stream");
  if (e2 != cudaSuccess) return cuda_error(e2, "compute stream");
  if (e3 != cudaSuccess) return cuda_error(e3, "copy-out stream");
  return UFAIR_OK;
}

}  // namespace ufair

using namespace ufair;

extern "C" {

int ufair_workspace_create(int device, int64_t chunk_members, ufair_workspace** out) {
  if (!out) return set_error(UFAIR_ERR_ARG, "ws out-pointer is NULL");
  if (chunk_members <= 0) chunk_members = 65536;
  chunk_members = (chunk_members + 127) / 128 * 128;  // whole CTAs; keeps every row 16-byte aligned
  ufair_workspace* ws = new (std::nothrow) ufair_workspace();
  if (!ws) return set_error(UFAIR_ERR_NOMEM, "out of host memory");
  ws->device = device;
  ws->chunk = chunk_members;
  DeviceGuard guard(device);
  cudaError_t e = guard.err;
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ws->s_in, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ws->s_run, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ws->s_out, cudaStreamNonBlocking);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&ws->st[i].in_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ws->st[i].run_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ws->st[i].out_done, cudaEventDisableTiming);
  }
  if (e != cudaSuccess) {
    ufair_workspace_destroy(ws);
    return cuda_error(e, "ufair_workspace_create");
  }
  *out = ws;
  return UFAIR_OK;
}

int ufair_workspace_destroy(ufair_workspace* ws) {
  if (!ws) return UFAIR_OK;
  DeviceGuard guard(ws->device);
  for (int i = 0; i < 2; ++i) {
    for (int j = 0; j < kStaged; ++j) ws->st[i].b[j].release();
    if (ws->st[i].in_done) cudaEventDestroy(ws->st[i].in_done);
    if (ws->st[i].run_done) cudaEventDestroy(ws->st[i].run_done);
    if (ws->st[i].out_done) cudaEventDestroy(ws->st[i].out_done);
  }
  ws->e_scen.release();
  ws->fext_scen.release();
  ws->hist_private.release();
  ws->mom_private.release();
  ws->hist_out.release();
  ws->mom_out.release();
  if (ws->s_in) cudaStreamDestroy(ws->s_in);
  if (ws->s_run) cudaStreamDestroy(ws->s_run);
  if (ws->s_out) cudaStreamDestroy(ws->s_out);
  delete ws;
  return UFAIR_OK;
}

int ufair_run_host_f64(ufair_workspace* ws, const ufair_desc* d, uint64_t* hist, double* moments) {
  return run_host<double>(ws, d, false, nullptr, hist, moments);
}
int ufair_run_host_f32(ufair_workspace* ws, const ufair_desc* d, uint64_t* hist, double* moments) {
  return run_host<float>(ws, d, false, nullptr, hist, moments);
}
int ufair_run_host_weighted_f64(ufair_workspace* ws, const ufair_desc* d, const uint32_t* weight, uint64_t* hist,
                                double* moments) {
  return run_host<double>(ws, d, true, weight, hist, moments);
}
int ufair_run_host_weighted_f32(ufair_workspace* ws, const ufair_desc* d, const uint32_t* weight, uint64_t* hist,
                                double* moments) {
  return run_host<float>(ws, d, true, weight, hist, moments);
}

}  // extern "C"

// ---- host-link probe: what the platform gives one process for page-locked host <-> device copies.
// bench.py runs it on every rank at once (barrier first) so that e2e can be stated as a fraction of
// the link ceiling measured in the same run, under the same number of concurrent ranks.
namespace ufair {
struct LinkProbe {
  void* host = nullptr;
  void* dev = nullptr;
  size_t cap = 0;
  int device = -1;
  cudaStream_t s_up = nullptr, s_down = nullptr;
  void release() {
    if (host) cudaFreeHost(host);
    if (dev) cudaFree(dev);
    if (s_up) cudaStreamDestroy(s_up);
    if (s_down) cudaStreamDestroy(s_down);
    host = dev = nullptr;
    s_up = s_down = nullptr;
    cap = 0;
    device = -1;
  }
};
static LinkProbe g_probe;

static double wall_seconds() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}
}  // namespace ufair

extern "C" int ufair_link_probe(int device, int64_t bytes_up, int64_t bytes_down, int32_t rows, int32_t reps, double* gbs,
                                double* seconds) {
  using namespace ufair;
  if (bytes_up <= 0 && bytes_down <= 0) {  // release the probe's buffers
    if (g_probe.device >= 0) {
      DeviceGuard guard(g_probe.device);
      g_probe.release();
    }
    return UFAIR_OK;
  }
  if (!gbs || reps < 1 || rows < 0 || bytes_up < 0 || bytes_down < 0)
    return set_error(UFAIR_ERR_ARG, "ufair_link_probe: bad arguments");
  if (rows > 1 && ((bytes_up % rows) != 0 || (bytes_down % rows) != 0))
    return set_error(UFAIR_ERR_ARG, "ufair_link_probe: byte counts must be multiples of rows");
  DeviceGuard guard(device);
  if (guard.err != cudaSuccess) return cuda_error(guard.err, "cudaSetDevice");
  // each direction owns its own part of both buffers; pitched copies use a host pitch of twice the row
  const size_t need = 2 * ((size_t)bytes_up + (size_t)bytes_down);
  if (g_probe.device != device || g_probe.cap < need) {
    g_probe.release();
    cudaError_t e = cudaHostAlloc(&g_probe.host, need, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaMalloc(&g_probe.dev, need);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&g_probe.s_up, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&g_probe.s_down, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      g_probe.release();
      return cuda_error(e, "ufair_link_probe: allocation");
    }
    memset(g_probe.host, 0, need);  // touch: the pages exist before anything is timed
    g_probe.cap = need;
    g_probe.device = device;
  }
  char* h_up = (char*)g_probe.host;
  char* h_down = h_up + 2 * (size_t)bytes_up;
  char* d_up = (char*)g_probe.dev;
  char* d_down = d_up + 2 * (size_t)bytes_up;
  auto copy = [&](bool up, cudaStream_t s) -> cudaError_t {
    if (rows > 1) {
      const size_t w = (size_t)(up ? bytes_up : bytes_down) / rows;
      return up ? cudaMemcpy2DAsync(d_up, w, h_up, 2 * w, w, rows, cudaMemcpyHostToDevice, s)
                : cudaMemcpy2DAsync(h_down, 2 * w, d_down, w, w, rows, cudaMemcpyDeviceToHost, s);
    }
    return up ? cudaMemcpyAsync(d_up, h_up, (size_t)bytes_up, cudaMemcpyHostToDevice, s)
              : cudaMemcpyAsync(h_down, d_down, (size_t)bytes_down, cudaMemcpyDeviceToHost, s);
  };
  const bool up = bytes_up > 0, down = bytes_down > 0;
  cudaError_t e = cudaSuccess;
  if (up) e = copy(true, g_probe.s_up);  // warm-up
  if (e == cudaSuccess && down) e = copy(false, g_probe.s_down);
  if (e == cudaSuccess) e = cudaStreamSynchronize(g_probe.s_up);
  if (e == cudaSuccess) e = cudaStreamSynchronize(g_probe.s_down);
  double t_up = 0.0, t_down = 0.0;
  const double t0 = wall_seconds();
  for (int r = 0; r < reps && e == cudaSuccess; ++r) {
    if (up) e = copy(true, g_probe.s_up);
    if (e == cudaSuccess && down) e = copy(false, g_probe.s_down);
  }
  // the shorter direction is waited for first, so that each direction's own completion time is seen
  const bool up_first = !down || (up && bytes_up <= bytes_down);
  for (int k = 0; k < 2 && e == cudaSuccess; ++k) {
    const bool do_up = (k == 0) == up_first;
    if (do_up && up) {
      e = cudaStreamSynchronize(g_probe.s_up);
      t_up = wall_seconds() - t0;
    } else if (!do_up && down) {
      e = cudaStreamSynchronize(g_probe.s_down);
      t_down = wall_seconds() - t0;
    }
  }
  if (e != cudaSuccess) return cuda_error(e, "ufair_link_probe: copy");
  gbs[0] = up ? (double)bytes_up * reps / 1e9 / t_up : 0.0;
  gbs[1] = down ? (double)bytes_down * reps / 1e9 / t_down : 0.0;
  if (seconds) *seconds = t_up > t_down ? t_up : t_down;
  return UFAIR_OK;
}
