// Library-level entry points: ABI introspection, launch accounting, the device-side wait guard / status word, and
// the HOST-buffer variants of the projection (host→device copy, kernels, device→host copy as a three-stream
// pipeline over a ring of staging slots, so that both PCIe directions and the kernels overlap).
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "dm_project.cuh"

namespace dm {
int64_t g_launches = 0;

int sm_count() {
  static int sms[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (sms[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    sms[dev] = n;
  }
  return sms[dev];
}

namespace {
constexpr int kMaxDevices = 64;

// ---- dependency-wait guard: one mapped pinned status word per device (ProjGuard, dm_project.cuh) ----------------
struct StatusWord {
  volatile uint32_t* host = nullptr;
  uint32_t* dev = nullptr;
  bool tried = false;
};
StatusWord g_status[kMaxDevices];
std::mutex g_status_mu;
unsigned long long g_spin_ns = kSpinLimitNs;
uint32_t g_dep_bias = 0;
int g_host_chunk = 0;  // test hook (dm_debug_set_host_chunk): frames per chunk of the host-buffer pipeline, 0 = automatic

// Pipeline of the HOST-buffer entries: three streams (host→device, kernels, device→host) and a ring of
// kSlots staging slots, chained with events.  The copy engine of each PCIe direction always has the next
// chunk queued (a two-stream A/B scheme left the H2D engine idle while the same stream's D2H ran).
// One Scratch per device, each behind its own mutex: two host threads on two devices do not serialise, and
// switching devices does not free anything.
constexpr int kSlots = 4;
struct Scratch {
  std::mutex mu;
  bool ready = false;
  cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[kSlots] = {}, ev_run[kSlots] = {}, ev_out[kSlots] = {};
  void* buf[kSlots] = {};   // staging: inputs + outputs of one chunk
  size_t buf_bytes[kSlots] = {};
  void* ws = nullptr;       // accumulation ring (kept zeroed by the kernel); kernels run on ONE stream
  size_t ws_bytes = 0;
};
Scratch g_scratch[kMaxDevices];

// caller holds sc.mu and has made `device` current
void release_locked(Scratch& sc) {
  for (int i = 0; i < kSlots; ++i) {
    if (sc.buf[i]) cudaFree(sc.buf[i]);
    if (sc.ev_in[i]) cudaEventDestroy(sc.ev_in[i]);
    if (sc.ev_run[i]) cudaEventDestroy(sc.ev_run[i]);
    if (sc.ev_out[i]) cudaEventDestroy(sc.ev_out[i]);
    sc.buf[i] = nullptr;
    sc.buf_bytes[i] = 0;
    sc.ev_in[i] = sc.ev_run[i] = sc.ev_out[i] = nullptr;
  }
  if (sc.ws) cudaFree(sc.ws);
  sc.ws = nullptr;
  sc.ws_bytes = 0;
  if (sc.s_in) cudaStreamDestroy(sc.s_in);
  if (sc.s_run) cudaStreamDestroy(sc.s_run);
  if (sc.s_out) cudaStreamDestroy(sc.s_out);
  sc.s_in = sc.s_run = sc.s_out = nullptr;
  sc.ready = false;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Restores the caller's current device on every exit path of the host entries.
struct DeviceScope {
  int prev = -1;
  bool changed = false;
  cudaError_t enter(int device) {
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    if (prev != device) {
      e = cudaSetDevice(device);
      changed = e == cudaSuccess;
    }
    return e;
  }
  ~DeviceScope() {
    if (changed) cudaSetDevice(prev);
  }
};
}  // namespace

ProjGuard proj_guard(int device) {
  ProjGuard g{g_spin_ns, g_dep_bias, nullptr};
  if (device < 0 || device >= kMaxDevices) return g;
  std::lock_guard<std::mutex> lk(g_status_mu);
  StatusWord& s = g_status[device];
  if (!s.tried) {  // the caller has made `device` current
    s.tried = true;
    void* h = nullptr;
    if (cudaHostAlloc(&h, 64, cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess) {
      *static_cast<volatile uint32_t*>(h) = 0u;
      void* d = nullptr;
      if (cudaHostGetDevicePointer(&d, h, 0) == cudaSuccess) {
        s.host = static_cast<volatile uint32_t*>(h);
        s.dev = static_cast<uint32_t*>(d);
      } else {
        cudaFreeHost(h);
      }
    }
    cudaGetLastError();  // without mapped memory the guard still skips the item and scrubs the workspace
  }
  g.status = s.dev;
  return g;
}

bool take_timeout(int device) {
  if (device < 0 || device >= kMaxDevices) return false;
  std::lock_guard<std::mutex> lk(g_status_mu);
  StatusWord& s = g_status[device];
  if (!s.host || *s.host == 0u) return false;
  *s.host = 0u;
  return true;
}
}  // namespace dm

using namespace dm;

extern "C" int dm_abi_version(void) { return DM_ABI_VERSION; }

extern "C" const char* dm_build_info(void) {
  return "dungeon_maps_b200 sm_100a nvcc " __DATE__ " --fmad=false";
}

extern "C" int64_t dm_launch_count(void) { return g_launches; }

extern "C" int32_t dm_sizeof_struct(int32_t id) {
  switch (id) {
    case 0: return sizeof(DmStep);
    case 1: return sizeof(DmProjSample);
    case 2: return sizeof(DmProjCfg);
    case 3: return sizeof(DmFlowSample);
    case 4: return sizeof(DmFlowCfg);
    case 5: return sizeof(DmFuseSource);
    case 6: return sizeof(DmFuseTarget);
    case 7: return sizeof(DmBuilderCfg);
    case 8: return sizeof(DmMapRef);
    case 9: return sizeof(DmMergeShape);
    case 10: return sizeof(DmPoseCfg);
    case 11: return sizeof(DmValueMapRef);
    default: return -1;
  }
}

extern "C" int dm_device_status(int32_t device) { return take_timeout(device) ? DM_ETIMEOUT : DM_OK; }

extern "C" void dm_debug_set_wait_guard(uint64_t spin_ns, uint32_t dep_bias) {
  g_spin_ns = spin_ns ? spin_ns : kSpinLimitNs;
  g_dep_bias = dep_bias;
}

extern "C" void dm_debug_set_host_chunk(int32_t frames) { g_host_chunk = frames > 0 ? frames : 0; }

// ---- parameter uploads (dm_upload_params) ---------------------------------------------------------------------
// Every call of the device entries needs a small host-built parameter block (per-sample transforms: 192 B a sample)
// on the device.  Copied on the caller's stream it sits between the kernels of the previous call and those of this
// one — a copy-engine round trip with the SMs idle (0.19 -> 0.28 ms per camera_affine_grid call with fresh poses) —
// and through torch it costs ~50 us of host time (pinned staging, torch.empty, two copy_, a content-keyed cache).
// Here: a ring of kUpSlots pinned + device slots per device, the copy on a stream of its own, the caller's stream waits
// for the copy's event.  A slot is recycled kUpSlots uploads later; its previous reader (a kernel the caller queued
// right after that upload returned) is covered by the marker the NEXT upload recorded on the caller's stream, which
// the copy stream waits for before it overwrites the device slot.
namespace {
constexpr int kUpSlots = 64;
constexpr size_t kUpSlotBytes = 64 * 1024;
struct Uploader {
  std::mutex mu;
  bool ready = false, failed = false;
  cudaStream_t copy = nullptr;
  char* host = nullptr;  // kUpSlots x kUpSlotBytes, pinned
  char* dev = nullptr;
  cudaEvent_t done[kUpSlots] = {};    // the copy into slot i has run
  cudaEvent_t marker[kUpSlots] = {};  // recorded on the caller's stream at upload n: all readers of uploads < n precede it
  cudaEvent_t moved = nullptr;        // the caller changed streams: everything queued on the old one
  cudaStream_t last = nullptr;
  unsigned long long n = 0;
};
Uploader g_up[kMaxDevices];
}  // namespace

extern "C" int dm_upload_params(const void* src, size_t nbytes, void* stream_, void** dev_ptr) {
  DM_TRACE();
  if (!src || !dev_ptr || nbytes == 0 || nbytes > kUpSlotBytes) return DM_EINVAL;
  int device = 0;
  DM_CUDA_OK(cudaGetDevice(&device));
  if (device < 0 || device >= kMaxDevices) return DM_EINVAL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  Uploader& u = g_up[device];
  std::lock_guard<std::mutex> lk(u.mu);
  if (!u.ready) {
    if (u.failed) return DM_EINVAL;
    u.failed = true;
    DM_CUDA_OK(cudaStreamCreateWithFlags(&u.copy, cudaStreamNonBlocking));
    DM_CUDA_OK(cudaHostAlloc(reinterpret_cast<void**>(&u.host), kUpSlots * kUpSlotBytes, cudaHostAllocDefault));
    DM_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&u.dev), kUpSlots * kUpSlotBytes));
    for (int i = 0; i < kUpSlots; ++i) {
      DM_CUDA_OK(cudaEventCreateWithFlags(&u.done[i], cudaEventDisableTiming));
      DM_CUDA_OK(cudaEventCreateWithFlags(&u.marker[i], cudaEventDisableTiming));
    }
    DM_CUDA_OK(cudaEventCreateWithFlags(&u.moved, cudaEventDisableTiming));
    u.failed = false;
    u.ready = true;
  }
  const int slot = (int)(u.n % kUpSlots);
  if (u.n > 0 && stream != u.last) {  // readers of earlier uploads sit on another stream: the markers do not cover them
    DM_CUDA_OK(cudaEventRecord(u.moved, u.last));
    DM_CUDA_OK(cudaStreamWaitEvent(u.copy, u.moved, 0));
  }
  u.last = stream;
  // everything the caller queued so far — the readers of all earlier uploads among it — precedes this marker
  DM_CUDA_OK(cudaEventRecord(u.marker[slot], stream));
  if (u.n >= (unsigned long long)kUpSlots) {
    // the slot's previous upload was n - kUpSlots: its copy has read the pinned slot (host wait, long done), and its
    // readers precede the marker of upload n - kUpSlots + 1, which the copy stream waits for
    DM_CUDA_OK(cudaEventSynchronize(u.done[slot]));
    DM_CUDA_OK(cudaStreamWaitEvent(u.copy, u.marker[(slot + 1) % kUpSlots], 0));
  }
  char* h = u.host + (size_t)slot * kUpSlotBytes;
  char* d = u.dev + (size_t)slot * kUpSlotBytes;
  memcpy(h, src, nbytes);
  DM_CUDA_OK(cudaMemcpyAsync(d, h, nbytes, cudaMemcpyHostToDevice, u.copy));
  DM_CUDA_OK(cudaEventRecord(u.done[slot], u.copy));
  DM_CUDA_OK(cudaStreamWaitEvent(stream, u.done[slot], 0));
  ++u.n;
  *dev_ptr = d;
  return DM_OK;
}

static void release_uploaders() {
  for (int dv = 0; dv < kMaxDevices; ++dv) {
    Uploader& u = g_up[dv];
    std::lock_guard<std::mutex> lk(u.mu);
    if (!u.ready) continue;
    if (cudaSetDevice(dv) != cudaSuccess) continue;
    cudaStreamSynchronize(u.copy);
    for (int i = 0; i < kUpSlots; ++i) { cudaEventDestroy(u.done[i]); cudaEventDestroy(u.marker[i]); }
    cudaEventDestroy(u.moved);
    cudaStreamDestroy(u.copy);
    cudaFreeHost(u.host);
    cudaFree(u.dev);
    u.ready = false; u.copy = nullptr; u.host = nullptr; u.dev = nullptr; u.moved = nullptr; u.last = nullptr; u.n = 0;
  }
}

extern "C" void dm_release_scratch(void) {
  int prev = -1;
  cudaGetDevice(&prev);
  for (int d = 0; d < kMaxDevices; ++d) {
    Scratch& sc = g_scratch[d];
    std::lock_guard<std::mutex> lk(sc.mu);
    if (!sc.ready) continue;
    if (cudaSetDevice(d) == cudaSuccess) release_locked(sc);
  }
  release_uploaders();
  if (prev >= 0) cudaSetDevice(prev);
  cudaGetLastError();
}

namespace {
// Shared body of dm_orth_project_host_f32 (values: (b, C, H, W) f32 planes) and dm_orth_project_labels_host_f32
// (labels: (b, 1, H, W) u8 class ids, cfg->C classes).
int orth_project_host(const float* depth, const float* values, const uint8_t* labels, const uint8_t* valid,
                      const DmProjSample* samples, const DmProjCfg* cfg, int32_t b, float* topdown, uint8_t* mask,
                      float* height, int32_t device) {
  if (!cfg || b < 0) return DM_EINVAL;
  if (b == 0) return DM_OK;
  if (!depth || !samples || !topdown || !mask) return DM_EINVAL;
  if (cfg->C > 0 && !values && !labels) return DM_EINVAL;
  if (device < 0 || device >= kMaxDevices) return DM_EINVAL;
  DeviceScope scope;
  DM_CUDA_OK(scope.enter(device));
  Scratch& sc = g_scratch[device];
  std::lock_guard<std::mutex> lk(sc.mu);
  if (!sc.ready) {
    DM_CUDA_OK(cudaStreamCreateWithFlags(&sc.s_in, cudaStreamNonBlocking));
    DM_CUDA_OK(cudaStreamCreateWithFlags(&sc.s_run, cudaStreamNonBlocking));
    DM_CUDA_OK(cudaStreamCreateWithFlags(&sc.s_out, cudaStreamNonBlocking));
    for (int i = 0; i < kSlots; ++i) {
      DM_CUDA_OK(cudaEventCreateWithFlags(&sc.ev_in[i], cudaEventDisableTiming));
      DM_CUDA_OK(cudaEventCreateWithFlags(&sc.ev_run[i], cudaEventDisableTiming));
      DM_CUDA_OK(cudaEventCreateWithFlags(&sc.ev_out[i], cudaEventDisableTiming));
    }
    sc.ready = true;
  }
  const size_t N = (size_t)cfg->H * cfg->W, M = (size_t)cfg->Mh * cfg->Mw;
  const int Cv = cfg->C > 0 ? cfg->C : 1;
  const bool want_h = cfg->C > 0 && cfg->want_height && height;
  const size_t value_bytes = labels ? N : N * 4 * (size_t)cfg->C;  // per frame
  // chunk: ≈ 80 MB of traffic per chunk — large enough for full-rate PCIe copies, small enough that the fill
  // (first chunk in) and drain (last chunk out) of the pipeline stay a few per cent of a 64-frame call
  const size_t frame_bytes = N * 4 + value_bytes + (valid ? N : 0) + M * (5 * (size_t)Cv + (want_h ? 4 : 0));
  int chunk = (int)((80u << 20) / (frame_bytes ? frame_bytes : 1));
  if (g_host_chunk > 0) chunk = g_host_chunk;
  if (chunk < 1) chunk = 1;
  if (chunk > 16) chunk = 16;
  if (chunk > b) chunk = b;
  // staging layout of one chunk (every section 256-byte aligned)
  const size_t o_depth = 0;
  const size_t o_values = align_up(o_depth + chunk * N * 4, 256);
  const size_t o_valid = align_up(o_values + (size_t)chunk * value_bytes, 256);
  const size_t o_samples = align_up(o_valid + (valid ? chunk * N : 0), 256);
  const size_t o_top = align_up(o_samples + chunk * sizeof(DmProjSample), 256);
  const size_t o_mask = align_up(o_top + (size_t)chunk * Cv * M * 4, 256);
  const size_t o_height = align_up(o_mask + (size_t)chunk * Cv * M, 256);
  const size_t total = align_up(o_height + (want_h ? chunk * M * 4 : 0), 256);
  const size_t ws_need = labels ? dm_orth_project_labels_workspace_bytes(cfg, chunk)
                                : dm_orth_project_workspace_bytes(cfg, chunk);
  if (ws_need == 0) return DM_EINVAL;
  for (int i = 0; i < kSlots; ++i) {
    if (sc.buf_bytes[i] < total) {
      if (sc.buf[i]) DM_CUDA_OK(cudaFree(sc.buf[i]));
      sc.buf[i] = nullptr; sc.buf_bytes[i] = 0;
      DM_CUDA_OK(cudaMalloc(&sc.buf[i], total));
      sc.buf_bytes[i] = total;
    }
  }
  if (sc.ws_bytes < ws_need) {
    if (sc.ws) DM_CUDA_OK(cudaFree(sc.ws));
    sc.ws = nullptr; sc.ws_bytes = 0;
    DM_CUDA_OK(cudaMalloc(&sc.ws, ws_need));
    DM_CUDA_OK(cudaMemset(sc.ws, 0, ws_need));
    sc.ws_bytes = ws_need;
  }
  int rc = DM_OK;
  int it = 0;
#define DM_STEP(expr)                                            \
  {                                                              \
    const cudaError_t e_ = (expr);                               \
    if (e_ != cudaSuccess) { rc = static_cast<int>(e_); break; } \
  }
  for (int f0 = 0; f0 < b && rc == DM_OK; f0 += chunk, ++it) {
    const int nf = (b - f0) < chunk ? (b - f0) : chunk;
    const int k = it % kSlots;
    char* base = static_cast<char*>(sc.buf[k]);
    float* d_depth = reinterpret_cast<float*>(base + o_depth);
    void* d_values = cfg->C > 0 ? static_cast<void*>(base + o_values) : nullptr;
    uint8_t* d_valid = valid ? reinterpret_cast<uint8_t*>(base + o_valid) : nullptr;
    DmProjSample* d_samples = reinterpret_cast<DmProjSample*>(base + o_samples);
    float* d_top = reinterpret_cast<float*>(base + o_top);
    uint8_t* d_mask = reinterpret_cast<uint8_t*>(base + o_mask);
    float* d_height = want_h ? reinterpret_cast<float*>(base + o_height) : nullptr;
    // host → device (the slot is free once its previous results have left)
    cudaStream_t si = sc.s_in;
    if (it >= kSlots) DM_STEP(cudaStreamWaitEvent(si, sc.ev_out[k], 0));
    DM_STEP(cudaMemcpyAsync(d_depth, depth + (size_t)f0 * N, (size_t)nf * N * 4, cudaMemcpyHostToDevice, si));
    if (d_values) {
      const char* src = labels ? reinterpret_cast<const char*>(labels) : reinterpret_cast<const char*>(values);
      DM_STEP(cudaMemcpyAsync(d_values, src + (size_t)f0 * value_bytes, (size_t)nf * value_bytes,
                              cudaMemcpyHostToDevice, si));
    }
    if (d_valid) DM_STEP(cudaMemcpyAsync(d_valid, valid + (size_t)f0 * N, (size_t)nf * N, cudaMemcpyHostToDevice, si));
    DM_STEP(cudaMemcpyAsync(d_samples, samples + f0, (size_t)nf * sizeof(DmProjSample), cudaMemcpyHostToDevice, si));
    DM_STEP(cudaEventRecord(sc.ev_in[k], si));
    // kernels
    cudaStream_t sr = sc.s_run;
    DM_STEP(cudaStreamWaitEvent(sr, sc.ev_in[k], 0));
    DmProjCfg c = *cfg;
    if (!want_h) c.want_height = 0;
    if (labels)
      rc = dm_orth_project_labels_f32(d_depth, static_cast<const uint8_t*>(d_values), d_valid, d_samples, &c, nf, d_top,
                                      d_mask, d_height, sc.ws, sc.ws_bytes, sr);
    else
      rc = dm_orth_project_f32(d_depth, static_cast<const float*>(d_values), d_valid, d_samples, &c, nf, d_top, d_mask,
                               d_height, sc.ws, sc.ws_bytes, sr);
    if (rc != DM_OK) break;
    DM_STEP(cudaEventRecord(sc.ev_run[k], sr));
    // device → host
    cudaStream_t so = sc.s_out;
    DM_STEP(cudaStreamWaitEvent(so, sc.ev_run[k], 0));
    DM_STEP(cudaMemcpyAsync(topdown + (size_t)f0 * Cv * M, d_top, (size_t)nf * Cv * M * 4, cudaMemcpyDeviceToHost, so));
    DM_STEP(cudaMemcpyAsync(mask + (size_t)f0 * Cv * M, d_mask, (size_t)nf * Cv * M, cudaMemcpyDeviceToHost, so));
    if (d_height)
      DM_STEP(cudaMemcpyAsync(height + (size_t)f0 * M, d_height, (size_t)nf * M * 4, cudaMemcpyDeviceToHost, so));
    DM_STEP(cudaEventRecord(sc.ev_out[k], so));
  }
#undef DM_STEP
  // every exit path drains the three streams: no copy into the caller's buffers is in flight after the return
  for (cudaStream_t st : {sc.s_in, sc.s_run, sc.s_out}) {
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess && rc == DM_OK) rc = static_cast<int>(e);
  }
  // (always consumed here, after the streams are drained: no stale flag is left for an unrelated later call)
  if (take_timeout(device) && rc == DM_OK) rc = DM_ETIMEOUT;  // the results in the caller's buffers are not valid
  return rc;
}
}  // namespace

extern "C" int dm_orth_project_host_f32(const float* depth, const float* values, const uint8_t* valid,
                                        const DmProjSample* samples, const DmProjCfg* cfg, int32_t b,
                                        float* topdown, uint8_t* mask, float* height, int32_t device) {
  DM_TRACE();
  if (cfg && cfg->C > 0 && !values) return DM_EINVAL;
  return orth_project_host(depth, values, nullptr, valid, samples, cfg, b, topdown, mask, height, device);
}

extern "C" int dm_orth_project_labels_host_f32(const float* depth, const uint8_t* labels, const uint8_t* valid,
                                               const DmProjSample* samples, const DmProjCfg* cfg, int32_t b,
                                               float* topdown, uint8_t* mask, float* height, int32_t device) {
  DM_TRACE();
  if (!cfg || cfg->C <= 0 || !labels) return DM_EINVAL;
  return orth_project_host(depth, nullptr, labels, valid, samples, cfg, b, topdown, mask, height, device);
}
