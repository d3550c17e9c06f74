// C-ABI glue: error reporting, device info, Chamfer forward dispatch.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include "common.cuh"

static thread_local char g_err[512] = "";

void vpn_set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// The only process-wide state: a launch counter (measurement aid, atomic), per-device caches of immutable device
// properties, and the tuning overrides of vpn_set_tuning.  No call depends on another call's state.
static std::atomic<unsigned long long> g_launches{0};
static std::atomic<int> g_tuning[vpn::kTuneCount];

int vpn_check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { vpn_set_error("%s: %s", what, cudaGetErrorString(e)); return VPN_ERR_CUDA; }
  return VPN_OK;
}

namespace vpn {
int chamfer_simple_direction(const float* A, const float* Bp, float* mn, int* idx, u64* key,
                             int B, int nA, int nB, int sm_count, cudaStream_t s);
int chamfer_smallp(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                   int B, int P, int M, cudaStream_t s);
int chamfer_smallp_limit();
int chamfer_tiled_supported(int B, int P, int M, int mode);
size_t chamfer_tiled_workspace_bytes(int B, int P, int M, int mode);
int chamfer_tiled_fwd(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                      int B, int P, int M, void* ws, size_t ws_bytes, int mode, cudaStream_t s, cudaEvent_t* ev);
}

static std::atomic<int> g_sm_count[64];
int vpn::device_sm_count() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev >= 0 && dev < 64 && (n = g_sm_count[dev].load(std::memory_order_relaxed)) > 0) return n;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  if (dev >= 0 && dev < 64) g_sm_count[dev].store(n, std::memory_order_relaxed);
  return n;
}
static int sm_count() { return vpn::device_sm_count(); }
int vpn::tuning_value(int key) { return (key >= 0 && key < vpn::kTuneCount) ? g_tuning[key].load(std::memory_order_relaxed) : 0; }

// Test / probe hook replacing the getenv() look-ups that used to sit on the launch path.
// key: "tiled_r" (4|8|16), "tc_nb" (4|8|16), "emd_cluster" (1|2|4|8), "tc_prune" (2 = tensor-core filter without the
// spatial pruning of chamfer_prep.cu), "serial_recovery" (1 = row and column recovery on one stream); value 0 restores the automatic choice.
extern "C" int vpn_set_tuning(const char* key, int value) {
  static const char* names[vpn::kTuneCount] = {"tiled_r", "tc_nb", "emd_cluster", "tc_prune", "serial_recovery", "ar_variant", "ar_ctas", "ar_threads", "ar_grid_div",
                                                "prep_near_cols", "prep_reps_cols", "prep_near_rows", "prep_reps_rows", "prep_probe", "prep_deterministic", "tc_hunits"};
  for (int k = 0; key && k < vpn::kTuneCount; ++k)
    if (strcmp(key, names[k]) == 0) { g_tuning[k].store(value, std::memory_order_relaxed); return VPN_OK; }
  vpn_set_error("vpn_set_tuning: unknown key"); return VPN_ERR_ARG;
}

extern "C" const char* vpn_last_error_string(void) { return g_err; }

extern "C" int vpn_abi_version(void) { return 2; }

// Number of kernels this library has launched in this process (bench.py reports the per-step delta).
extern "C" unsigned long long vpn_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" int vpn_device_info(int* sms, int* cc_major, int* cc_minor, int* clock_khz) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { vpn_set_error("cudaGetDevice: %s", cudaGetErrorString(e)); return VPN_ERR_CUDA; }
  cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev);
  cudaDeviceGetAttribute(clock_khz, cudaDevAttrClockRate, dev);
  return VPN_OK;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// impl: 0 = auto (tensor-core filter when the shape allows, else the CUDA-core tiled kernel, else generic),
//       1 = generic kernel only,
//       2 / 3 / 4 = CUDA-core tiled kernel with exact / FMA-difference / centred-expansion hot-loop arithmetic,
//       5 = tcgen05 tensor-core filter (chamfer_tc.cu)
//       (2-5 fail on shapes the kernel rejects).  Results are bit-identical for every impl.
static int impl_mode(int impl) { return impl == 0 ? -1 : impl - 2; }
extern "C" int vpn_chamfer_workspace_bytes(int B, int P, int M, int impl, size_t* bytes) {
  if (B < 0 || P <= 0 || M <= 0 || !bytes) { vpn_set_error("chamfer workspace: bad arguments"); return VPN_ERR_ARG; }
  size_t simple = align256((size_t)B * P * 8) + align256((size_t)B * M * 8);
  if (impl < 0 || impl > 5) { vpn_set_error("chamfer workspace: bad impl %d", impl); return VPN_ERR_ARG; }
  size_t tiled = (impl != 1 && vpn::chamfer_tiled_supported(B, P, M, impl_mode(impl))) ? vpn::chamfer_tiled_workspace_bytes(B, P, M, impl_mode(impl)) : 0;
  *bytes = simple > tiled ? simple : tiled;
  return VPN_OK;
}

static int chamfer_fwd_impl(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                            int B, int P, int M, void* workspace, size_t workspace_bytes, int impl, cudaStream_t s,
                            cudaEvent_t* ev) {
  if (B < 0 || P <= 0 || M <= 0) { vpn_set_error("chamfer fwd: bad shape B=%d P=%d M=%d", B, P, M); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (B > 65535) { vpn_set_error("chamfer fwd: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (!p1 || !p2 || !min1 || !idx1 || !min2 || !idx2 || !workspace) { vpn_set_error("chamfer fwd: null pointer"); return VPN_ERR_ARG; }
  if (impl < 0 || impl > 5) { vpn_set_error("chamfer fwd: bad impl %d", impl); return VPN_ERR_ARG; }
  bool tiled_ok = impl != 1 && vpn::chamfer_tiled_supported(B, P, M, impl_mode(impl)) != 0;
  if (impl >= 2 && !tiled_ok) { vpn_set_error("chamfer fwd: tiled kernel does not support this shape"); return VPN_ERR_SHAPE; }
  if (impl != 1 && tiled_ok) {
    int mode = impl_mode(impl);
    return vpn::chamfer_tiled_fwd(p1, p2, min1, idx1, min2, idx2, B, P, M, workspace, workspace_bytes, mode, s, ev);
  }
  size_t need = align256((size_t)B * P * 8) + align256((size_t)B * M * 8);
  if (workspace_bytes < need) { vpn_set_error("chamfer fwd: workspace too small (%zu < %zu)", workspace_bytes, need); return VPN_ERR_WORKSPACE; }
  vpn::u64* key1 = reinterpret_cast<vpn::u64*>(workspace);
  vpn::u64* key2 = reinterpret_cast<vpn::u64*>(reinterpret_cast<char*>(workspace) + align256((size_t)B * P * 8));
  if (impl == 0 && P <= vpn::chamfer_smallp_limit() && !ev) return vpn::chamfer_smallp(p1, p2, min1, idx1, min2, idx2, B, P, M, s);
  if (ev) { cudaEventRecord(ev[0], s); }
  int rc = vpn::chamfer_simple_direction(p1, p2, min1, idx1, key1, B, P, M, sm_count(), s);
  if (rc) return rc;
  if (ev) { cudaEventRecord(ev[1], s); cudaEventRecord(ev[2], s); cudaEventRecord(ev[3], s); }
  rc = vpn::chamfer_simple_direction(p2, p1, min2, idx2, key2, B, M, P, sm_count(), s);
  if (ev) { cudaEventRecord(ev[4], s); }
  return rc;
}

namespace vpn {
int chamfer_tiled_uses_tc(int B, int P, int M, int mode);
int chamfer_tiled_stats(int B, int P, int M, int mode, const void* ws, unsigned long long* out, cudaStream_t s);
}
// Share of the distance matrix the tensor-core filter skipped in the last vpn_chamfer_fwd on this workspace
// (stages = 128 x 256 blocks of pairs, counted per direction).  Zero for the other implementations.  Synchronises.
extern "C" int vpn_chamfer_prune_stats(const void* workspace, int B, int P, int M, int impl, unsigned long long* stages,
                                       unsigned long long* skipped, void* stream) {
  if (!workspace || !stages || !skipped || impl < 0 || impl > 5) { vpn_set_error("chamfer stats: bad arguments"); return VPN_ERR_ARG; }
  unsigned long long out[16] = {0};
  int rc = VPN_OK;
  if (impl != 1 && vpn::chamfer_tiled_supported(B, P, M, impl_mode(impl)))
    rc = vpn::chamfer_tiled_stats(B, P, M, impl_mode(impl), workspace, out, (cudaStream_t)stream);
  *stages = out[0]; *skipped = out[1];
  return rc;
}
// All 16 counters of the tensor-core filter (probe): [0] stages, [1] skipped, [2..5] cycles of epilogue warp 0 summed over
// the CTAs (prologue, phase 0, phase 1, tail), [6] / [7] live stages of phase 0 / 1, [8] live chunks, [9] operand passes.
extern "C" int vpn_chamfer_tc_counters(const void* workspace, int B, int P, int M, int impl, unsigned long long* out16, void* stream) {
  if (!workspace || !out16 || impl < 0 || impl > 5) { vpn_set_error("chamfer counters: bad arguments"); return VPN_ERR_ARG; }
  for (int i = 0; i < 16; ++i) out16[i] = 0;
  if (impl != 1 && vpn::chamfer_tiled_supported(B, P, M, impl_mode(impl)))
    return vpn::chamfer_tiled_stats(B, P, M, impl_mode(impl), workspace, out16, (cudaStream_t)stream);
  return VPN_OK;
}
extern "C" const char* vpn_chamfer_main_kernel(int B, int P, int M, int impl) {
  if (impl < 0 || impl > 5 || B <= 0 || P <= 0 || M <= 0) return "invalid";
  if (impl != 1 && vpn::chamfer_tiled_supported(B, P, M, impl_mode(impl)))
    return vpn::chamfer_tiled_uses_tc(B, P, M, impl_mode(impl)) ? "chamfer_tc_kernel" : "chamfer_tiled_kernel";
  if (impl == 0 && P <= vpn::chamfer_smallp_limit()) return "chamfer_smallp_fwd_kernel";
  return "chamfer_simple_kernel";
}

extern "C" int vpn_chamfer_fwd(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                               int B, int P, int M, void* workspace, size_t workspace_bytes, int impl, void* stream) {
  return chamfer_fwd_impl(p1, p2, min1, idx1, min2, idx2, B, P, M, workspace, workspace_bytes, impl, (cudaStream_t)stream, nullptr);
}

// Measurement variant: runs the forward `reps` times with CUDA events between its stages on `stream`
// and returns the mean device time of each stage in stage_ms[4] (HOST pointer):
//   tiled  : [0] main kernel, [1] MODE_DIFF fall-back launch, [2] row recovery, [3] column recovery
//   generic: [0] direction 1, [1] 0, [2] 0, [3] direction 2.        Synchronises the stream.
extern "C" int vpn_chamfer_fwd_timed(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                                     int B, int P, int M, void* workspace, size_t workspace_bytes, int impl, int reps,
                                     float* stage_ms, void* stream) {
  if (reps < 1 || !stage_ms) { vpn_set_error("chamfer timed: bad arguments"); return VPN_ERR_ARG; }
  cudaStream_t s = (cudaStream_t)stream;
  cudaEvent_t ev[5];
  for (int i = 0; i < 5; ++i) if (cudaEventCreate(&ev[i]) != cudaSuccess) { vpn_set_error("chamfer timed: event create failed"); return VPN_ERR_CUDA; }
  double acc[4] = {0, 0, 0, 0};
  int rc = VPN_OK;
  for (int r = 0; r < reps && rc == VPN_OK; ++r) {
    rc = chamfer_fwd_impl(p1, p2, min1, idx1, min2, idx2, B, P, M, workspace, workspace_bytes, impl, s, ev);
    if (rc) break;
    if (cudaEventSynchronize(ev[4]) != cudaSuccess) { vpn_set_error("chamfer timed: %s", cudaGetErrorString(cudaGetLastError())); rc = VPN_ERR_CUDA; break; }
    for (int i = 0; i < 4; ++i) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); acc[i] += ms; }
  }
  for (int i = 0; i < 5; ++i) cudaEventDestroy(ev[i]);
  if (rc == VPN_OK) for (int i = 0; i < 4; ++i) stage_ms[i] = (float)(acc[i] / reps);
  return rc;
}
