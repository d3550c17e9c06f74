// Earth mover's distance approximation by the auction algorithm (SURVEY.md section 8f "next" #1).
//
// Replaces modules/loss/emd (emd_module.py:29-79 -> emd.cpp:6-23 -> emd_cuda.cu:227-316): the reference runs
// 7 launches per iteration (351 for the training setting eps = 0.005, iters = 50, train.py:188-195) and lets racing
// writes decide ties.  Here ONE launch runs the whole auction: a thread-block cluster of up to 8 CTAs per sample
// (sized so that the batch fills the 148 SMs), each CTA owning a slice of the bidders and keeping the objects'
// coordinates plus a per-iteration copy of the prices in its shared memory; the per-object state is shared through
// an L2-resident workspace with atomics, phases are separated by cluster barriers, and ties are resolved
// deterministically (lowest index wins), so the result is reproducible run to run.
//   per iteration   compact the unassigned bidders
//                   Bid    : one warp per bidder, lanes stride over the objects: value = 3 - |x2 - x1| - price,
//                            best (first maximum) / second best, warp merge; increment = best - better + eps;
//                            atomicMax of the object's largest increment          (emd_cuda.cu:95-179)
//                   GetMax : the lowest bidder within 1e-6 of the object's maximum wins   (:181-194)
//                   Assign : winner takes the object, evicts the previous owner, price += increment (:196-216);
//                            in the last iteration every unassigned bidder takes its object unconditionally
//   finally         dist = |x1 - x2[assignment]|^2                                  (:218-226)
// Arithmetic: fp32, every operation rounded separately (the reference mixes a double literal and nvcc's FMA
// contraction; its results are an approximation and not reproducible bit for bit in any case).
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace vpn {

constexpr int kEmdThreads = 1024;
constexpr int kEmdMaxCluster = 8;
constexpr int kEmdObjSmemMaxN = 12288;         // 16 n bytes of object coordinates + prices fit in shared memory
constexpr int kEmdWsWords = 8;                 // workspace words per point: price, assign, assign_inv, max_inc, winner, x, y, z

// Per-sample state shared by the CTAs of a cluster lives in the caller's workspace (HBM, L2 resident: 32 n bytes).
struct EmdGlobal {
  float* price; int* assign; int* assign_inv; int* max_inc; int* winner; float *x, *y, *z; int* total;
};
__device__ __forceinline__ EmdGlobal emd_global(unsigned char* ws, int b, int n) {
  EmdGlobal g;
  int* base = reinterpret_cast<int*>(ws) + (size_t)b * ((size_t)kEmdWsWords * n + 4);
  g.total = base;                                             // [0], [1]: unassigned bidders of the sample, by iteration parity
  float* f = reinterpret_cast<float*>(base + 4);
  g.price = f; g.x = f + (size_t)n; g.y = f + 2 * (size_t)n; g.z = f + 3 * (size_t)n;
  int* i = reinterpret_cast<int*>(f + 4 * (size_t)n);
  g.assign = i; g.assign_inv = i + (size_t)n; g.max_inc = i + 2 * (size_t)n; g.winner = i + 3 * (size_t)n;
  return g;
}

struct Top2 { float best, better; int i; };
// multiset top-2 merge; equal best values: the lower index keeps the object, the other becomes the runner-up
__device__ __forceinline__ Top2 top2_merge(const Top2& a, const Top2& b) {
  Top2 r;
  const bool a_wins = (a.best > b.best) || (a.best == b.best && a.i < b.i);
  if (a_wins) { r.best = a.best; r.i = a.i; r.better = fmaxf(a.better, b.best); }
  else        { r.best = b.best; r.i = b.i; r.better = fmaxf(b.better, a.best); }
  return r;
}

// grid: x = sample * C + cluster rank; launched with cluster dimension C.  CTA r of the cluster owns the bidders
// [r * per, (r + 1) * per), per = ceil(n / C): it lists its unassigned ones, bids, and applies their assignments;
// the per-object state (price, largest increment, winner, owner) is shared through the workspace with atomics, and
// the phases are separated by cluster barriers.  OBJ_SMEM: object coordinates and a per-iteration copy of the prices
// in shared memory (n <= 12288), else read through L1/L2.
// dynamic shared memory: [OBJ_SMEM: x, y, z, price (4 n floats)] un, bid (per ints), inc (per floats)
template <bool OBJ_SMEM>
__global__ void __launch_bounds__(kEmdThreads, 1)
emd_auction_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2, float* __restrict__ dist,
                   int* __restrict__ assignment, unsigned char* __restrict__ ws, int n, int C, float eps, int iters) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  __shared__ int s_cnt;
  cg::cluster_group cluster = cg::this_cluster();
  const int b = blockIdx.x / C, rank = blockIdx.x % C;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (n + C - 1) / C;
  const int j_lo = min(n, rank * per), j_hi = min(n, j_lo + per);
  const EmdGlobal g = emd_global(ws, b, n);
  float* sf = reinterpret_cast<float*>(s_dyn);
  const float* ox = OBJ_SMEM ? sf : g.x;
  const float* oy = OBJ_SMEM ? sf + n : g.y;
  const float* oz = OBJ_SMEM ? sf + 2 * (size_t)n : g.z;
  float* sprice = sf + 3 * (size_t)n;                                  // OBJ_SMEM only
  int* s_un = reinterpret_cast<int*>(sf + (OBJ_SMEM ? 4 * (size_t)n : 0));
  int* s_bid = s_un + per;
  float* s_inc = reinterpret_cast<float*>(s_bid + per);
  const float* X1 = xyz1 + (size_t)b * n * 3;
  const float* X2 = xyz2 + (size_t)b * n * 3;
  const int neg_big = __float_as_int(-1e9f);
  for (int k = j_lo + tid; k < j_hi; k += kEmdThreads) {                 // this CTA's slice of the shared state
    g.price[k] = 0.f; g.assign[k] = -1; g.assign_inv[k] = -1; g.max_inc[k] = neg_big; g.winner[k] = 0x7fffffff;
    if (!OBJ_SMEM) { g.x[k] = X2[3 * k]; g.y[k] = X2[3 * k + 1]; g.z[k] = X2[3 * k + 2]; }
  }
  if (OBJ_SMEM)
    for (int k = tid; k < n; k += kEmdThreads) { sf[k] = X2[3 * k]; sf[n + k] = X2[3 * k + 1]; sf[2 * (size_t)n + k] = X2[3 * k + 2]; }
  if (rank == 0 && tid == 0) { g.total[0] = 0; g.total[1] = 0; }
  if (tid == 0) s_cnt = 0;
  cluster.sync();
  for (int it = 0; it < iters; ++it) {
    const bool last = (it == iters - 1);
    const int par = it & 1;
    // ---- this CTA's unassigned bidders (any order: the phases below do not depend on it); price copy
    for (int j0 = j_lo; j0 < j_hi; j0 += kEmdThreads) {
      const int j = j0 + tid;
      const bool un = j < j_hi && __ldcg(&g.assign[j]) == -1;          // written by other CTAs: read through L2
      const unsigned bal = __ballot_sync(0xffffffffu, un);
      int base = 0;
      if (lane == 0 && bal) base = atomicAdd(&s_cnt, __popc(bal));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (un) s_un[base + __popc(bal & ((1u << lane) - 1u))] = j;
    }
    if (OBJ_SMEM) for (int k = tid; k < n; k += kEmdThreads) sprice[k] = __ldcg(&g.price[k]);
    __syncthreads();
    const int cnt = s_cnt;
    if (tid == 0 && cnt) atomicAdd(&g.total[par], cnt);
    cluster.sync();
    if (__ldcg(&g.total[par]) == 0) break;                         // everything assigned: further iterations change nothing
    if (rank == 0 && tid == 0) g.total[par ^ 1] = 0;
    const float* pr = OBJ_SMEM ? sprice : g.price;
    // ---- Bid
    for (int u = warp; u < cnt; u += kEmdThreads / 32) {
      const int j = s_un[u];
      const float x1 = X1[3 * j], y1 = X1[3 * j + 1], z1 = X1[3 * j + 2];
      Top2 t; t.best = -1e9f; t.better = -1e9f; t.i = 0x7fffffff;
      for (int k = lane; k < n; k += 32) {
        const float dx = __fsub_rn(ox[k], x1), dy = __fsub_rn(oy[k], y1), dz = __fsub_rn(oz[k], z1);
        const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
        const float v = __fsub_rn(__fsub_rn(3.0f, __fsqrt_rn(d2)), OBJ_SMEM ? pr[k] : __ldcg(&pr[k]));
        if (v > t.best) { t.better = t.best; t.best = v; t.i = k; }
        else if (v > t.better) t.better = v;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        Top2 other;
        other.best = __shfl_xor_sync(0xffffffffu, t.best, o);
        other.better = __shfl_xor_sync(0xffffffffu, t.better, o);
        other.i = __shfl_xor_sync(0xffffffffu, t.i, o);
        t = top2_merge(t, other);
      }
      if (lane == 0) {
        const float inc = __fadd_rn(__fsub_rn(t.best, t.better), eps);
        s_bid[u] = t.i; s_inc[u] = inc;
        atomicMax(&g.max_inc[t.i], __float_as_int(inc));    // increments are >= eps >= 0: integer order = float order
      }
    }
    cluster.sync();
    // ---- GetMax: lowest bidder within 1e-6 of the object's largest increment
    for (int u = tid; u < cnt; u += kEmdThreads) {
      const int t = s_bid[u];
      const double inc = (double)s_inc[u], mx = (double)__int_as_float(__ldcg(&g.max_inc[t]));
      if (inc - 1e-6 <= mx && mx <= inc + 1e-6) atomicMin(&g.winner[t], s_un[u]);
    }
    cluster.sync();
    // ---- Assign
    for (int u = tid; u < cnt; u += kEmdThreads) {
      const int j = s_un[u], t = s_bid[u];
      if (last || __ldcg(&g.winner[t]) == j) {
        const int old = __ldcg(&g.assign_inv[t]);
        if (!last && old != -1) g.assign[old] = -1;
        g.assign_inv[t] = j;
        g.assign[j] = t;
        g.price[t] = __fadd_rn(__ldcg(&g.price[t]), s_inc[u]);
        g.max_inc[t] = neg_big;
      }
    }
    cluster.sync();
    // reset the winners of the objects that were bid on (after every Assign thread of the cluster has read them)
    for (int u = tid; u < cnt; u += kEmdThreads) g.winner[s_bid[u]] = 0x7fffffff;
    if (tid == 0) s_cnt = 0;
    __syncthreads();
  }
  cluster.sync();
  for (int j = j_lo + tid; j < j_hi; j += kEmdThreads) {
    const int k = __ldcg(&g.assign[j]);
    float d2 = 0.f;
    if (k >= 0) {
      const float dx = __fsub_rn(X1[3 * j], X2[3 * k]), dy = __fsub_rn(X1[3 * j + 1], X2[3 * k + 1]), dz = __fsub_rn(X1[3 * j + 2], X2[3 * k + 2]);
      d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    }
    dist[(size_t)b * n + j] = d2;
    assignment[(size_t)b * n + j] = k;
  }
}

// NmDistanceGradKernel (emd_cuda.cu:283-300): grad_xyz1 = 2 g (x1 - x2[assignment])
__global__ void emd_bwd_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2,
                               const int* __restrict__ assignment, const float* __restrict__ gdist,
                               float* __restrict__ gxyz1, size_t total, int n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t b = i / n;
  const int k = assignment[i];
  const float g = gdist[i] * 2.0f;
  const float* a = xyz1 + 3 * i;
  const float* t = xyz2 + 3 * (b * n + (k < 0 ? 0 : k));
  gxyz1[3 * i] = g * (a[0] - t[0]); gxyz1[3 * i + 1] = g * (a[1] - t[1]); gxyz1[3 * i + 2] = g * (a[2] - t[2]);
}

// Loss head of train.py:188-195 / train_gcn.py:91-95, torch.sqrt(dist).mean() per sample: loss[b] = weight * (sum_j sqrt(dist[b,j]) / n).
// Stage 1: kEmdLossSlices blocks per sample; block s sums the elements s * 256 + t + k * 256 * kEmdLossSlices in thread t,
// then warps and blocks in a fixed tree.  Stage 2 adds the slices in index order.  The summation order depends on n only
// (not on B, the auction's cluster size or the stream), so a sample's loss is the same bits in any batch.
constexpr int kEmdLossSlices = 32;
constexpr int kEmdLossThreads = 256;

__global__ void __launch_bounds__(kEmdLossThreads)
emd_loss_partial_kernel(const float* __restrict__ dist, float* __restrict__ partial, int n) {
  __shared__ float red[kEmdLossThreads / 32];
  const int b = blockIdx.x / kEmdLossSlices, sl = blockIdx.x % kEmdLossSlices;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* d = dist + (size_t)b * n;
  float s = 0.f;
  for (int j = sl * kEmdLossThreads + threadIdx.x; j < n; j += kEmdLossThreads * kEmdLossSlices) s = __fadd_rn(s, __fsqrt_rn(d[j]));
  s = warp_sum(s);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
    for (int w = 0; w < kEmdLossThreads / 32; ++w) a += red[w];
    partial[blockIdx.x] = a;
  }
}

__global__ void emd_loss_final_kernel(const float* __restrict__ partial, float weight, float* __restrict__ loss, int B, int n) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float a = 0.f;
  for (int k = 0; k < kEmdLossSlices; ++k) a += partial[(size_t)b * kEmdLossSlices + k];
  loss[b] = weight * (a / (float)n);
}

// Backward of the head and of the auction's dist in one pass, in autograd's operation order through
// torch.sqrt(dist).mean(dim=1) * weight followed by NmDistanceGradKernel (emd_cuda.cu:283-300):
//   g = (grad_loss[b] * weight) / n;  g = g / (2 sqrt(d));  grad_xyz1 = (2 g) (x1 - x2[assignment]).
// d == 0 gives inf * 0 = NaN, as in the reference.
__global__ void emd_loss_bwd_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2,
                                    const int* __restrict__ assignment, const float* __restrict__ dist,
                                    const float* __restrict__ grad_loss, float weight, float* __restrict__ gxyz1,
                                    size_t total, int n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t b = i / n;
  const int k = assignment[i];
  float g = __fdiv_rn(__fmul_rn(grad_loss[b], weight), (float)n);
  g = __fdiv_rn(g, __fmul_rn(2.0f, __fsqrt_rn(dist[i])));
  g = __fmul_rn(g, 2.0f);
  const float* a = xyz1 + 3 * i;
  const float* t = xyz2 + 3 * (b * n + (k < 0 ? 0 : k));
  gxyz1[3 * i] = __fmul_rn(g, __fsub_rn(a[0], t[0]));
  gxyz1[3 * i + 1] = __fmul_rn(g, __fsub_rn(a[1], t[1]));
  gxyz1[3 * i + 2] = __fmul_rn(g, __fsub_rn(a[2], t[2]));
}

}  // namespace vpn

using namespace vpn;

static size_t emd_ws_bytes(int B, int n) { return (size_t)B * ((size_t)kEmdWsWords * n + 4) * 4; }

// CTAs per sample: enough to fill the GPU (148 SMs, one 1024-thread CTA each), at most 8 (portable cluster size)
static int emd_cluster_size(int B, int n) {
  int c = 1;
  while (c < kEmdMaxCluster && (long long)B * c * 2 <= 160 && n / (c * 2) >= 256) c *= 2;
  { int v = tuning_value(kTuneEmdCluster); if (v == 1 || v == 2 || v == 4 || v == 8) c = v; }     // vpn_set_tuning("emd_cluster")
  return c;
}

extern "C" int vpn_emd_workspace_bytes(int B, int n, size_t* bytes) {
  if (B < 0 || n <= 0 || !bytes) { vpn_set_error("emd workspace: bad arguments"); return VPN_ERR_ARG; }
  *bytes = emd_ws_bytes(B, n);
  return VPN_OK;
}

template <bool OBJ_SMEM>
static int emd_launch(const float* xyz1, const float* xyz2, float* dist, int* assignment, unsigned char* ws,
                      int B, int n, int C, float eps, int iters, cudaStream_t s) {
  const int per = (n + C - 1) / C;
  const size_t smem = (OBJ_SMEM ? (size_t)16 * n : 0) + (size_t)12 * per;
  static DeviceOnce once;
  if (smem > 48 * 1024 && set_dyn_smem(emd_auction_kernel<OBJ_SMEM>, 224 * 1024, once) != cudaSuccess) {
    vpn_set_error("emd fwd: smem attribute"); return VPN_ERR_CUDA;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(B * C)); cfg.blockDim = dim3(kEmdThreads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, emd_auction_kernel<OBJ_SMEM>, xyz1, xyz2, dist, assignment, ws, n, C, eps, iters);
  if (e != cudaSuccess) { vpn_set_error("emd fwd: launch: %s", cudaGetErrorString(e)); return VPN_ERR_CUDA; }
  return vpn_check_launch("emd_auction_kernel");
}

extern "C" int vpn_emd_fwd(const float* xyz1, const float* xyz2, float* dist, int* assignment, void* workspace,
                           size_t workspace_bytes, int B, int n, float eps, int iters, void* stream) {
  if (B < 0 || n <= 0) { vpn_set_error("emd fwd: bad shape B=%d n=%d", B, n); return VPN_ERR_SHAPE; }
  if (iters < 1 || !(eps >= 0.f)) { vpn_set_error("emd fwd: need iters >= 1 and eps >= 0"); return VPN_ERR_ARG; }
  if (B == 0) return VPN_OK;
  if (!xyz1 || !xyz2 || !dist || !assignment || !workspace) { vpn_set_error("emd fwd: null pointer"); return VPN_ERR_ARG; }
  if (workspace_bytes < emd_ws_bytes(B, n)) { vpn_set_error("emd fwd: workspace too small (%zu < %zu)", workspace_bytes, emd_ws_bytes(B, n)); return VPN_ERR_WORKSPACE; }
  const int C = emd_cluster_size(B, n);
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t smem_obj = (size_t)16 * n + (size_t)12 * ((n + C - 1) / C);
  if (n <= kEmdObjSmemMaxN && smem_obj <= 220 * 1024) return emd_launch<true>(xyz1, xyz2, dist, assignment, ws, B, n, C, eps, iters, s);
  return emd_launch<false>(xyz1, xyz2, dist, assignment, ws, B, n, C, eps, iters, s);
}

extern "C" int vpn_emd_bwd(const float* xyz1, const float* xyz2, const int* assignment, const float* grad_dist,
                           float* grad_xyz1, int B, int n, void* stream) {
  if (B < 0 || n <= 0) { vpn_set_error("emd bwd: bad shape"); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (!xyz1 || !xyz2 || !assignment || !grad_dist || !grad_xyz1) { vpn_set_error("emd bwd: null pointer"); return VPN_ERR_ARG; }
  const size_t total = (size_t)B * n;
  emd_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(xyz1, xyz2, assignment, grad_dist, grad_xyz1, total, n);
  return vpn_check_launch("emd_bwd_kernel");
}

// scratch: >= 32 * B floats of device memory (partial sums)
extern "C" int vpn_emd_loss_fwd(const float* dist, float weight, float* loss, float* scratch, int B, int n, void* stream) {
  if (B < 0 || n <= 0) { vpn_set_error("emd loss: bad shape B=%d n=%d", B, n); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (!dist || !loss || !scratch) { vpn_set_error("emd loss: null pointer"); return VPN_ERR_ARG; }
  cudaStream_t s = (cudaStream_t)stream;
  emd_loss_partial_kernel<<<(unsigned)B * kEmdLossSlices, kEmdLossThreads, 0, s>>>(dist, scratch, n);
  int rc = vpn_check_launch("emd_loss_partial_kernel");
  if (rc) return rc;
  emd_loss_final_kernel<<<(B + 127) / 128, 128, 0, s>>>(scratch, weight, loss, B, n);
  return vpn_check_launch("emd_loss_final_kernel");
}

extern "C" int vpn_emd_loss_bwd(const float* xyz1, const float* xyz2, const int* assignment, const float* dist,
                                const float* grad_loss, float weight, float* grad_xyz1, int B, int n, void* stream) {
  if (B < 0 || n <= 0) { vpn_set_error("emd loss bwd: bad shape B=%d n=%d", B, n); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (!xyz1 || !xyz2 || !assignment || !dist || !grad_loss || !grad_xyz1) { vpn_set_error("emd loss bwd: null pointer"); return VPN_ERR_ARG; }
  const size_t total = (size_t)B * n;
  emd_loss_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(xyz1, xyz2, assignment, dist, grad_loss,
                                                                                       weight, grad_xyz1, total, n);
  return vpn_check_launch("emd_loss_bwd_kernel");
}
