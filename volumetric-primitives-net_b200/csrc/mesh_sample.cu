// Area-weighted surface sampling of a batch of triangle meshes with shared topology.
//
// Replaces the per-sample Python loop over kaolin's TriangleMesh.sample at train_sphere.py:71-80 (and
// dataset/dataset.py:162-165): face areas -> discrete distribution -> face choice -> sqrt-u barycentric point
//     p = (1 - sqrt(u1)) v0 + sqrt(u1) (1 - u2) v1 + sqrt(u1) u2 v2.
// kaolin draws the face with torch.distributions.Categorical and the barycentric pair with two Uniform samples;
// here all three draws are explicit inputs u (B, n, 3) and the face is the inverse CDF of u0 (first face whose
// cumulative area share exceeds u0), so that the oracle can replay the same draws.  One launch builds every
// sample's CDF (one CTA per mesh, shared-memory scan), one launch places the points.
#include "common.cuh"

namespace vpn {

constexpr int kMsThreads = 256;

// 2 * area of face f of mesh `verts` (kaolin: sqrt(a + b + c) / 2 with a, b, c the squared cross-product components
// of the edge vectors (v0 - v1) and (v1 - v2))
__device__ __forceinline__ float face_area(const float* __restrict__ verts, const int* __restrict__ faces, int f) {
  const int i0 = faces[3 * f], i1 = faces[3 * f + 1], i2 = faces[3 * f + 2];
  // every operation rounded separately, as the chain of torch ops in kaolin does (no FMA contraction)
  const float x1 = __fsub_rn(verts[3 * i0], verts[3 * i1]), x2 = __fsub_rn(verts[3 * i0 + 1], verts[3 * i1 + 1]), x3 = __fsub_rn(verts[3 * i0 + 2], verts[3 * i1 + 2]);
  const float y1 = __fsub_rn(verts[3 * i1], verts[3 * i2]), y2 = __fsub_rn(verts[3 * i1 + 1], verts[3 * i2 + 1]), y3 = __fsub_rn(verts[3 * i1 + 2], verts[3 * i2 + 2]);
  const float a = __fsub_rn(__fmul_rn(x2, y3), __fmul_rn(x3, y2));
  const float bb = __fsub_rn(__fmul_rn(x3, y1), __fmul_rn(x1, y3));
  const float c = __fsub_rn(__fmul_rn(x1, y2), __fmul_rn(x2, y1));
  return __fdiv_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(bb, bb)), __fmul_rn(c, c))), 2.0f);
}

// grid: x = mesh.  cdf (B, F): inclusive prefix sums of area / (sum + eps), in face order (sequential per chunk,
// fixed combination order: deterministic).
__global__ void __launch_bounds__(kMsThreads)
mesh_cdf_kernel(const float* __restrict__ verts, const int* __restrict__ faces, float* __restrict__ cdf,
                int V, int F, float eps) {
  __shared__ float part[kMsThreads];
  __shared__ float total_s;
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* vb = verts + (size_t)b * V * 3;
  float* cb = cdf + (size_t)b * F;
  const int per = (F + kMsThreads - 1) / kMsThreads;
  const int f0 = tid * per, f1 = min(F, f0 + per);
  float run = 0.f;
  for (int f = f0; f < f1; ++f) { run = __fadd_rn(run, face_area(vb, faces, f)); cb[f] = run; }      // local inclusive sums
  part[tid] = run;
  __syncthreads();
  if (tid == 0) {
    float acc = 0.f;
    for (int i = 0; i < kMsThreads; ++i) { const float p = part[i]; part[i] = acc; acc = __fadd_rn(acc, p); }
    total_s = acc;
  }
  __syncthreads();
  const float base = part[tid], denom = __fadd_rn(total_s, eps);
  for (int f = f0; f < f1; ++f) cb[f] = __fdiv_rn(__fadd_rn(cb[f], base), denom);
}

// grid: x = blocks of points, y = mesh
__global__ void __launch_bounds__(kMsThreads)
mesh_sample_kernel(const float* __restrict__ verts, const int* __restrict__ faces, const float* __restrict__ cdf,
                   const float* __restrict__ u, float* __restrict__ points, int* __restrict__ face_idx,
                   int V, int F, int n) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * kMsThreads + threadIdx.x;
  if (i >= n) return;
  const float* ub = u + ((size_t)b * n + i) * 3;
  const float* cb = cdf + (size_t)b * F;
  const float u0 = ub[0];
  int lo = 0, hi = F - 1;                          // first face with cdf > u0 (last face if rounding leaves none)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cb[mid] > u0) hi = mid; else lo = mid + 1;
  }
  const float* vb = verts + (size_t)b * V * 3;
  const int i0 = faces[3 * lo], i1 = faces[3 * lo + 1], i2 = faces[3 * lo + 2];
  const float su = __fsqrt_rn(ub[1]), vv = ub[2];
  const float w0 = __fsub_rn(1.0f, su), w1 = __fmul_rn(su, __fsub_rn(1.0f, vv)), w2 = __fmul_rn(su, vv);
  float* p = points + ((size_t)b * n + i) * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c)
    p[c] = __fadd_rn(__fadd_rn(__fmul_rn(w0, vb[3 * i0 + c]), __fmul_rn(w1, vb[3 * i1 + c])), __fmul_rn(w2, vb[3 * i2 + c]));
  face_idx[(size_t)b * n + i] = lo;
}

// grad_verts (B, V, 3) must be zeroed by the caller; the face choice is piecewise constant (no gradient), the
// barycentric weights are constants.
__global__ void __launch_bounds__(kMsThreads)
mesh_sample_bwd_kernel(const int* __restrict__ faces, const float* __restrict__ u, const int* __restrict__ face_idx,
                       const float* __restrict__ grad_points, float* __restrict__ grad_verts, int V, int n) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * kMsThreads + threadIdx.x;
  if (i >= n) return;
  const float* ub = u + ((size_t)b * n + i) * 3;
  const int f = face_idx[(size_t)b * n + i];
  const float su = __fsqrt_rn(ub[1]), vv = ub[2];
  const float w[3] = {__fsub_rn(1.0f, su), __fmul_rn(su, __fsub_rn(1.0f, vv)), __fmul_rn(su, vv)};
  const float* g = grad_points + ((size_t)b * n + i) * 3;
  float* gv = grad_verts + (size_t)b * V * 3;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int vi = faces[3 * f + k];
#pragma unroll
    for (int c = 0; c < 3; ++c) atomicAdd(&gv[3 * vi + c], w[k] * g[c]);
  }
}

// ---- backward as a gather with a fixed summation order ------------------------------------------------------------
// The atomic kernel above piles ~n * 9 / (3 V) read-modify-writes onto every float of grad_verts (~127 at B = 1,
// n = 16384 on the 386-vertex sphere) in an order that changes from run to run.  Here, per mesh:
//   mesh_sample_sort_kernel        stable counting sort of the samples by face: per-segment histograms, a scan, then a
//                                  scatter in sample-index order -> order (B, n) = per-face runs, starts (B, F+1)
//   mesh_sample_face_grad_kernel   one warp per face: the 3 corner sums of w_k * g over the face's run (lane-strided,
//                                  then a fixed butterfly) -> face_grad (B, F, 3, 3)
//   mesh_sample_vertex_grad_kernel one thread per vertex: its incident (face, corner) sums in the order of the caller's
//                                  vertex -> (face, corner) CSR, written over grad_verts
// Every order depends only on the mesh's own face_idx and n, so a mesh's gradient is the same bits in every run and in
// every batch.  No global atomics, no memset.
constexpr int kMsSortThreads = 1024;
constexpr int kMsSortWarps = kMsSortThreads / 32;
constexpr int kMsSortSmemInts = 200 * 1024 / 4;
constexpr int kMsFaceWarps = 8;

// Segments of a mesh's samples counted separately (one warp each) and where their (segments + 1) * F histogram lives:
// shared memory while it leaves at least 8 segments, else the workspace (32 segments).
__host__ __device__ inline int ms_sort_segments(int F, bool* in_smem) {
  const int s = kMsSortSmemInts / F - 1;
  *in_smem = s >= 8;
  return *in_smem ? (s < kMsSortWarps ? s : kMsSortWarps) : kMsSortWarps;
}

// grid: x = mesh; dynamic smem: (S + 1) F ints when the histogram is in shared memory.  hist_ws: (B, S + 1, F) ints of
// the workspace otherwise.  Rows 0..S-1 of the histogram count segment s, row S holds the face's run start.
__global__ void __launch_bounds__(kMsSortThreads)
mesh_sample_sort_kernel(const int* __restrict__ face_idx, int* __restrict__ order, int* __restrict__ starts,
                        int* __restrict__ hist_ws, int F, int n, int S, int in_smem) {
  extern __shared__ int ms_hist_smem[];
  __shared__ int warp_tot[kMsSortWarps];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int* hist = in_smem ? ms_hist_smem : hist_ws + (size_t)b * (S + 1) * F;
  int* first = hist + (size_t)S * F;
  const int* fb = face_idx + (size_t)b * n;
  int* ob = order + (size_t)b * n;
  int* sb = starts + (size_t)b * (F + 1);
  for (int i = tid; i < S * F; i += kMsSortThreads) hist[i] = 0;
  __syncthreads();
  const int seg = (n + S - 1) / S;
  const int j0 = warp * seg, j1 = min(n, j0 + seg);
  const unsigned lt = (1u << lane) - 1u;
  // counts per segment: the lanes that share a face are counted by the lowest of them (no atomics)
  if (warp < S) {
    for (int base = j0; base < j1; base += 32) {
      const int j = base + lane;
      int f = j < j1 ? fb[j] : -1;
      if (f >= F) f = -1;                                                  // out-of-range faces contribute nothing
      const unsigned peers = __match_any_sync(0xffffffffu, f);
      if (f >= 0 && (peers & lt) == 0) hist[warp * F + f] += __popc(peers);
      __syncwarp();
    }
  }
  __syncthreads();
  // per face: exclusive prefix over the segments, total in `first`
  for (int f = tid; f < F; f += kMsSortThreads) {
    int run = 0;
    for (int s = 0; s < S; ++s) { const int c = hist[s * F + f]; hist[s * F + f] = run; run += c; }
    first[f] = run;
  }
  __syncthreads();
  // exclusive scan of the face totals: a contiguous chunk of faces per thread, then the chunk sums across the block
  const int per = (F + kMsSortThreads - 1) / kMsSortThreads;
  const int f0 = min(F, tid * per), f1 = min(F, f0 + per);
  int local = 0;
  for (int f = f0; f < f1; ++f) local += first[f];
  int incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int x = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += x; }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int t = warp_tot[lane], ti = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int x = __shfl_up_sync(0xffffffffu, ti, o); if (lane >= o) ti += x; }
    warp_tot[lane] = ti - t;
  }
  __syncthreads();
  int run = warp_tot[warp] + incl - local;
  for (int f = f0; f < f1; ++f) { const int c = first[f]; first[f] = run; sb[f] = run; run += c; }
  if (tid == kMsSortThreads - 1) sb[F] = run;                               // the last thread's chunk ends at F
  __syncthreads();
  for (int i = tid; i < S * F; i += kMsSortThreads) hist[i] += first[i % F];
  __syncthreads();
  // scatter in sample-index order: segment by segment, 32 samples at a time, ranked by lane among the same face
  if (warp < S) {
    for (int base = j0; base < j1; base += 32) {
      const int j = base + lane;
      int f = j < j1 ? fb[j] : -1;
      if (f >= F) f = -1;
      const unsigned peers = __match_any_sync(0xffffffffu, f);
      int slot = 0;
      if (f >= 0) slot = hist[warp * F + f] + __popc(peers & lt);
      __syncwarp();
      if (f >= 0) {
        ob[slot] = j;
        if ((peers & lt) == 0) hist[warp * F + f] += __popc(peers);
      }
      __syncwarp();
    }
  }
}

// grid: x = blocks of kMsFaceWarps faces (one warp per face), y = mesh.  face_grad (B, F, 3 corners, 3 coordinates).
__global__ void __launch_bounds__(kMsFaceWarps * 32)
mesh_sample_face_grad_kernel(const float* __restrict__ u, const float* __restrict__ grad_points, const int* __restrict__ order,
                             const int* __restrict__ starts, float* __restrict__ face_grad, int F, int n) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int f = blockIdx.x * kMsFaceWarps + (threadIdx.x >> 5);
  if (f >= F) return;
  const int* sb = starts + (size_t)b * (F + 1);
  const int k0 = sb[f], k1 = sb[f + 1];
  float acc[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) acc[i] = 0.f;
  for (int k = k0 + lane; k < k1; k += 32) {
    const size_t j = (size_t)b * n + order[(size_t)b * n + k];
    const float* ub = u + j * 3;
    // the weights of mesh_sample_bwd_kernel, each product rounded before it is summed
    const float su = __fsqrt_rn(ub[1]), vv = ub[2];
    const float w[3] = {__fsub_rn(1.0f, su), __fmul_rn(su, __fsub_rn(1.0f, vv)), __fmul_rn(su, vv)};
    const float g[3] = {grad_points[j * 3], grad_points[j * 3 + 1], grad_points[j * 3 + 2]};
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int d = 0; d < 3; ++d) acc[3 * c + d] = __fadd_rn(acc[3 * c + d], __fmul_rn(w[c], g[d]));
  }
  float mine = 0.f;
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const float s = warp_sum(acc[i]);                                      // xor butterfly: the same bits in every lane
    if (lane == i) mine = s;
  }
  if (lane < 9) face_grad[((size_t)b * F + f) * 9 + lane] = mine;
}

// grid: x = blocks of vertices, y = mesh.  adj_entries holds 3 f + corner, grouped by vertex by adj_offsets (V + 1).
__global__ void __launch_bounds__(kMsThreads)
mesh_sample_vertex_grad_kernel(const float* __restrict__ face_grad, const int* __restrict__ adj_offsets,
                               const int* __restrict__ adj_entries, float* __restrict__ grad_verts, int V, int F) {
  const int b = blockIdx.y;
  const int v = blockIdx.x * kMsThreads + threadIdx.x;
  if (v >= V) return;
  const float* fg = face_grad + (size_t)b * F * 9;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
  for (int e = adj_offsets[v], e1 = adj_offsets[v + 1]; e < e1; ++e) {
    const float* t = fg + (size_t)adj_entries[e] * 3;
    a0 = __fadd_rn(a0, t[0]); a1 = __fadd_rn(a1, t[1]); a2 = __fadd_rn(a2, t[2]);
  }
  float* gv = grad_verts + ((size_t)b * V + v) * 3;
  gv[0] = a0; gv[1] = a1; gv[2] = a2;
}

// workspace carve-up shared by the size query and the launch
struct MsBwdLayout { size_t order, starts, face_grad, hist, total; };
inline MsBwdLayout ms_bwd_layout(int B, int F, int n) {
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  bool in_smem;
  const int S = ms_sort_segments(F, &in_smem);
  MsBwdLayout l;
  l.order = 0;
  l.starts = up((size_t)B * n * 4);
  l.face_grad = l.starts + up((size_t)B * (F + 1) * 4);
  l.hist = l.face_grad + up((size_t)B * F * 9 * 4);
  l.total = l.hist + (in_smem ? 0 : up((size_t)B * (S + 1) * F * 4));
  return l;
}

}  // namespace vpn

extern "C" int vpn_mesh_sample_fwd(const float* verts, const int* faces, const float* u, float* points, int* face_idx,
                                   float* cdf, int B, int V, int F, int n, void* stream) {
  if (B < 0 || V <= 0 || F <= 0 || n <= 0) { vpn_set_error("mesh sample fwd: bad shape B=%d V=%d F=%d n=%d", B, V, F, n); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (!verts || !faces || !u || !points || !face_idx || !cdf) { vpn_set_error("mesh sample fwd: null pointer"); return VPN_ERR_ARG; }
  if (B > 65535) { vpn_set_error("mesh sample fwd: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  cudaStream_t s = (cudaStream_t)stream;
  vpn::mesh_cdf_kernel<<<B, vpn::kMsThreads, 0, s>>>(verts, faces, cdf, V, F, 1e-10f);
  int rc = vpn_check_launch("mesh_cdf_kernel");
  if (rc) return rc;
  vpn::mesh_sample_kernel<<<dim3((n + vpn::kMsThreads - 1) / vpn::kMsThreads, B), vpn::kMsThreads, 0, s>>>(verts, faces, cdf, u, points, face_idx, V, F, n);
  return vpn_check_launch("mesh_sample_kernel");
}

extern "C" int vpn_mesh_sample_bwd(const int* faces, const float* u, const int* face_idx, const float* grad_points,
                                   float* grad_verts, int B, int V, int F, int n, void* stream) {
  if (B < 0 || V <= 0 || F <= 0 || n <= 0) { vpn_set_error("mesh sample bwd: bad shape"); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (!faces || !u || !face_idx || !grad_points || !grad_verts) { vpn_set_error("mesh sample bwd: null pointer"); return VPN_ERR_ARG; }
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(grad_verts, 0, (size_t)B * V * 3 * sizeof(float), s) != cudaSuccess) { vpn_set_error("mesh sample bwd: memset failed"); return VPN_ERR_CUDA; }
  vpn::mesh_sample_bwd_kernel<<<dim3((n + vpn::kMsThreads - 1) / vpn::kMsThreads, B), vpn::kMsThreads, 0, s>>>(faces, u, face_idx, grad_points, grad_verts, V, n);
  return vpn_check_launch("mesh_sample_bwd_kernel");
}

extern "C" int vpn_mesh_sample_bwd_workspace_bytes(int B, int F, int n, size_t* bytes) {
  if (B < 0 || F <= 0 || n <= 0 || !bytes) { vpn_set_error("mesh sample bwd workspace: bad arguments"); return VPN_ERR_ARG; }
  *bytes = vpn::ms_bwd_layout(B, F, n).total;
  return VPN_OK;
}

extern "C" int vpn_mesh_sample_bwd_sorted(const int* faces, const float* u, const int* face_idx, const float* grad_points,
                                          float* grad_verts, const int* adj_offsets, const int* adj_entries, void* workspace,
                                          size_t workspace_bytes, int B, int V, int F, int n, void* stream) {
  using namespace vpn;
  if (B < 0 || V <= 0 || F <= 0 || n <= 0) { vpn_set_error("mesh sample bwd sorted: bad shape B=%d V=%d F=%d n=%d", B, V, F, n); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (B > 65535) { vpn_set_error("mesh sample bwd sorted: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (!faces || !u || !face_idx || !grad_points || !grad_verts || !adj_offsets || !adj_entries || !workspace) {
    vpn_set_error("mesh sample bwd sorted: null pointer"); return VPN_ERR_ARG;
  }
  const MsBwdLayout l = ms_bwd_layout(B, F, n);
  if (workspace_bytes < l.total) { vpn_set_error("mesh sample bwd sorted: workspace too small (%zu < %zu)", workspace_bytes, l.total); return VPN_ERR_WORKSPACE; }
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = reinterpret_cast<char*>(workspace);
  int* order = reinterpret_cast<int*>(ws + l.order);
  int* starts = reinterpret_cast<int*>(ws + l.starts);
  float* face_grad = reinterpret_cast<float*>(ws + l.face_grad);
  int* hist = reinterpret_cast<int*>(ws + l.hist);
  bool in_smem;
  const int S = ms_sort_segments(F, &in_smem);
  const size_t smem = in_smem ? (size_t)(S + 1) * F * sizeof(int) : 0;
  static DeviceOnce once;
  if (smem > 48 * 1024 && set_dyn_smem(mesh_sample_sort_kernel, kMsSortSmemInts * 4, once) != cudaSuccess) {
    vpn_set_error("mesh sample bwd sorted: smem attribute"); return VPN_ERR_CUDA;
  }
  mesh_sample_sort_kernel<<<B, kMsSortThreads, smem, s>>>(face_idx, order, starts, hist, F, n, S, in_smem ? 1 : 0);
  int rc = vpn_check_launch("mesh_sample_sort_kernel");
  if (rc) return rc;
  mesh_sample_face_grad_kernel<<<dim3((F + kMsFaceWarps - 1) / kMsFaceWarps, B), kMsFaceWarps * 32, 0, s>>>(
      u, grad_points, order, starts, face_grad, F, n);
  rc = vpn_check_launch("mesh_sample_face_grad_kernel");
  if (rc) return rc;
  mesh_sample_vertex_grad_kernel<<<dim3((V + kMsThreads - 1) / kMsThreads, B), kMsThreads, 0, s>>>(
      face_grad, adj_offsets, adj_entries, grad_verts, V, F);
  return vpn_check_launch("mesh_sample_vertex_grad_kernel");
}
