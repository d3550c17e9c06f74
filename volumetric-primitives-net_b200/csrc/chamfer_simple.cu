// Chamfer nearest-neighbour search, generic path + backward.
//
// Reference arithmetic (modules/loss/chamfer_distance.py:14-23), per pair:
//   d = fl(fl(fl(dx*dx) + fl(dy*dy)) + fl(dz*dz)),  dx = fl(p.x - t.x) ...   (no FMA contraction)
//   v = sqrt(d);  min over the other cloud;  ties -> FIRST index (torch.min).
// This file holds the shape-agnostic kernel (any P, M >= 1): used for ragged clouds and as the
// on-device cross-check of the tiled kernel in chamfer_tiled.cu.  Both directions are the same kernel
// with the clouds swapped.  Results are combined across column segments with a 64-bit atomicMin on
// (float_bits(v) << 32 | index): for non-negative floats that orders by value, then by lowest
// index, which is exactly the reference's tie rule, independent of scheduling.
// A small first cloud (P <= kSmallP; VP-diverse: P = K = 16, modules/loss/vp_diverse.py:12-18) has its
// own one-launch forward and one-launch gather backward, a thread-block cluster per sample.  Also here:
// the backward of the other shapes and the loss head of chamfer_distance.py:25-30.
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace vpn {

constexpr int kSimpleThreads = 128;
constexpr int kSimpleRows = 2;            // rows per thread
constexpr int kSimpleTile = 1024;         // columns staged in shared memory per step

__device__ __forceinline__ float exact_d2(float ax, float ay, float az, float bx, float by, float bz) {
  float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// rows: cloud A (B, nA, 3) ; cols: cloud B (B, nB, 3).  key (B, nA) u64, pre-filled with 0xFF..FF.
// grid: x = row block, y = column segment, z = sample.
__global__ void __launch_bounds__(kSimpleThreads)
chamfer_simple_kernel(const float* __restrict__ A, const float* __restrict__ Bp, u64* __restrict__ key,
                      int nA, int nB, int seg_len) {
  __shared__ float4 tile[kSimpleTile];
  const int b = blockIdx.z;
  const float* a = A + (size_t)b * nA * 3;
  const float* t = Bp + (size_t)b * nB * 3;
  const int row0 = (blockIdx.x * kSimpleThreads + threadIdx.x) * kSimpleRows;
  float px[kSimpleRows], py[kSimpleRows], pz[kSimpleRows];
  float best_d[kSimpleRows], best_v[kSimpleRows];
  int best_j[kSimpleRows];
#pragma unroll
  for (int r = 0; r < kSimpleRows; ++r) {
    int i = min(row0 + r, nA - 1);
    px[r] = a[3 * (size_t)i]; py[r] = a[3 * (size_t)i + 1]; pz[r] = a[3 * (size_t)i + 2];
    best_d[r] = __int_as_float(0x7f800000); best_v[r] = best_d[r]; best_j[r] = 0;
  }
  const int c_begin = blockIdx.y * seg_len;
  const int c_end = min(nB, c_begin + seg_len);
  for (int c0 = c_begin; c0 < c_end; c0 += kSimpleTile) {
    const int cnt = min(kSimpleTile, c_end - c0);
    __syncthreads();
    for (int k = threadIdx.x; k < cnt; k += kSimpleThreads) {
      const float* s = t + 3 * (size_t)(c0 + k);
      tile[k] = make_float4(s[0], s[1], s[2], 0.f);
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < cnt; ++k) {
      float4 q = tile[k];
#pragma unroll
      for (int r = 0; r < kSimpleRows; ++r) {
        float d = exact_d2(px[r], py[r], pz[r], q.x, q.y, q.z);
        if (d < best_d[r]) {
          // Rare path.  d improves the squared distance; the index only moves if the ROUNDED sqrt
          // improves too, because the reference minimises sqrt(d) and keeps the first index of a tie.
          float v = sqrtf(d);
          if (v < best_v[r]) { best_v[r] = v; best_j[r] = c0 + k; }
          best_d[r] = d;
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < kSimpleRows; ++r) {
    int i = row0 + r;
    if (i < nA && c_begin < c_end) {
      u64 kv = ((u64)__float_as_uint(best_v[r]) << 32) | (unsigned)best_j[r];
      atomicMin(&key[(size_t)b * nA + i], kv);
    }
  }
}

__global__ void chamfer_unpack_kernel(const u64* __restrict__ key, float* __restrict__ mn, int* __restrict__ idx, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 k = key[i];
  mn[i] = __uint_as_float((unsigned)(k >> 32));
  idx[i] = (int)(unsigned)(k & 0xffffffffu);
}

// Backward (what autograd does through chamfer_distance.py:14-23 given the arg-mins):
//   row term : dL/dp1[i] = (g1[i] / (2 v1[i])) * 2 (p1[i] - p2[idx1[i]])          -> plain store
//   col term : dL/dp1[idx2[j]] += (g2[j] / (2 v2[j])) * 2 (p1[idx2[j]] - p2[j])    -> atomic scatter (P > kSmallP)
// and the negatives into dL/dp2 when requested.  v == 0 gives inf * 0 = NaN, as in the reference.
//
// Upstream gradient of min1 / min2 (Upstream): a full tensor g (B,n); or the per-sample gradient gl (B) of the fused
// loss w1*mean(min1) + w2*mean(min2) times `scale` (= w1/P or w2/M); or, for the batch mean weight * mean_b(loss_b), the
// scalar gl[0]: ((gl[0] * weight) * (1/B)) * scale.  That is autograd's order through `loss.mean() * weight`: the mul
// backward, then the mean backward (torch divides a CUDA tensor by a scalar as a multiply by its float reciprocal), then
// the per-sample scale, so the points' gradients are the bits of the torch composition.
struct Upstream {
  const float* g;         // (B,n) or NULL
  const float* gl;        // (B) per-sample, or (1) when inv_count != 0
  float scale, weight, inv_count;
};
__device__ __forceinline__ float upstream(const Upstream& u, int b, size_t k) {
  if (u.g) return u.g[k];
  const float gb = u.inv_count != 0.f ? __fmul_rn(__fmul_rn(u.gl[0], u.weight), u.inv_count) : u.gl[b];
  return __fmul_rn(gb, u.scale);
}

// One thread = 4 consecutive rows: the streamed operands (points 48 B, arg-mins 16 B, minima 16 B) and the result (48 B)
// move as 16-byte accesses when the layout allows (vec_ok: P % 4 == 0 and 16-byte aligned bases); only the gathered
// targets are scalar loads.  HBM bound: (12 + 4 + 4 + 12) B streamed + 12 B gathered per row.
__global__ void __launch_bounds__(256)
chamfer_bwd_rows_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                        const float* __restrict__ min1, const int* __restrict__ idx1,
                        const Upstream u1, float* __restrict__ gp1, float* __restrict__ gp2, int P, int M, int vec_ok) {
  const int b = blockIdx.y;
  const int i0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i0 >= P) return;
  const size_t r0 = (size_t)b * P + i0;
  const int cnt = min(4, P - i0);
  const float* g1 = u1.g;
  float a[12], mn[4], up[4], o[12];
  int j[4];
  if (vec_ok) {
    const float4* a4 = reinterpret_cast<const float4*>(p1 + 3 * r0);
    const float4 x0 = a4[0], x1 = a4[1], x2 = a4[2];
    const int4 jj = *reinterpret_cast<const int4*>(idx1 + r0);
    const float4 mm = *reinterpret_cast<const float4*>(min1 + r0);
    a[0] = x0.x; a[1] = x0.y; a[2] = x0.z; a[3] = x0.w; a[4] = x1.x; a[5] = x1.y; a[6] = x1.z; a[7] = x1.w;
    a[8] = x2.x; a[9] = x2.y; a[10] = x2.z; a[11] = x2.w;
    j[0] = jj.x; j[1] = jj.y; j[2] = jj.z; j[3] = jj.w;
    mn[0] = mm.x; mn[1] = mm.y; mn[2] = mm.z; mn[3] = mm.w;
    if (g1) { const float4 gg = *reinterpret_cast<const float4*>(g1 + r0); up[0] = gg.x; up[1] = gg.y; up[2] = gg.z; up[3] = gg.w; }
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const bool ok = k < cnt;
      j[k] = ok ? idx1[r0 + k] : 0; mn[k] = ok ? min1[r0 + k] : 1.f;
      if (g1) up[k] = ok ? g1[r0 + k] : 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) a[3 * k + c] = ok ? p1[3 * (r0 + k) + c] : 0.f;
    }
  }
  if (!g1) { const float u = upstream(u1, b, 0); up[0] = up[1] = up[2] = up[3] = u; }
  float t[12];
#pragma unroll
  for (int k = 0; k < 4; ++k) {                          // the four gathers are in flight together
    const float* tp = p2 + 3 * ((size_t)b * M + j[k]);
    t[3 * k] = tp[0]; t[3 * k + 1] = tp[1]; t[3 * k + 2] = tp[2];
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float coef = up[k] / (2.0f * mn[k]);
#pragma unroll
    for (int c = 0; c < 3; ++c) o[3 * k + c] = coef * (2.0f * (a[3 * k + c] - t[3 * k + c]));
  }
  if (vec_ok) {
    float4* o4 = reinterpret_cast<float4*>(gp1 + 3 * r0);
    o4[0] = make_float4(o[0], o[1], o[2], o[3]); o4[1] = make_float4(o[4], o[5], o[6], o[7]); o4[2] = make_float4(o[8], o[9], o[10], o[11]);
  } else {
    for (int k = 0; k < cnt; ++k) { gp1[3 * (r0 + k)] = o[3 * k]; gp1[3 * (r0 + k) + 1] = o[3 * k + 1]; gp1[3 * (r0 + k) + 2] = o[3 * k + 2]; }
  }
  if (gp2) {
    for (int k = 0; k < cnt; ++k) {
      float* q = gp2 + 3 * ((size_t)b * M + j[k]);
      atomicAdd(q, -o[3 * k]); atomicAdd(q + 1, -o[3 * k + 1]); atomicAdd(q + 2, -o[3 * k + 2]);
    }
  }
}

static inline int bwd_rows_vec_ok(const float* p1, const float* min1, const int* idx1, const float* g1, const float* gp1, int P) {
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return (P % 4 == 0) && al(p1) && al(min1) && al(idx1) && al(gp1) && (g1 == nullptr || al(g1));
}

// P > kSmallP only: one thread per target, global atomic scatter into the arg-min row.
__global__ void chamfer_bwd_cols_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                                        const float* __restrict__ min2, const int* __restrict__ idx2, const Upstream u2,
                                        float* __restrict__ gp1, float* __restrict__ gp2, int P, int M) {
  const int b = blockIdx.y;
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= M) return;
  size_t cj = (size_t)b * M + j;
  int i = idx2[cj];
  const float* a = p1 + 3 * ((size_t)b * P + i);
  const float* t = p2 + 3 * cj;
  float up = upstream(u2, b, cj);
  float coef = up / (2.0f * min2[cj]);
  float cx = coef * (2.0f * (a[0] - t[0])), cy = coef * (2.0f * (a[1] - t[1])), cz = coef * (2.0f * (a[2] - t[2]));
  float* o = gp1 + 3 * ((size_t)b * P + i);
  atomicAdd(o, cx); atomicAdd(o + 1, cy); atomicAdd(o + 2, cz);
  if (gp2) {
    float* o2 = gp2 + 3 * cj;
    atomicAdd(o2, -cx); atomicAdd(o2 + 1, -cy); atomicAdd(o2 + 2, -cz);
  }
}

// ---- Small first cloud (P <= kSmallP: the K primitive centres of VP-diverse, vp_diverse.py:12-18) ----
// A thread-block cluster per sample; CTA r of the cluster owns the targets of slice r.  The cluster size depends on M
// only (never on B), so a sample's results are the same bits alone and inside any batch.
constexpr int kSmallP = 256;
constexpr int kSmallMaxCluster = 16;                          // non-portable cluster size (B200 allows 16)
constexpr int kSmallFwdThreads = 512;
constexpr int kSmallFwdTargets = 2;                           // targets per thread per pass
constexpr int kSmallSlice = kSmallFwdThreads * kSmallFwdTargets;

static int smallp_cluster(int M) { return min(kSmallMaxCluster, (M + kSmallSlice - 1) / kSmallSlice); }

// Forward, both directions in one launch, no global atomics.  Column minimum: each target walks the P centres in
// ascending order (first index on ties).  Row minima: per centre, the (float_bits(v) << 32 | j) keys of a warp are
// reduced with two __reduce_min_sync and kept per warp in shared memory, then per CTA, then across the cluster's CTAs
// through distributed shared memory.  A minimum of exact keys does not depend on the order it is taken in: the results
// are the reference's bits (IEEE sqrt, first index on ties).
__global__ void __launch_bounds__(kSmallFwdThreads)
chamfer_smallp_fwd_kernel(const float* __restrict__ p1, const float* __restrict__ p2, float* __restrict__ min1,
                          int* __restrict__ idx1, float* __restrict__ min2, int* __restrict__ idx2, int P, int M) {
  constexpr int NW = kSmallFwdThreads / 32, T = kSmallFwdTargets;
  __shared__ float4 cen[kSmallP];
  __shared__ u64 wkey[NW * kSmallP];                          // [warp][centre]; wkey[0..P) then holds the CTA's minima
  cg::cluster_group cluster = cg::this_cluster();
  const int b = blockIdx.y, rank = (int)cluster.block_rank(), CL = (int)cluster.num_blocks();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = threadIdx.x; k < P; k += kSmallFwdThreads) {
    const float* a = p1 + 3 * ((size_t)b * P + k);
    cen[k] = make_float4(a[0], a[1], a[2], 0.f);
  }
  for (int k = threadIdx.x; k < NW * P; k += kSmallFwdThreads) wkey[k] = ~0ull;
  __syncthreads();
  const float* tb = p2 + 3 * (size_t)b * M;
  for (int base = rank * kSmallSlice; base < M; base += CL * kSmallSlice) {
    float tx[T], ty[T], tz[T], bv[T];
    int bi[T], j[T];
#pragma unroll
    for (int r = 0; r < T; ++r) {
      j[r] = base + threadIdx.x + r * kSmallFwdThreads;
      const float* t = tb + 3 * (size_t)min(j[r], M - 1);
      tx[r] = t[0]; ty[r] = t[1]; tz[r] = t[2];
      bv[r] = __int_as_float(0x7f800000); bi[r] = 0;
    }
    for (int k = 0; k < P; ++k) {
      const float4 c = cen[k];
      unsigned tv = 0xffffffffu, tj = 0xffffffffu;
#pragma unroll
      for (int r = 0; r < T; ++r) {
        const float v = sqrtf(exact_d2(c.x, c.y, c.z, tx[r], ty[r], tz[r]));
        if (v < bv[r]) { bv[r] = v; bi[r] = k; }                 // ascending k: first index on ties
        const unsigned vb = j[r] < M ? __float_as_uint(v) : 0xffffffffu;
        if (vb < tv) { tv = vb; tj = (unsigned)j[r]; }           // ascending j within the thread
      }
      const unsigned vmin = __reduce_min_sync(0xffffffffu, tv);
      const unsigned jmin = __reduce_min_sync(0xffffffffu, tv == vmin ? tj : 0xffffffffu);
      if (lane == 0 && vmin != 0xffffffffu) {
        const u64 key = ((u64)vmin << 32) | jmin;
        if (key < wkey[warp * P + k]) wkey[warp * P + k] = key;  // this lane is the slot's only writer
      }
    }
#pragma unroll
    for (int r = 0; r < T; ++r)
      if (j[r] < M) { min2[(size_t)b * M + j[r]] = bv[r]; idx2[(size_t)b * M + j[r]] = bi[r]; }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < P; k += kSmallFwdThreads) {
    u64 m = wkey[k];
    for (int w = 1; w < NW; ++w) m = min(m, wkey[w * P + k]);
    wkey[k] = m;
  }
  cluster.sync();
  for (int k = rank + CL * threadIdx.x; k < P; k += CL * kSmallFwdThreads) {
    u64 m = ~0ull;
    for (int r = 0; r < CL; ++r) m = min(m, *cluster.map_shared_rank(&wkey[k], r));
    min1[(size_t)b * P + k] = __uint_as_float((unsigned)(m >> 32));
    idx1[(size_t)b * P + k] = (int)(unsigned)(m & 0xffffffffu);
  }
  cluster.sync();                                             // the other CTAs' shared memory stays alive until read
}

// Backward, one gather launch, no memset and no atomics: grad_p1 (and grad_p2) are written with plain stores.
// Every CTA computes the row terms of all P centres.  CTA r stages the column terms of its target slice, chunk by
// chunk, and sums them per centre in a fixed order: G = threads / P parts per centre, part g taking every G-th target
// of the chunk in ascending order; then the parts in order.  The CTAs' sums are added in rank order through
// distributed shared memory, and the row term is added last.  grad_p2[j] = (sum, ascending i, of -row term i over the
// centres whose arg-min is j) - column term j, the order the atomic path's memset / row / column passes apply.
constexpr int kSmallBwdThreads = 256;
constexpr int kSmallBwdChunk = 1024;

__global__ void __launch_bounds__(kSmallBwdThreads)
chamfer_smallp_bwd_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                          const float* __restrict__ min1, const int* __restrict__ idx1,
                          const float* __restrict__ min2, const int* __restrict__ idx2, const Upstream u1, const Upstream u2,
                          float* __restrict__ gp1, float* __restrict__ gp2, int P, int M, int slice) {
  __shared__ float ro[kSmallP * 3];                           // row term of every centre
  __shared__ int ix1[kSmallP];
  __shared__ float4 cc[kSmallBwdChunk];                       // column term (x, y, z) and arg-min centre of a target
  __shared__ float part[kSmallBwdThreads * 3];
  __shared__ float csum[kSmallP * 3];                         // this CTA's column sum per centre
  cg::cluster_group cluster = cg::this_cluster();
  const int b = blockIdx.y, rank = (int)cluster.block_rank(), CL = (int)cluster.num_blocks();
  for (int i = threadIdx.x; i < P; i += kSmallBwdThreads) {
    const size_t r = (size_t)b * P + i;
    const int j = idx1[r];
    const float* a = p1 + 3 * r;
    const float* t = p2 + 3 * ((size_t)b * M + j);
    const float coef = upstream(u1, b, r) / (2.0f * min1[r]);
#pragma unroll
    for (int c = 0; c < 3; ++c) ro[3 * i + c] = coef * (2.0f * (a[c] - t[c]));
    ix1[i] = j;
  }
  const int G = kSmallBwdThreads / P, ci = threadIdx.x % P, g = threadIdx.x / P;
  const bool scan = threadIdx.x < G * P;
  float sx = 0.f, sy = 0.f, sz = 0.f;
  const int j0 = min(M, rank * slice), j1 = min(M, j0 + slice);
  for (int c0 = j0; c0 < j1; c0 += kSmallBwdChunk) {
    const int n = min(kSmallBwdChunk, j1 - c0);
    __syncthreads();                                          // row terms ready / previous chunk consumed
    for (int s = threadIdx.x; s < n; s += kSmallBwdThreads) {
      const int j = c0 + s;
      const size_t cj = (size_t)b * M + j;
      const int i = idx2[cj];
      const float* a = p1 + 3 * ((size_t)b * P + i);
      const float* t = p2 + 3 * cj;
      const float coef = upstream(u2, b, cj) / (2.0f * min2[cj]);
      const float cx = coef * (2.0f * (a[0] - t[0])), cy = coef * (2.0f * (a[1] - t[1])), cz = coef * (2.0f * (a[2] - t[2]));
      cc[s] = make_float4(cx, cy, cz, __int_as_float(i));
      if (gp2) {
        float gx = 0.f, gy = 0.f, gz = 0.f;
        for (int q = 0; q < P; ++q)
          if (ix1[q] == j) { gx += -ro[3 * q]; gy += -ro[3 * q + 1]; gz += -ro[3 * q + 2]; }
        gp2[3 * cj] = gx + -cx; gp2[3 * cj + 1] = gy + -cy; gp2[3 * cj + 2] = gz + -cz;
      }
    }
    __syncthreads();
    if (scan) {
#pragma unroll 4
      for (int s = g; s < n; s += G) {
        const float4 e = cc[s];
        if (__float_as_int(e.w) == ci) { sx += e.x; sy += e.y; sz += e.z; }
      }
    }
  }
  if (scan) { part[3 * threadIdx.x] = sx; part[3 * threadIdx.x + 1] = sy; part[3 * threadIdx.x + 2] = sz; }
  __syncthreads();
  for (int i = threadIdx.x; i < P; i += kSmallBwdThreads) {
    float x = 0.f, y = 0.f, z = 0.f;
    for (int q = 0; q < G; ++q) { x += part[3 * (q * P + i)]; y += part[3 * (q * P + i) + 1]; z += part[3 * (q * P + i) + 2]; }
    csum[3 * i] = x; csum[3 * i + 1] = y; csum[3 * i + 2] = z;
  }
  cluster.sync();
  for (int i = rank + CL * threadIdx.x; i < P; i += CL * kSmallBwdThreads) {
    float x = 0.f, y = 0.f, z = 0.f;
    for (int r = 0; r < CL; ++r) {
      const float* s = cluster.map_shared_rank(csum, r);
      x += s[3 * i]; y += s[3 * i + 1]; z += s[3 * i + 2];
    }
    float* o = gp1 + 3 * ((size_t)b * P + i);
    o[0] = ro[3 * i] + x; o[1] = ro[3 * i + 1] + y; o[2] = ro[3 * i + 2] + z;
  }
  cluster.sync();
}

// grid (CL, B), one cluster of CL CTAs per sample
template <typename K, typename... Args>
static int launch_small_cluster(K kernel, const char* name, int threads, int B, int CL, cudaStream_t s, DeviceOnce& once,
                                Args... args) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  const unsigned long long bit = dev >= 0 && dev < 64 ? (1ull << dev) : 0ull;
  if (e == cudaSuccess && CL > 8 && !(bit && (once.mask.load(std::memory_order_acquire) & bit))) {
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e == cudaSuccess && bit) once.mask.fetch_or(bit, std::memory_order_release);
  }
  if (e != cudaSuccess) { vpn_set_error("%s: cluster attribute: %s", name, cudaGetErrorString(e)); return VPN_ERR_CUDA; }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)CL, (unsigned)B); cfg.blockDim = dim3(threads); cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, kernel, args...);
  if (e != cudaSuccess) { vpn_set_error("%s: launch: %s", name, cudaGetErrorString(e)); return VPN_ERR_CUDA; }
  return vpn_check_launch(name);
}

// Backward of both directions: the gather kernel for a small first cloud, else the row pass (plain stores) followed by
// the column pass (atomic scatter).  grad_p1 is overwritten; grad_p2 (optional) too.
static int chamfer_bwd_launch(const float* p1, const float* p2, const float* min1, const int* idx1, const float* min2,
                              const int* idx2, const Upstream& u1, const Upstream& u2, float* grad_p1, float* grad_p2,
                              int B, int P, int M, cudaStream_t s) {
  if (P <= kSmallP) {
    static DeviceOnce once;
    const int CL = smallp_cluster(M);
    return launch_small_cluster(chamfer_smallp_bwd_kernel, "chamfer_smallp_bwd_kernel", kSmallBwdThreads, B, CL, s, once,
                                p1, p2, min1, idx1, min2, idx2, u1, u2, grad_p1, grad_p2, P, M, (M + CL - 1) / CL);
  }
  if (grad_p2 && cudaMemsetAsync(grad_p2, 0, (size_t)B * M * 3 * sizeof(float), s) != cudaSuccess) {
    vpn_set_error("chamfer bwd: memset failed"); return VPN_ERR_CUDA;
  }
  chamfer_bwd_rows_kernel<<<dim3((P + 1023) / 1024, B), 256, 0, s>>>(p1, p2, min1, idx1, u1, grad_p1, grad_p2, P, M,
                                                                     bwd_rows_vec_ok(p1, min1, idx1, u1.g, grad_p1, P));
  int rc = vpn_check_launch("chamfer_bwd_rows_kernel");
  if (rc) return rc;
  chamfer_bwd_cols_kernel<<<dim3((M + 255) / 256, B), 256, 0, s>>>(p1, p2, min2, idx2, u2, grad_p1, grad_p2, P, M);
  return vpn_check_launch("chamfer_bwd_cols_kernel");
}

// per sample: loss[b] = w1 * mean(min1[b]) + w2 * mean(min2[b])      (chamfer_distance.py:25-28)
// stage 1: kLossSlices blocks per sample write partial sums; stage 2 adds them in a fixed order (deterministic).
constexpr int kLossSlices = 32;

__global__ void __launch_bounds__(256)
chamfer_loss_partial_kernel(const float* __restrict__ min1, const float* __restrict__ min2,
                            float2* __restrict__ partial, int P, int M) {
  __shared__ float red[2][8];
  const int b = blockIdx.y, sl = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float s1 = 0.f, s2 = 0.f;
  for (int i = sl * blockDim.x + threadIdx.x; i < P; i += blockDim.x * kLossSlices) s1 += min1[(size_t)b * P + i];
  for (int i = sl * blockDim.x + threadIdx.x; i < M; i += blockDim.x * kLossSlices) s2 += min2[(size_t)b * M + i];
  s1 = warp_sum(s1); s2 = warp_sum(s2);
  if (lane == 0) { red[0][warp] = s1; red[1][warp] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c = 0.f;
    for (int w = 0; w < 8; ++w) { a += red[0][w]; c += red[1][w]; }
    partial[(size_t)b * kLossSlices + sl] = make_float2(a, c);
  }
}

// loss (optional): the per-sample values.  mean (optional, one block): weight * (sum_b loss[b] / B), each thread adding its
// samples in ascending b, then the threads in a fixed tree (warp shuffles, then the warps in order).
constexpr int kLossFinalThreads = 128;

__global__ void __launch_bounds__(kLossFinalThreads)
chamfer_loss_final_kernel(const float2* __restrict__ partial, float w1, float w2, float* __restrict__ loss,
                          float* __restrict__ mean, float weight, int B, int P, int M) {
  __shared__ float red[kLossFinalThreads / 32];
  float s = 0.f;
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    float a = 0.f, c = 0.f;
    for (int k = 0; k < kLossSlices; ++k) { float2 v = partial[(size_t)b * kLossSlices + k]; a += v.x; c += v.y; }
    const float l = __fmaf_rn(w1, a / (float)P, __fmul_rn(w2, c / (float)M));     // the contraction nvcc chose before
    if (loss) loss[b] = l;
    s += l;
  }
  if (!mean) return;
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kLossFinalThreads / 32; ++w) t += red[w];
    mean[0] = weight * (t / (float)B);
  }
}

// one direction: for every row of A the nearest column of Bp
int chamfer_simple_direction(const float* A, const float* Bp, float* mn, int* idx, u64* key,
                             int B, int nA, int nB, int sm_count, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(key, 0xFF, (size_t)B * nA * sizeof(u64), s);
  if (e != cudaSuccess) { vpn_set_error("chamfer: memset failed: %s", cudaGetErrorString(e)); return VPN_ERR_CUDA; }
  int row_blocks = (nA + kSimpleThreads * kSimpleRows - 1) / (kSimpleThreads * kSimpleRows);
  // split the columns so that small row counts still fill the SMs
  long long want = 4LL * sm_count;
  int segs = (int)((want + (long long)row_blocks * B - 1) / ((long long)row_blocks * B));
  int max_segs = (nB + kSimpleTile - 1) / kSimpleTile;
  if (segs > max_segs) segs = max_segs;
  if (segs < 1) segs = 1;
  int seg_len = (nB + segs - 1) / segs;
  seg_len = ((seg_len + 31) / 32) * 32;
  segs = (nB + seg_len - 1) / seg_len;
  dim3 grid(row_blocks, segs, B);
  chamfer_simple_kernel<<<grid, kSimpleThreads, 0, s>>>(A, Bp, key, nA, nB, seg_len);
  int rc = vpn_check_launch("chamfer_simple_kernel");
  if (rc) return rc;
  size_t n = (size_t)B * nA;
  chamfer_unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(key, mn, idx, n);
  return vpn_check_launch("chamfer_unpack_kernel");
}

// both directions in one launch for a small first cloud (P <= kSmallP)
int chamfer_smallp(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                   int B, int P, int M, cudaStream_t s) {
  static DeviceOnce once;
  return launch_small_cluster(chamfer_smallp_fwd_kernel, "chamfer_smallp_fwd_kernel", kSmallFwdThreads, B, smallp_cluster(M),
                              s, once, p1, p2, min1, idx1, min2, idx2, P, M);
}
int chamfer_smallp_limit() { return kSmallP; }

}  // namespace vpn

using namespace vpn;

extern "C" int vpn_chamfer_bwd(const float* p1, const float* p2, const float* min1, const int* idx1,
                               const float* min2, const int* idx2, const float* g1, const float* g2,
                               float* grad_p1, float* grad_p2, int B, int P, int M, void* stream) {
  if (B < 0 || P <= 0 || M <= 0) { vpn_set_error("chamfer bwd: bad shape"); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (B > 65535) { vpn_set_error("chamfer bwd: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (!p1 || !p2 || !min1 || !idx1 || !min2 || !idx2 || !g1 || !g2 || !grad_p1) {
    vpn_set_error("chamfer bwd: null pointer"); return VPN_ERR_ARG;
  }
  const Upstream u1 = {g1, nullptr, 0.f, 0.f, 0.f}, u2 = {g2, nullptr, 0.f, 0.f, 0.f};
  return chamfer_bwd_launch(p1, p2, min1, idx1, min2, idx2, u1, u2, grad_p1, grad_p2, B, P, M, (cudaStream_t)stream);
}

static int chamfer_loss_head(const float* min1, const float* min2, float w1, float w2, float* loss, float* mean,
                             float weight, float* scratch, int B, int P, int M, cudaStream_t s) {
  float2* partial = reinterpret_cast<float2*>(scratch);
  chamfer_loss_partial_kernel<<<dim3(kLossSlices, B), 256, 0, s>>>(min1, min2, partial, P, M);
  int rc = vpn_check_launch("chamfer_loss_partial_kernel");
  if (rc) return rc;
  const int blocks = mean ? 1 : (B + kLossFinalThreads - 1) / kLossFinalThreads;
  chamfer_loss_final_kernel<<<blocks, kLossFinalThreads, 0, s>>>(partial, w1, w2, loss, mean, weight, B, P, M);
  return vpn_check_launch("chamfer_loss_final_kernel");
}

// scratch: >= 64 * B floats of device memory (partial sums)
extern "C" int vpn_chamfer_loss_fwd(const float* min1, const float* min2, float w1, float w2, float* loss,
                                    float* scratch, int B, int P, int M, void* stream) {
  if (B < 0 || P <= 0 || M <= 0) { vpn_set_error("chamfer loss: bad shape"); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (B > 65535) { vpn_set_error("chamfer loss: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (!min1 || !min2 || !loss || !scratch) { vpn_set_error("chamfer loss: null pointer"); return VPN_ERR_ARG; }
  return chamfer_loss_head(min1, min2, w1, w2, loss, nullptr, 0.f, scratch, B, P, M, (cudaStream_t)stream);
}

extern "C" int vpn_chamfer_loss_bwd(const float* p1, const float* p2, const float* min1, const int* idx1,
                                    const float* min2, const int* idx2, const float* grad_loss, float w1, float w2,
                                    float* grad_p1, float* grad_p2, int B, int P, int M, void* stream) {
  if (B < 0 || P <= 0 || M <= 0) { vpn_set_error("chamfer loss bwd: bad shape"); return VPN_ERR_SHAPE; }
  if (B == 0) return VPN_OK;
  if (B > 65535) { vpn_set_error("chamfer loss bwd: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (!p1 || !p2 || !min1 || !idx1 || !min2 || !idx2 || !grad_loss || !grad_p1) {
    vpn_set_error("chamfer loss bwd: null pointer"); return VPN_ERR_ARG;
  }
  const Upstream u1 = {nullptr, grad_loss, w1 / (float)P, 0.f, 0.f}, u2 = {nullptr, grad_loss, w2 / (float)M, 0.f, 0.f};
  return chamfer_bwd_launch(p1, p2, min1, idx1, min2, idx2, u1, u2, grad_p1, grad_p2, B, P, M, (cudaStream_t)stream);
}

// loss (1 float) = weight * mean over b of (w1*mean(min1[b]) + w2*mean(min2[b])); scratch: >= 64 * B floats
extern "C" int vpn_chamfer_loss_mean_fwd(const float* min1, const float* min2, float w1, float w2, float weight,
                                         float* loss, float* scratch, int B, int P, int M, void* stream) {
  if (B <= 0 || P <= 0 || M <= 0) { vpn_set_error("chamfer loss mean: bad shape B=%d P=%d M=%d", B, P, M); return VPN_ERR_SHAPE; }
  if (B > 65535) { vpn_set_error("chamfer loss mean: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (!min1 || !min2 || !loss || !scratch) { vpn_set_error("chamfer loss mean: null pointer"); return VPN_ERR_ARG; }
  return chamfer_loss_head(min1, min2, w1, w2, nullptr, loss, weight, scratch, B, P, M, (cudaStream_t)stream);
}

// grad_loss: the scalar upstream gradient of vpn_chamfer_loss_mean_fwd's output, read on the device
extern "C" int vpn_chamfer_loss_mean_bwd(const float* p1, const float* p2, const float* min1, const int* idx1,
                                         const float* min2, const int* idx2, const float* grad_loss, float w1, float w2,
                                         float weight, float* grad_p1, float* grad_p2, int B, int P, int M, void* stream) {
  if (B <= 0 || P <= 0 || M <= 0) { vpn_set_error("chamfer loss mean bwd: bad shape B=%d P=%d M=%d", B, P, M); return VPN_ERR_SHAPE; }
  if (B > 65535) { vpn_set_error("chamfer loss mean bwd: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (!p1 || !p2 || !min1 || !idx1 || !min2 || !idx2 || !grad_loss || !grad_p1) {
    vpn_set_error("chamfer loss mean bwd: null pointer"); return VPN_ERR_ARG;
  }
  const float inv_b = 1.0f / (float)B;
  const Upstream u1 = {nullptr, grad_loss, w1 / (float)P, weight, inv_b}, u2 = {nullptr, grad_loss, w2 / (float)M, weight, inv_b};
  return chamfer_bwd_launch(p1, p2, min1, idx1, min2, idx2, u1, u2, grad_p1, grad_p2, B, P, M, (cudaStream_t)stream);
}
