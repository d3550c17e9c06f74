// Fused primitive instantiation: canonical surface sample (or template vertex, or caller points)
// -> scale -> rotate -> translate, forward and backward, one pass over HBM.
//
// Replaces, per primitive and per step, the ~25 ATen launches (+ 12*B .item() host syncs for cuboids)
// of the reference chain
//   modules/sampling/sphere.py:22-43, modules/sampling/cuboid.py:8-101      (canonical samplers)
//   modules/transform/rotate.py:7-72, translate.py:4-8, transform.py:6-18   (pose)
//   modules/meshing/sphere.py:8-27, cuboid.py:8-27                           (template vertices)
// HBM-bound: forward reads the uniforms (8 B sphere / 12 B cuboid per point) and writes 12 B per
// point; nothing else round-trips memory.
#include "common.cuh"

namespace vpn {

enum { KIND_SPHERE = 0, KIND_CUBOID = 1, KIND_TEMPLATE = 2, KIND_POINTS = 3 };

struct PrimShared {
  Pose pose;
  float v[3];
  float t[3];
  int cum[6];       // cuboid: inclusive prefix sums of the per-face point counts
};

// modules/sampling/cuboid.py:30-53 (get_faces_points): every op separately rounded, round-half-even.
__device__ __forceinline__ void cuboid_counts(const float* v, int N, int* cnt) {
  float w = v[0], h = v[1], d = v[2];
  float hd = __fmul_rn(h, d), dw = __fmul_rn(d, w), wh = __fmul_rn(w, h);
  float total = __fmul_rn(__fadd_rn(__fadd_rn(hd, dw), wh), 2.0f);
  float area[3] = {hd, dw, wh};
  float nf = (float)N;
  int sum = 0;
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    float wgt = __fdiv_rn(area[f >> 1], total);
    int c = (int)rintf(__fmul_rn(nf, wgt));
    cnt[f] = c; sum += c;
  }
  cnt[5] = N - sum;
}

__device__ __forceinline__ void load_prim(int KIND, PrimShared& ps, const float* v, const float* q,
                                          const float* t, int prim, int N) {
  make_pose(q + 4 * (size_t)prim, ps.pose);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    ps.v[i] = (KIND == KIND_POINTS) ? 1.0f : v[3 * (size_t)prim + i];
    ps.t[i] = t ? t[3 * (size_t)prim + i] : 0.0f;
  }
  if (KIND == KIND_CUBOID) {
    int cnt[6];
    cuboid_counts(ps.v, N, cnt);
    int run = 0;
#pragma unroll
    for (int f = 0; f < 6; ++f) { run += cnt[f]; ps.cum[f] = run; }
  }
}

// Source words per point: 2 uniforms (sphere) or 3 floats (cuboid uniforms, template vertex, caller point).
template <int KIND> struct SrcWidth { static constexpr int value = (KIND == KIND_SPHERE) ? 2 : 3; };

constexpr int kPoseThreads = 256;
constexpr int kPosePointsPerThread = 4;      // consecutive points per thread and step: 48-byte (3 x float4) accesses
constexpr int kPoseSteps = 2;                // steps per CTA: a CTA covers 2048 points of one primitive

// The source words of 4 consecutive points starting at n0, 16-byte loads when the layout allows.
template <int KIND>
__device__ __forceinline__ void load_src4(const float* __restrict__ src, size_t prim, int n0, int N, int vec_ok,
                                          float (&u)[4 * SrcWidth<KIND>::value]) {
  constexpr int W = SrcWidth<KIND>::value;
  const float* base = (KIND == KIND_TEMPLATE) ? src + (size_t)W * n0 : src + (size_t)W * (prim * (size_t)N + n0);
  if (vec_ok && n0 + 4 <= N) {
    const float4* b4 = reinterpret_cast<const float4*>(base);
#pragma unroll
    for (int i = 0; i < W; ++i) { float4 x = b4[i]; u[4 * i] = x.x; u[4 * i + 1] = x.y; u[4 * i + 2] = x.z; u[4 * i + 3] = x.w; }
  } else {
#pragma unroll
    for (int i = 0; i < 4 * W; ++i) u[i] = (n0 + i / W < N) ? base[i] : 0.f;
  }
}

// Unit "direction" d of point n such that canonical = d (.) v   (for KIND_POINTS: canonical = d); u = the point's
// source words.
template <int KIND>
__device__ __forceinline__ void canonical_dir(const PrimShared& ps, const float* u, int n, float* d) {
  if (KIND == KIND_SPHERE) {
    // sphere.py:26-27,37-43.  u = [elev draw, azim draw]
    float elev = __fadd_rn(-acosf(__fsub_rn(1.0f, __fmul_rn(2.0f, u[0]))), 1.5707963705062866f);
    float azim = __fmul_rn(__fmul_rn(u[1], 2.0f), VPN_PI);
    float ce = cosf(elev), se = sinf(elev);
    d[0] = __fmul_rn(ce, sinf(azim));
    d[1] = se;
    d[2] = __fmul_rn(ce, cosf(azim));
  } else if (KIND == KIND_CUBOID) {
    // cuboid.py:56-101.  u = three uniforms; the face of point n pins one coordinate to +-1
    d[0] = fmaf(2.0f, u[0], -1.0f);
    d[1] = fmaf(2.0f, u[1], -1.0f);
    d[2] = fmaf(2.0f, u[2], -1.0f);
    int face = 5;
#pragma unroll
    for (int f = 4; f >= 0; --f) if (n < ps.cum[f]) face = f;
    float pin = (face & 1) ? -1.0f : 1.0f;
    if ((face >> 1) == 0) d[0] = pin; else if ((face >> 1) == 1) d[1] = pin; else d[2] = pin;
  } else {
    // template vertex (meshing/sphere.py:17, cuboid.py:17) or caller point
    d[0] = u[0]; d[1] = u[1]; d[2] = u[2];
  }
}

__device__ __forceinline__ void rotate_add(const PrimShared& ps, const float* c, float* o) {
  const float* r = ps.pose.r;
  o[0] = __fadd_rn(fmaf(r[2], c[2], fmaf(r[1], c[1], r[0] * c[0])), ps.t[0]);
  o[1] = __fadd_rn(fmaf(r[5], c[2], fmaf(r[4], c[1], r[3] * c[0])), ps.t[1]);
  o[2] = __fadd_rn(fmaf(r[8], c[2], fmaf(r[7], c[1], r[6] * c[0])), ps.t[2]);
}

// One CTA's slice of one primitive: points [y * 2048, y * 2048 + 2048) of the primitive's N, y = blockIdx.y.  Its source
// rows are those of primitive src_prim of src (all of src for the shared template), its output rows those of primitive
// out_prim of out; its pose (v, q, t) is primitive prim's.
// All source loads of the CTA are issued before the pose (sin, cos, sqrt, divisions by one thread) is waited for.
template <int KIND>
__device__ __forceinline__ void pose_fwd_body(PrimShared& ps, const float* __restrict__ v, const float* __restrict__ q,
                                              const float* __restrict__ t, const float* __restrict__ src, size_t src_prim,
                                              float* __restrict__ out, size_t out_prim, size_t prim, int N, int vec_ok,
                                              unsigned tid) {
  constexpr int W = SrcWidth<KIND>::value;
  const int base_n = blockIdx.y * (kPoseThreads * kPosePointsPerThread * kPoseSteps) + tid * kPosePointsPerThread;
  pdl_enter();      // launched with launch_pdl: this CTA may already be resident while the previous kernel drains
  float u[kPoseSteps][4 * W];
#pragma unroll
  for (int s = 0; s < kPoseSteps; ++s) {
    const int n0 = base_n + s * kPoseThreads * kPosePointsPerThread;
    if (n0 < N) load_src4<KIND>(src, src_prim, n0, N, vec_ok, u[s]);
  }
  if (tid == 0) load_prim(KIND, ps, v, q, t, (int)prim, N);
  __syncthreads();
#pragma unroll
  for (int s = 0; s < kPoseSteps; ++s) {
    const int n0 = base_n + s * kPoseThreads * kPosePointsPerThread;
    if (n0 >= N) break;
    float o[kPosePointsPerThread][3];
    const int cnt = min(kPosePointsPerThread, N - n0);
#pragma unroll
    for (int i = 0; i < kPosePointsPerThread; ++i) {
      if (i < cnt) {
        float d[3], c[3];
        canonical_dir<KIND>(ps, &u[s][W * i], n0 + i, d);
        c[0] = __fmul_rn(d[0], ps.v[0]); c[1] = __fmul_rn(d[1], ps.v[1]); c[2] = __fmul_rn(d[2], ps.v[2]);
        rotate_add(ps, c, o[i]);
      }
    }
    float* dst = out + 3 * (out_prim * (size_t)N + n0);
    if (vec_ok && cnt == kPosePointsPerThread) {
      float4* d4 = reinterpret_cast<float4*>(dst);
      d4[0] = make_float4(o[0][0], o[0][1], o[0][2], o[1][0]);
      d4[1] = make_float4(o[1][1], o[1][2], o[2][0], o[2][1]);
      d4[2] = make_float4(o[2][2], o[3][0], o[3][1], o[3][2]);
    } else {
      for (int i = 0; i < cnt; ++i) { dst[3 * i] = o[i][0]; dst[3 * i + 1] = o[i][1]; dst[3 * i + 2] = o[i][2]; }
    }
  }
}

// grid: x = primitive (b*K + k), y = slice of kPoseThreads * kPosePointsPerThread * kPoseSteps points.
// Launched as a programmatic dependent launch: the launch latency overlaps the tail of the previous kernel.
template <int KIND>
__global__ void __launch_bounds__(kPoseThreads)
pose_fwd_kernel(const float* __restrict__ v, const float* __restrict__ q, const float* __restrict__ t,
                const float* __restrict__ src, float* __restrict__ out, int N, int vec_ok) {
  __shared__ PrimShared ps;
  const size_t prim = blockIdx.x;
  pose_fwd_body<KIND>(ps, v, q, t, src, prim, out, prim, prim, N, vec_ok, threadIdx.x);
}

// A mixed assembly: primitive k of every sample is a cuboid when k < Kc, else a sphere (train.py's order).
// Output row of the first point of primitive (b, k): b * (Kc*Nc + (K-Kc)*Ns) + (k < Kc ? k*Nc : Kc*Nc + (k-Kc)*Ns).
struct MixedPrim {
  bool cuboid;
  int N;
  size_t row;       // first output row
  size_t src_prim;  // index of the primitive among those of its kind (b*Kc + k or b*(K-Kc) + k-Kc)
};

__device__ __forceinline__ MixedPrim mixed_prim(int prim, int K, int Kc, int Nc, int Ns) {
  const int b = prim / K, k = prim - b * K, Ks = K - Kc;
  MixedPrim m;
  m.cuboid = k < Kc;
  m.N = m.cuboid ? Nc : Ns;
  m.row = (size_t)b * ((size_t)Kc * Nc + (size_t)Ks * Ns) + (m.cuboid ? (size_t)k * Nc : (size_t)Kc * Nc + (size_t)(k - Kc) * Ns);
  m.src_prim = m.cuboid ? (size_t)b * Kc + k : (size_t)b * Ks + (k - Kc);
  return m;
}

// One launch over all B*K primitives of a mixed assembly.  The kind is uniform across a CTA, which runs the same body
// as pose_fwd_kernel<kind> on the same source rows: the primitive's points are the bits the single-kind kernel writes.
// TEMPLATE: src_c / src_s are the cuboid / sphere templates; otherwise the (B,Kc,N,3) / (B,K-Kc,N,2) uniforms.
// grid.y covers the larger kind; CTAs past the end of a primitive's slices return.
template <bool TEMPLATE>
__global__ void __launch_bounds__(kPoseThreads)
pose_mixed_fwd_kernel(const float* __restrict__ v, const float* __restrict__ q, const float* __restrict__ t,
                      const float* __restrict__ src_c, const float* __restrict__ src_s, float* __restrict__ out,
                      int K, int Kc, int Nc, int Ns, int vec_ok) {
  __shared__ PrimShared ps;
  const int prim = blockIdx.x;
  const MixedPrim m = mixed_prim(prim, K, Kc, Nc, Ns);
  if ((int)blockIdx.y * (kPoseThreads * kPosePointsPerThread * kPoseSteps) >= m.N) return;     // before any memory access
  float* dst = out + 3 * m.row;
  if (TEMPLATE) {
    pose_fwd_body<KIND_TEMPLATE>(ps, v, q, t, m.cuboid ? src_c : src_s, 0, dst, 0, prim, m.N, vec_ok, threadIdx.x);
  } else if (m.cuboid) {
    pose_fwd_body<KIND_CUBOID>(ps, v, q, t, src_c, m.src_prim, dst, 0, prim, m.N, vec_ok, threadIdx.x);
  } else {
    pose_fwd_body<KIND_SPHERE>(ps, v, q, t, src_s, m.src_prim, dst, 0, prim, m.N, vec_ok, threadIdx.x);
  }
}

// Backward, stage 1: per block partial sums of
//   [0..8]  G = sum_n g_n (x) c_n      (dL/dR)
//   [9..11] sum_n g_n                  (dL/dt)
//   [12..14] sum_n (R^T g_n) (.) d_n   (dL/dv)
// over one CTA's slice y = blockIdx.y of one primitive, written to slot prim * gridDim.y + y of `partial` (16 floats
// a slot).  Its source rows are those of primitive src_prim of src, its gradient rows (gout, and gpts) those of
// primitive g_prim.
// KIND_POINTS also writes dL/dpoints = R^T g.
template <int KIND>
__device__ __forceinline__ void pose_bwd_partial_body(PrimShared& ps, float (&red)[kPoseThreads / 32][16],
                                                      const float* __restrict__ v, const float* __restrict__ q,
                                                      const float* __restrict__ src, size_t src_prim,
                                                      const float* __restrict__ gout, size_t g_prim,
                                                      float* __restrict__ partial, float* __restrict__ gpts, size_t prim,
                                                      int N, int vec_ok, unsigned tid) {
  constexpr int W = SrcWidth<KIND>::value;
  const int base_n = blockIdx.y * (kPoseThreads * kPosePointsPerThread * kPoseSteps) + tid * kPosePointsPerThread;
  float acc[15];
#pragma unroll
  for (int i = 0; i < 15; ++i) acc[i] = 0.f;
  // two steps' worth of loads in flight at a time (source words + upstream gradient: 6 x float4 per step)
  float u[2][4 * W], gg[2][12];
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int n0 = base_n + s * kPoseThreads * kPosePointsPerThread;
    if (n0 < N) { load_src4<KIND>(src, src_prim, n0, N, vec_ok, u[s]); load_src4<KIND_POINTS>(gout, g_prim, n0, N, vec_ok, gg[s]); }
  }
  if (tid == 0) load_prim(KIND, ps, v, q, nullptr, (int)prim, N);
  __syncthreads();
  const float* r = ps.pose.r;
#pragma unroll
  for (int s = 0; s < kPoseSteps; ++s) {
    const int n0 = base_n + s * kPoseThreads * kPosePointsPerThread;
    if (n0 < N) {
#pragma unroll
      for (int i = 0; i < kPosePointsPerThread; ++i) {
        const int n = n0 + i;
        if (n < N) {
          float d[3], c[3], rg[3];
          canonical_dir<KIND>(ps, &u[s & 1][W * i], n, d);
          const float* g = &gg[s & 1][3 * i];
#pragma unroll
          for (int a = 0; a < 3; ++a) c[a] = d[a] * ps.v[a];
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) acc[3 * a + b] += g[a] * c[b];
#pragma unroll
          for (int a = 0; a < 3; ++a) acc[9 + a] += g[a];
#pragma unroll
          for (int a = 0; a < 3; ++a) rg[a] = r[a] * g[0] + r[3 + a] * g[1] + r[6 + a] * g[2];
#pragma unroll
          for (int a = 0; a < 3; ++a) acc[12 + a] += rg[a] * d[a];
          if (KIND == KIND_POINTS && gpts) {
            float* o = gpts + 3 * (g_prim * (size_t)N + n);
            o[0] = rg[0]; o[1] = rg[1]; o[2] = rg[2];
          }
        }
      }
    }
    if (s + 2 < kPoseSteps) {
      const int n2 = base_n + (s + 2) * kPoseThreads * kPosePointsPerThread;
      if (n2 < N) { load_src4<KIND>(src, src_prim, n2, N, vec_ok, u[s & 1]); load_src4<KIND_POINTS>(gout, g_prim, n2, N, vec_ok, gg[s & 1]); }
    }
  }
  const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int i = 0; i < 15; ++i) {
    float s = warp_sum(acc[i]);
    if (lane == 0) red[warp][i] = s;
  }
  __syncthreads();
  if (tid < 15) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kPoseThreads / 32; ++w) s += red[w][tid];
    partial[(prim * gridDim.y + blockIdx.y) * 16 + tid] = s;
  }
}

// partial: slot (prim * gridDim.y + slice) of 16 floats.
template <int KIND>
__global__ void __launch_bounds__(kPoseThreads, 3)
pose_bwd_partial_kernel(const float* __restrict__ v, const float* __restrict__ q,
                        const float* __restrict__ src, const float* __restrict__ gout,
                        float* __restrict__ partial, float* __restrict__ gpts, int N, int vec_ok) {
  __shared__ PrimShared ps;
  __shared__ float red[kPoseThreads / 32][16];
  const size_t prim = blockIdx.x;
  pose_bwd_partial_body<KIND>(ps, red, v, q, src, prim, gout, prim, partial, gpts, prim, N, vec_ok, threadIdx.x);
}

// Mixed assembly (see pose_mixed_fwd_kernel): each CTA runs pose_bwd_partial_kernel<kind>'s body on its primitive's
// rows and slice, so slot (prim * gridDim.y + slice) holds the bits the single-kind kernel writes for that slice.
// Slots past a primitive's slices_for(N of its kind) are neither written nor read.  Two CTAs per SM instead of three:
// the cuboid and sphere bodies in one kernel need more than the 80 registers that three allow.
template <bool TEMPLATE>
__global__ void __launch_bounds__(kPoseThreads, 2)
pose_mixed_bwd_partial_kernel(const float* __restrict__ v, const float* __restrict__ q, const float* __restrict__ src_c,
                              const float* __restrict__ src_s, const float* __restrict__ gout, float* __restrict__ partial,
                              int K, int Kc, int Nc, int Ns, int vec_ok) {
  __shared__ PrimShared ps;
  __shared__ float red[kPoseThreads / 32][16];
  const int prim = blockIdx.x;
  const MixedPrim m = mixed_prim(prim, K, Kc, Nc, Ns);
  if ((int)blockIdx.y * (kPoseThreads * kPosePointsPerThread * kPoseSteps) >= m.N) return;
  const float* g = gout + 3 * m.row;
  if (TEMPLATE) {
    pose_bwd_partial_body<KIND_TEMPLATE>(ps, red, v, q, m.cuboid ? src_c : src_s, 0, g, 0, partial, nullptr, prim, m.N, vec_ok, threadIdx.x);
  } else if (m.cuboid) {
    pose_bwd_partial_body<KIND_CUBOID>(ps, red, v, q, src_c, m.src_prim, g, 0, partial, nullptr, prim, m.N, vec_ok, threadIdx.x);
  } else {
    pose_bwd_partial_body<KIND_SPHERE>(ps, red, v, q, src_s, m.src_prim, g, 0, partial, nullptr, prim, m.N, vec_ok, threadIdx.x);
  }
}

// Backward, stage 2 tail for one primitive: acc = its summed slots; chains dL/dR to dL/dq and stores the gradients.
__device__ __forceinline__ void pose_bwd_chain(const float* __restrict__ q, const float (&acc)[15], int prim,
                                               float* __restrict__ gv, float* __restrict__ gq, float* __restrict__ gt) {
  if (gq) {
    Pose pose; make_pose(q + 4 * (size_t)prim, pose);
    float g4[4]; pose_backward(q + 4 * (size_t)prim, pose, acc, g4);
#pragma unroll
    for (int i = 0; i < 4; ++i) gq[4 * (size_t)prim + i] = g4[i];
  }
  if (gt) { gt[3 * (size_t)prim] = acc[9]; gt[3 * (size_t)prim + 1] = acc[10]; gt[3 * (size_t)prim + 2] = acc[11]; }
  if (gv) { gv[3 * (size_t)prim] = acc[12]; gv[3 * (size_t)prim + 1] = acc[13]; gv[3 * (size_t)prim + 2] = acc[14]; }
}

// Backward, stage 2: one thread per primitive sums the slices (fixed order: deterministic) and
// chains dL/dR to dL/dq.
__global__ void pose_bwd_final_kernel(const float* __restrict__ q, const float* __restrict__ partial,
                                      float* __restrict__ gv, float* __restrict__ gq, float* __restrict__ gt,
                                      int nprim, int nslices) {
  int prim = blockIdx.x * blockDim.x + threadIdx.x;
  if (prim >= nprim) return;
  float acc[15];
#pragma unroll
  for (int i = 0; i < 15; ++i) acc[i] = 0.f;
  for (int s = 0; s < nslices; ++s) {
    const float* p = partial + ((size_t)prim * nslices + s) * 16;
#pragma unroll
    for (int i = 0; i < 15; ++i) acc[i] += p[i];
  }
  pose_bwd_chain(q, acc, prim, gv, gq, gt);
}

// Mixed assembly: primitive prim's slots start at slot prim * stride; it sums the slices_for(N of its kind) slots its
// partial CTAs wrote, in the order pose_bwd_final_kernel sums them.
__global__ void pose_mixed_bwd_final_kernel(const float* __restrict__ q, const float* __restrict__ partial,
                                            float* __restrict__ gv, float* __restrict__ gq, float* __restrict__ gt,
                                            int nprim, int K, int Kc, int ns_c, int ns_s, int stride) {
  int prim = blockIdx.x * blockDim.x + threadIdx.x;
  if (prim >= nprim) return;
  const int nslices = (prim % K) < Kc ? ns_c : ns_s;
  float acc[15];
#pragma unroll
  for (int i = 0; i < 15; ++i) acc[i] = 0.f;
  for (int s = 0; s < nslices; ++s) {
    const float* p = partial + ((size_t)prim * stride + s) * 16;
#pragma unroll
    for (int i = 0; i < 15; ++i) acc[i] += p[i];
  }
  pose_bwd_chain(q, acc, prim, gv, gq, gt);
}

__global__ void cuboid_counts_kernel(const float* __restrict__ v, int* __restrict__ counts, int nprim, int N) {
  int prim = blockIdx.x * blockDim.x + threadIdx.x;
  if (prim >= nprim) return;
  float vv[3] = {v[3 * prim], v[3 * prim + 1], v[3 * prim + 2]};
  int cnt[6]; cuboid_counts(vv, N, cnt);
#pragma unroll
  for (int f = 0; f < 6; ++f) counts[6 * prim + f] = cnt[f];
}

static inline int slices_for(int N) {
  int per = kPoseThreads * kPosePointsPerThread * kPoseSteps;
  return (N + per - 1) / per;
}

}  // namespace vpn

using namespace vpn;

extern "C" int vpn_pose_bwd_workspace_floats(int nprim, int N, size_t* floats) {
  if (nprim < 0 || N <= 0 || !floats) { vpn_set_error("pose workspace: bad arguments"); return VPN_ERR_ARG; }
  *floats = (size_t)nprim * slices_for(N) * 16;
  return VPN_OK;
}

// kind: 0 sphere (src = uniforms (nprim,N,2)), 1 cuboid (src = uniforms (nprim,N,3)),
//       2 template (src = vertices (N,3) shared), 3 points (src = points (nprim,N,3); v ignored)
extern "C" int vpn_pose_points_fwd(int kind, const float* v, const float* q, const float* t, const float* src,
                                   float* out, int nprim, int N, void* stream) {
  if (nprim < 0 || N <= 0 || kind < 0 || kind > 3) { vpn_set_error("pose fwd: bad shape/kind"); return VPN_ERR_SHAPE; }
  if (nprim == 0) return VPN_OK;
  if (!q || !src || !out || (kind != KIND_POINTS && !v)) { vpn_set_error("pose fwd: null pointer"); return VPN_ERR_ARG; }
  dim3 grid(nprim, slices_for(N)), block(kPoseThreads);
  cudaStream_t s = (cudaStream_t)stream;
  int vec_ok = (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  switch (kind) {
    case KIND_SPHERE:   launch_pdl(pose_fwd_kernel<KIND_SPHERE>, grid, block, 0, s, v, q, t, src, out, N, vec_ok); break;
    case KIND_CUBOID:   launch_pdl(pose_fwd_kernel<KIND_CUBOID>, grid, block, 0, s, v, q, t, src, out, N, vec_ok); break;
    case KIND_TEMPLATE: launch_pdl(pose_fwd_kernel<KIND_TEMPLATE>, grid, block, 0, s, v, q, t, src, out, N, vec_ok); break;
    default:            launch_pdl(pose_fwd_kernel<KIND_POINTS>, grid, block, 0, s, v, q, t, src, out, N, vec_ok); break;
  }
  return vpn_check_launch("pose_fwd_kernel");
}

// Measurement variant: `reps` forward launches back to back on `stream`, launch i reading srcs[i % nsrc] (HOST array
// of device pointers: rotate more bytes than L2 holds and every launch reads cold inputs), one CUDA-event pair around
// the whole stream of launches; *ms_per_launch (HOST) = elapsed / reps.  Synchronises.
extern "C" int vpn_pose_points_fwd_timed(int kind, const float* v, const float* q, const float* t, const float* const* srcs,
                                         int nsrc, float* out, int nprim, int N, int reps, float* ms_per_launch, void* stream) {
  if (!srcs || nsrc < 1 || reps < 1 || !ms_per_launch) { vpn_set_error("pose timed: bad arguments"); return VPN_ERR_ARG; }
  cudaStream_t s = (cudaStream_t)stream;
  cudaEvent_t e0, e1;
  if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) { vpn_set_error("pose timed: event create failed"); return VPN_ERR_CUDA; }
  int rc = VPN_OK;
  for (int i = 0; i < nsrc && rc == VPN_OK; ++i) rc = vpn_pose_points_fwd(kind, v, q, t, srcs[i], out, nprim, N, stream);   // warm-up
  cudaEventRecord(e0, s);
  for (int i = 0; i < reps && rc == VPN_OK; ++i) rc = vpn_pose_points_fwd(kind, v, q, t, srcs[i % nsrc], out, nprim, N, stream);
  cudaEventRecord(e1, s);
  if (rc == VPN_OK && cudaEventSynchronize(e1) != cudaSuccess) { vpn_set_error("pose timed: %s", cudaGetErrorString(cudaGetLastError())); rc = VPN_ERR_CUDA; }
  if (rc == VPN_OK) { float ms = 0.f; cudaEventElapsedTime(&ms, e0, e1); *ms_per_launch = ms / reps; }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return rc;
}

extern "C" int vpn_pose_points_bwd(int kind, const float* v, const float* q, const float* src, const float* grad_out,
                                   float* grad_v, float* grad_q, float* grad_t, float* grad_points,
                                   float* workspace, size_t workspace_floats, int nprim, int N, void* stream) {
  if (nprim < 0 || N <= 0 || kind < 0 || kind > 3) { vpn_set_error("pose bwd: bad shape/kind"); return VPN_ERR_SHAPE; }
  if (nprim == 0) return VPN_OK;
  if (!q || !src || !grad_out || !workspace || (kind != KIND_POINTS && !v)) { vpn_set_error("pose bwd: null pointer"); return VPN_ERR_ARG; }
  int ns = slices_for(N);
  if (workspace_floats < (size_t)nprim * ns * 16) { vpn_set_error("pose bwd: workspace too small"); return VPN_ERR_WORKSPACE; }
  dim3 grid(nprim, ns), block(kPoseThreads);
  cudaStream_t s = (cudaStream_t)stream;
  int vec_ok = (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(grad_out) & 15) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  switch (kind) {
    case KIND_SPHERE:   pose_bwd_partial_kernel<KIND_SPHERE><<<grid, block, 0, s>>>(v, q, src, grad_out, workspace, nullptr, N, vec_ok); break;
    case KIND_CUBOID:   pose_bwd_partial_kernel<KIND_CUBOID><<<grid, block, 0, s>>>(v, q, src, grad_out, workspace, nullptr, N, vec_ok); break;
    case KIND_TEMPLATE: pose_bwd_partial_kernel<KIND_TEMPLATE><<<grid, block, 0, s>>>(v, q, src, grad_out, workspace, nullptr, N, vec_ok); break;
    default:            pose_bwd_partial_kernel<KIND_POINTS><<<grid, block, 0, s>>>(v, q, src, grad_out, workspace, grad_points, N, vec_ok); break;
  }
  int rc = vpn_check_launch("pose_bwd_partial_kernel");
  if (rc) return rc;
  pose_bwd_final_kernel<<<(nprim + 127) / 128, 128, 0, s>>>(q, workspace, kind == KIND_POINTS ? nullptr : grad_v,
                                                              grad_q, grad_t, nprim, ns);
  return vpn_check_launch("pose_bwd_final_kernel");
}

// Mixed cuboid + sphere assemblies: primitive b*K + k is a cuboid when k < Kc, else a sphere.
// mode 0 = sampled: src_c = cuboid uniforms (B,Kc,N,3), src_s = sphere uniforms (B,K-Kc,N,2), Nc = Ns = N;
// mode 1 = template: src_c = cuboid template (Nc,3), src_s = sphere template (Ns,3).
// out (B, Kc*Nc + (K-Kc)*Ns, 3).  A kind without primitives may pass a NULL source.
static int mixed_args(const char* what, int mode, int B, int K, int Kc, int Nc, int Ns, const float* src_c,
                      const float* src_s) {
  if (mode != 0 && mode != 1) { vpn_set_error("%s: mode must be 0 (sampled) or 1 (template)", what); return VPN_ERR_ARG; }
  if (B <= 0 || K <= 0 || Nc <= 0 || Ns <= 0 || Kc < 0 || Kc > K || (mode == 0 && Nc != Ns)) {
    vpn_set_error("%s: bad shape B=%d K=%d Kc=%d Nc=%d Ns=%d", what, B, K, Kc, Nc, Ns);
    return VPN_ERR_SHAPE;
  }
  if ((Kc > 0 && !src_c) || (Kc < K && !src_s)) { vpn_set_error("%s: null source for a kind that is present", what); return VPN_ERR_ARG; }
  return VPN_OK;
}

static int mixed_slices(int K, int Kc, int Nc, int Ns) {
  return max(Kc > 0 ? slices_for(Nc) : 0, Kc < K ? slices_for(Ns) : 0);
}

// 16-byte accesses when every primitive's rows start on a 16-byte boundary: point counts of the present kinds divisible
// by 4 (row offsets are then multiples of 4 points) and aligned base pointers.
static int mixed_vec_ok(int K, int Kc, int Nc, int Ns, const float* src_c, const float* src_s, const float* rows) {
  auto al = [](const float* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return (Kc == 0 || (Nc % 4 == 0 && al(src_c))) && (Kc == K || (Ns % 4 == 0 && al(src_s))) && al(rows);
}

extern "C" int vpn_pose_mixed_fwd(int mode, const float* v, const float* q, const float* t, const float* src_c,
                                  const float* src_s, float* out, int B, int K, int Kc, int Nc, int Ns, void* stream) {
  int rc = mixed_args("pose mixed fwd", mode, B, K, Kc, Nc, Ns, src_c, src_s);
  if (rc) return rc;
  if (!v || !q || !out) { vpn_set_error("pose mixed fwd: null pointer"); return VPN_ERR_ARG; }
  dim3 grid(B * K, mixed_slices(K, Kc, Nc, Ns)), block(kPoseThreads);
  cudaStream_t s = (cudaStream_t)stream;
  int vec_ok = mixed_vec_ok(K, Kc, Nc, Ns, src_c, src_s, out);
  if (mode == 1) launch_pdl(pose_mixed_fwd_kernel<true>, grid, block, 0, s, v, q, t, src_c, src_s, out, K, Kc, Nc, Ns, vec_ok);
  else           launch_pdl(pose_mixed_fwd_kernel<false>, grid, block, 0, s, v, q, t, src_c, src_s, out, K, Kc, Nc, Ns, vec_ok);
  return vpn_check_launch("pose_mixed_fwd_kernel");
}

extern "C" int vpn_pose_mixed_bwd_workspace_floats(int B, int K, int Kc, int Nc, int Ns, size_t* floats) {
  if (B <= 0 || K <= 0 || Nc <= 0 || Ns <= 0 || Kc < 0 || Kc > K) { vpn_set_error("pose mixed workspace: bad shape"); return VPN_ERR_SHAPE; }
  if (!floats) { vpn_set_error("pose mixed workspace: null pointer"); return VPN_ERR_ARG; }
  *floats = (size_t)B * K * mixed_slices(K, Kc, Nc, Ns) * 16;
  return VPN_OK;
}

// grad_out (B, Kc*Nc + (K-Kc)*Ns, 3) -> grad_v (B*K,3), grad_q (B*K,4), grad_t (B*K,3); any may be NULL.
extern "C" int vpn_pose_mixed_bwd(int mode, const float* v, const float* q, const float* src_c, const float* src_s,
                                  const float* grad_out, float* grad_v, float* grad_q, float* grad_t, float* workspace,
                                  size_t workspace_floats, int B, int K, int Kc, int Nc, int Ns, void* stream) {
  int rc = mixed_args("pose mixed bwd", mode, B, K, Kc, Nc, Ns, src_c, src_s);
  if (rc) return rc;
  if (!v || !q || !grad_out || !workspace) { vpn_set_error("pose mixed bwd: null pointer"); return VPN_ERR_ARG; }
  const int ns = mixed_slices(K, Kc, Nc, Ns), nprim = B * K;
  if (workspace_floats < (size_t)nprim * ns * 16) { vpn_set_error("pose mixed bwd: workspace too small"); return VPN_ERR_WORKSPACE; }
  dim3 grid(nprim, ns), block(kPoseThreads);
  cudaStream_t s = (cudaStream_t)stream;
  int vec_ok = mixed_vec_ok(K, Kc, Nc, Ns, src_c, src_s, grad_out);
  if (mode == 1) pose_mixed_bwd_partial_kernel<true><<<grid, block, 0, s>>>(v, q, src_c, src_s, grad_out, workspace, K, Kc, Nc, Ns, vec_ok);
  else           pose_mixed_bwd_partial_kernel<false><<<grid, block, 0, s>>>(v, q, src_c, src_s, grad_out, workspace, K, Kc, Nc, Ns, vec_ok);
  rc = vpn_check_launch("pose_mixed_bwd_partial_kernel");
  if (rc) return rc;
  pose_mixed_bwd_final_kernel<<<(nprim + 127) / 128, 128, 0, s>>>(q, workspace, grad_v, grad_q, grad_t, nprim, K, Kc,
                                                                    slices_for(Nc), slices_for(Ns), ns);
  return vpn_check_launch("pose_mixed_bwd_final_kernel");
}

extern "C" int vpn_cuboid_face_counts(const float* v, int* counts, int nprim, int N, void* stream) {
  if (nprim < 0 || N <= 0) { vpn_set_error("cuboid counts: bad shape"); return VPN_ERR_SHAPE; }
  if (nprim == 0) return VPN_OK;
  if (!v || !counts) { vpn_set_error("cuboid counts: null pointer"); return VPN_ERR_ARG; }
  cuboid_counts_kernel<<<(nprim + 127) / 128, 128, 0, (cudaStream_t)stream>>>(v, counts, nprim, N);
  return vpn_check_launch("cuboid_counts_kernel");
}
