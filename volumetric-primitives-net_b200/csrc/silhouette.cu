// Differentiable soft-silhouette rasteriser (alpha channel of DIB-R's VertexColor renderer).
//
// Replaces the per-sample loop of modules/loss/silhouette.py:13-23 over
// modules/render/vertex_renderer.py:15-26 -> kaolin.graphics.DIBRenderer.forward (third party, not
// vendored by the reference): here the whole batch is one launch per stage.
//   project  : one thread per vertex  - camera transform + perspective divide
//   faces    : one thread per face    - screen triangle (x multiplier), front-face flag, normal
//   raster   : one CTA per 16x16 screen tile and sample - faces are binned per tile in shared memory
//              IN FACE-INDEX ORDER (ballot + prefix popcount), because DIB-R's soft term is order
//              dependent: only the first `knum` faces whose expanded bbox holds the pixel count.
//   backward : same binning; per uncovered pixel the <= knum recorded faces are differentiated and
//              scattered with atomics into a per-face screen-space gradient buffer (B,F,6), which a
//              last kernel chains through the projection into vertex gradients.
// Arithmetic follows DIB-R's expression order operation by operation (explicit
// round-to-nearest intrinsics, no FMA contraction; the order is written out in DESIGN.md): the algorithm works on coordinates scaled by
// 1000 and is cancellation prone, so a different rounding sequence moves alpha by ~1e-3.
#include "common.cuh"

namespace vpn {

constexpr int kTile = 16;
constexpr int kRThreads = kTile * kTile;
constexpr int kKnumMax = 32;

struct RasterParams {
  int H, W, F, knum;
  float expand, mult, delta, eps;
  int cull_soft;      // 1: back faces (normal.z < 0) are skipped by the soft pass too; 0 (DIB-R): only by the coverage pass
};

struct __align__(16) FaceRec { float ax, ay, bx, by, cx, cy, front, pad; };

__device__ __forceinline__ float min3(float a, float b, float c) { return fminf(fminf(a, b), c); }
__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// cam = rot (v - pos);  xy = (cam.xy * proj.xy) / (cam.z * proj.z)
__global__ void sil_project_kernel(const float* __restrict__ verts, const float* __restrict__ rot,
                                   const float* __restrict__ pos, float px, float py, float pz,
                                   float* __restrict__ cam, float* __restrict__ xy, int V) {
  const int b = blockIdx.y;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const float* r = rot + 9 * (size_t)b;
  const float* p = pos + 3 * (size_t)b;
  const float* v = verts + 3 * ((size_t)b * V + i);
  float dx = __fsub_rn(v[0], p[0]), dy = __fsub_rn(v[1], p[1]), dz = __fsub_rn(v[2], p[2]);
  float c[3];
#pragma unroll
  for (int k = 0; k < 3; ++k)
    c[k] = __fadd_rn(__fadd_rn(__fmul_rn(dx, r[3 * k]), __fmul_rn(dy, r[3 * k + 1])), __fmul_rn(dz, r[3 * k + 2]));
  float* co = cam + 3 * ((size_t)b * V + i);
  co[0] = c[0]; co[1] = c[1]; co[2] = c[2];
  float zz = __fmul_rn(c[2], pz);
  float* o = xy + 2 * ((size_t)b * V + i);
  o[0] = __fdiv_rn(__fmul_rn(c[0], px), zz);
  o[1] = __fdiv_rn(__fmul_rn(c[1], py), zz);
}

// Also writes, per GROUP of 32 consecutive faces (one warp here; 8 groups = one binning step of the rasteriser), the
// union of the expanded bounding boxes of the faces that can matter: (min xmin, max xmax, min ymin, max ymax).
__global__ void __launch_bounds__(256)
sil_faces_kernel(const float* __restrict__ cam, const float* __restrict__ xy,
                 const int* __restrict__ faces, FaceRec* __restrict__ rec,
                 float* __restrict__ normals, float4* __restrict__ group_box, int V, int F, float mult, float em,
                 int cull_soft) {
  const int b = blockIdx.y;
  int f = blockIdx.x * blockDim.x + threadIdx.x;
  const float inf = __int_as_float(0x7f800000);
  float4 box = make_float4(inf, -inf, inf, -inf);
  if (f < F) {
  int i0 = faces[3 * f], i1 = faces[3 * f + 1], i2 = faces[3 * f + 2];
  const float* c0 = cam + 3 * ((size_t)b * V + i0);
  const float* c1 = cam + 3 * ((size_t)b * V + i1);
  const float* c2 = cam + 3 * ((size_t)b * V + i2);
  float e1x = __fsub_rn(c1[0], c0[0]), e1y = __fsub_rn(c1[1], c0[1]), e1z = __fsub_rn(c1[2], c0[2]);
  float e2x = __fsub_rn(c2[0], c0[0]), e2y = __fsub_rn(c2[1], c0[1]), e2z = __fsub_rn(c2[2], c0[2]);
  float nx = __fsub_rn(__fmul_rn(e1y, e2z), __fmul_rn(e1z, e2y));
  float ny = __fsub_rn(__fmul_rn(e1z, e2x), __fmul_rn(e1x, e2z));
  float nz = __fsub_rn(__fmul_rn(e1x, e2y), __fmul_rn(e1y, e2x));
  const float* s0 = xy + 2 * ((size_t)b * V + i0);
  const float* s1 = xy + 2 * ((size_t)b * V + i1);
  const float* s2 = xy + 2 * ((size_t)b * V + i2);
  FaceRec r;
  r.ax = __fmul_rn(s0[0], mult); r.ay = __fmul_rn(s0[1], mult);
  r.bx = __fmul_rn(s1[0], mult); r.by = __fmul_rn(s1[1], mult);
  r.cx = __fmul_rn(s2[0], mult); r.cy = __fmul_rn(s2[1], mult);
  r.front = (nz >= 0.0f) ? 1.0f : 0.0f;      // kaolin: `if (direction < 0) continue;`
  r.pad = 0.f;
  // A face with a non-finite coordinate (a NaN vertex, or one on the camera plane: cam.z = 0) takes part in neither
  // pass.  fminf / fmaxf drop NaN, so one NaN vertex would still leave a box around the other two: all six coordinates
  // become NaN, every box test of walk_warp_faces fails, and the face's group box below stays empty.
  const bool finite = isfinite(r.ax) && isfinite(r.ay) && isfinite(r.bx) && isfinite(r.by) && isfinite(r.cx) && isfinite(r.cy);
  if (!finite) r.ax = r.ay = r.bx = r.by = r.cx = r.cy = __int_as_float(0x7fffffff);
  rec[(size_t)b * F + f] = r;
  if (normals) {
    float len = sqrtf(nx * nx + ny * ny + nz * nz) + 1e-15f;
    float* n = normals + 3 * ((size_t)b * F + f);
    n[0] = nx / len; n[1] = ny / len; n[2] = nz / len;
  }
  if (finite && (r.front > 0.5f || !cull_soft))
    box = make_float4(__fsub_rn(min3(r.ax, r.bx, r.cx), em), __fadd_rn(max3(r.ax, r.bx, r.cx), em),
                      __fsub_rn(min3(r.ay, r.by, r.cy), em), __fadd_rn(max3(r.ay, r.by, r.cy), em));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    box.x = fminf(box.x, __shfl_xor_sync(0xffffffffu, box.x, o)); box.y = fmaxf(box.y, __shfl_xor_sync(0xffffffffu, box.y, o));
    box.z = fminf(box.z, __shfl_xor_sync(0xffffffffu, box.z, o)); box.w = fmaxf(box.w, __shfl_xor_sync(0xffffffffu, box.w, o));
  }
  if ((threadIdx.x & 31) == 0) group_box[((size_t)b * gridDim.x + blockIdx.x) * 8 + (threadIdx.x >> 5)] = box;
}

// Squared distance pixel -> triangle, DIB-R's 6 cases; returns d2 and the winning case (first minimum).
__device__ __forceinline__ float tri_dist2(const FaceRec& r, float X, float Y, float mult, float eps, int& which) {
  const float vx[3] = {r.ax, r.bx, r.cx}, vy[3] = {r.ay, r.by, r.cy};
  float best = 0.f; which = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    float x1 = vx[i], y1 = vy[i], x2 = vx[(i + 1) % 3], y2 = vy[(i + 1) % 3];
    float A = __fsub_rn(y2, y1), Bc = __fsub_rn(x1, x2);
    float C = __fsub_rn(__fmul_rn(x2, y1), __fmul_rn(x1, y2));
    float up = __fadd_rn(__fadd_rn(__fmul_rn(A, X), __fmul_rn(Bc, Y)), C);
    float down = __fadd_rn(__fmul_rn(A, A), __fmul_rn(Bc, Bc));
    float de = __fadd_rn(down, eps);
    float AB = __fmul_rn(A, Bc);
    float x3 = __fdiv_rn(__fsub_rn(__fsub_rn(__fmul_rn(__fmul_rn(Bc, Bc), X), __fmul_rn(AB, Y)), __fmul_rn(A, C)), de);
    float y3 = __fdiv_rn(__fsub_rn(__fsub_rn(__fmul_rn(__fmul_rn(A, A), Y), __fmul_rn(AB, X)), __fmul_rn(Bc, C)), de);
    float direct = __fadd_rn(__fmul_rn(__fsub_rn(x3, x1), __fsub_rn(x3, x2)), __fmul_rn(__fsub_rn(y3, y1), __fsub_rn(y3, y2)));
    float pd = (direct > 0.f) ? __fmul_rn(__fmul_rn(4.f, mult), mult) : __fdiv_rn(__fmul_rn(up, up), de);
    if (i == 0 || pd < best) { best = pd; which = i; }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    float ddx = __fsub_rn(X, vx[i]), ddy = __fsub_rn(Y, vy[i]);
    float pd = __fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy));
    if (pd < best) { best = pd; which = 3 + i; }
  }
  return best;
}

__device__ __forceinline__ bool inside_tri(const FaceRec& r, float X, float Y, float eps) {
  float m = __fsub_rn(r.bx, r.ax), p = __fsub_rn(r.by, r.ay), n = __fsub_rn(r.cx, r.ax), q = __fsub_rn(r.cy, r.ay);
  float s = __fsub_rn(X, r.ax), t = __fsub_rn(Y, r.ay);
  float k1 = __fsub_rn(__fmul_rn(s, q), __fmul_rn(n, t));
  float k2 = __fsub_rn(__fmul_rn(m, t), __fmul_rn(s, p));
  float k3 = __fadd_rn(__fsub_rn(__fmul_rn(m, q), __fmul_rn(n, p)), eps);
  float w1 = __fdiv_rn(k1, k3), w2 = __fdiv_rn(k2, k3);
  float w0 = __fsub_rn(__fsub_rn(1.0f, w1), w2);
  return w0 >= 0.f && w1 >= 0.f && w2 >= 0.f;
}

// Warp-autonomous face walker: calls fn(face_index, record, tight bbox) on every lane for the faces that can touch the
// calling WARP's 8 x 4 pixel block (wxL..wyT: pixel-centre extent), in face-index order, with no block-level barrier.
// (A CTA-cooperative binning was measured first: 41 % of its stall samples were warps waiting at the per-batch
// __syncthreads for the warp with the most faces - profiles/r02a_ncu_lines_raster.md.)
//   1. groups of 32 consecutive faces whose union box (sil_faces_kernel) misses the block are never loaded: the lanes
//      test 32 group boxes at a time;
//   2. of a live group, lane l holds face 32 g + l and tests its expanded box against the block; the hits are broadcast
//      one by one (7 shuffles) and every lane runs fn on its own pixel.
// The next live group's records are in flight while the current group's hits are walked.
template <typename Fn>
__device__ __forceinline__ void walk_warp_faces(const FaceRec* __restrict__ rec, const float4* __restrict__ group_box,
                                                int F, float wxL, float wxR, float wyB, float wyT, float em, int cull_soft,
                                                Fn fn) {
  const int lane = threadIdx.x & 31;
  const int ngroups = (F + 31) >> 5;
  for (int g0 = 0; g0 < ngroups; g0 += 32) {
    bool live = false;
    if (g0 + lane < ngroups) {
      const float4 bb = group_box[g0 + lane];
      live = bb.x <= wxR && bb.y > wxL && bb.z <= wyT && bb.w > wyB;
    }
    unsigned groups = __ballot_sync(0xffffffffu, live);
    if (!groups) continue;
    int g = g0 + __ffs((int)groups) - 1;
    groups &= groups - 1;
    FaceRec rnext;
    bool have = g * 32 + lane < F;
    if (have) rnext = rec[g * 32 + lane];
    while (true) {
      const FaceRec r = rnext;
      const int fbase = g * 32;
      bool hit = false;
      if (have) {
        const float xmin = __fsub_rn(min3(r.ax, r.bx, r.cx), em), xmax = __fadd_rn(max3(r.ax, r.bx, r.cx), em);
        const float ymin = __fsub_rn(min3(r.ay, r.by, r.cy), em), ymax = __fadd_rn(max3(r.ay, r.by, r.cy), em);
        hit = (r.front > 0.5f || !cull_soft) && xmin <= wxR && xmax > wxL && ymin <= wyT && ymax > wyB;
      }
      const bool more = groups != 0u;
      if (more) {
        g = g0 + __ffs((int)groups) - 1;
        groups &= groups - 1;
        have = g * 32 + lane < F;
        if (have) rnext = rec[g * 32 + lane];
      }
      for (unsigned bits = __ballot_sync(0xffffffffu, hit); bits; bits &= bits - 1) {
        const int src = __ffs((int)bits) - 1;
        FaceRec q;
        q.ax = __shfl_sync(0xffffffffu, r.ax, src); q.ay = __shfl_sync(0xffffffffu, r.ay, src);
        q.bx = __shfl_sync(0xffffffffu, r.bx, src); q.by = __shfl_sync(0xffffffffu, r.by, src);
        q.cx = __shfl_sync(0xffffffffu, r.cx, src); q.cy = __shfl_sync(0xffffffffu, r.cy, src);
        q.front = __shfl_sync(0xffffffffu, r.front, src); q.pad = 0.f;
        const float4 tb = make_float4(min3(q.ax, q.bx, q.cx), max3(q.ax, q.bx, q.cx), min3(q.ay, q.by, q.cy), max3(q.ay, q.by, q.cy));
        fn(fbase + src, q, tb);
      }
      if (!more) break;
    }
  }
}

// Thread / list slot p of a tile -> pixel inside the tile: a warp covers an 8 x 4 block (not a 16 x 2 strip), which
// makes its footprint small in both directions for the warp-level face cull of walk_tile_faces.
__device__ __forceinline__ void tile_px(int p, int& px, int& py) {
  const int warp = p >> 5, lane = p & 31;
  px = ((warp & 1) << 3) + (lane & 7);
  py = ((warp >> 1) << 2) + (lane >> 3);
}

__device__ __forceinline__ void pixel_coords(const RasterParams& rp, int w, int h, float& X, float& Y) {
  X = __fmul_rn(__fdiv_rn(rp.mult, (float)rp.W), (float)(2 * w + 1 - rp.W));
  Y = __fmul_rn(__fdiv_rn(rp.mult, (float)rp.H), (float)(rp.H - 2 * h - 1));
}

// Per-tile candidate lists in dynamic shared memory, [k][pixel] so that a pixel's thread writes conflict free, sized by the
// call's knum (30 in DIB-R: 53.8 KB for the backward - four CTAs per SM where kKnumMax rows allowed three):
//   backward  fac f32 [knum][256] prob, cand u16 [knum][256] face index of the pixel's k-th soft candidate (F <= 65535),
//             which u8 [knum][256] winning distance case
//   forward   ONE u32 [knum][256]: the face index until the item has been evaluated, then the bits of 1 - prob (the lane
//             that evaluates an item is the only one to read its face index): 30 KB, five CTAs per SM
struct TileLists { unsigned short* cand; float* fac; unsigned char* which; };
__device__ __forceinline__ TileLists tile_lists(unsigned char* p, int knum) {
  TileLists t;
  t.fac = reinterpret_cast<float*>(p); p += (size_t)knum * kRThreads * sizeof(float);
  t.cand = reinterpret_cast<unsigned short*>(p); p += (size_t)knum * kRThreads * sizeof(unsigned short);
  t.which = p;
  return t;
}
__host__ __device__ inline size_t tile_list_bytes_fwd(int knum) { return (size_t)knum * kRThreads * sizeof(unsigned); }
__host__ __device__ inline size_t tile_list_bytes_bwd(int knum) { return (size_t)knum * kRThreads * (sizeof(float) + sizeof(unsigned short) + 1); }

// Exclusive prefix sum of cnt over the warp's 32 pixels; *total = sum.
__device__ __forceinline__ int warp_offsets(int cnt, int* total) {
  const int lane = threadIdx.x & 31;
  int inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  *total = __shfl_sync(0xffffffffu, inc, 31);
  return inc - cnt;
}
// lane (pixel of the warp) that owns work item `it`: largest p with off_p <= it (off = this lane's exclusive offset)
__device__ __forceinline__ int item_lane(int off, int it) {
  int lo = 0, hi = 31;
#pragma unroll
  for (int step = 0; step < 5; ++step) {
    const int mid = (lo + hi + 1) >> 1;
    if (__shfl_sync(0xffffffffu, off, mid) <= it) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// The soft term costs ~200 instructions per (pixel, face) pair and only a few pixels of a warp lie inside a face's
// expanded box, so a warp does its 8 x 4 pixel block in three passes (warp-synchronous, no block barrier anywhere):
//   A  pixel-parallel, cheap: walk the faces in index order; coverage test; remember the first knum candidates
//   B  work-parallel, dense : one (pixel, candidate) item per lane - distance, prob            (all lanes busy)
//   C  pixel-parallel       : product of the pixel's factors in candidate order (the order DIB-R multiplies in)
// grid: x = tile x, y = tile y, z = sample; CTA = 8 warps = one 16 x 16 tile
__global__ void __launch_bounds__(kRThreads)
sil_raster_fwd_kernel(const FaceRec* __restrict__ rec_all, const float4* __restrict__ box_all, float* __restrict__ alpha,
                      unsigned char* __restrict__ covered_out, RasterParams rp) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  unsigned* slot = reinterpret_cast<unsigned*>(s_dyn);           // [k][pixel]: face index, then the bits of 1 - prob
  const int b = blockIdx.z, tid = threadIdx.x, lane = tid & 31, wbase = tid & ~31;
  int px, py; tile_px(tid, px, py);
  const int w = blockIdx.x * kTile + px, h = blockIdx.y * kTile + py;
  const bool in_img = (w < rp.W && h < rp.H);
  if (!__any_sync(0xffffffffu, in_img)) return;
  const FaceRec* rec = rec_all + (size_t)b * rp.F;
  float X, Y; pixel_coords(rp, min(w, rp.W - 1), min(h, rp.H - 1), X, Y);
  // pixel-centre extent of this warp's 8 x 4 block (x grows with w, y shrinks with h)
  float wxL, wxR, wyT, wyB;
  pixel_coords(rp, min(w - (px & 7), rp.W - 1), min(h - (py & 3), rp.H - 1), wxL, wyT);
  pixel_coords(rp, min(w - (px & 7) + 7, rp.W - 1), min(h - (py & 3) + 3, rp.H - 1), wxR, wyB);
  const float em = __fmul_rn(rp.expand, rp.mult);
  bool covered = false; int cnt = 0;
  const float4* boxes = box_all + (size_t)b * ((rp.F + kRThreads - 1) / kRThreads) * 8;
  walk_warp_faces(rec, boxes, rp.F, wxL, wxR, wyB, wyT, em, rp.cull_soft, [&](int f, const FaceRec& r, const float4& tb) {
    if (covered) return;                                // alpha is 1 whatever follows
    const float txmin = tb.x, txmax = tb.y, tymin = tb.z, tymax = tb.w;
    if (!(X >= __fsub_rn(txmin, em) && X < __fadd_rn(txmax, em) && Y >= __fsub_rn(tymin, em) && Y < __fadd_rn(tymax, em))) return;
    // coverage (hard pass): front faces only.  A back face that holds the pixel is an ordinary soft candidate.
    if (r.front > 0.5f && X >= txmin && X < txmax && Y >= tymin && Y < tymax && inside_tri(r, X, Y, rp.eps)) { covered = true; return; }
    if (cnt < rp.knum) { slot[cnt * kRThreads + tid] = (unsigned)f; ++cnt; }
  });
  const int mine = (in_img && !covered) ? cnt : 0;
  int total;
  const int off = warp_offsets(mine, &total);
  __syncwarp();
  for (int it = lane; it < ((total + 31) & ~31); it += 32) {
    const bool on = it < total;
    const int pl = item_lane(off, on ? it : 0);                           // all lanes take part in the shuffles
    const int k = it - __shfl_sync(0xffffffffu, off, pl);
    const float PX = __shfl_sync(0xffffffffu, X, pl), PY = __shfl_sync(0xffffffffu, Y, pl);
    if (on) {
      const FaceRec r = rec[slot[k * kRThreads + wbase + pl]];
      int which;
      const float d2 = tri_dist2(r, PX, PY, rp.mult, rp.eps, which);
      const float z = __fdiv_rn(__fdiv_rn(__fmul_rn(rp.delta, d2), rp.mult), rp.mult);
      slot[k * kRThreads + wbase + pl] = __float_as_uint(__fsub_rn(1.0f, expf(-z)));
    }
  }
  __syncwarp();
  if (in_img) {
    float prod = 1.0f;
    for (int k = 0; k < mine; ++k) prod = __fmul_rn(prod, __uint_as_float(slot[k * kRThreads + tid]));
    const size_t o = ((size_t)b * rp.H + h) * rp.W + w;
    alpha[o] = covered ? 1.0f : __fsub_rn(1.0f, prod);
    covered_out[o] = covered ? 1 : 0;
  }
}

// Backward of the soft term: d alpha / d (scaled screen coords of the recorded faces).  Same three passes; pass C is
// work-parallel too: one (pixel, candidate) item per lane, scattered into the per-face buffer with atomics.
__global__ void __launch_bounds__(kRThreads)
sil_raster_bwd_kernel(const FaceRec* __restrict__ rec_all, const float4* __restrict__ box_all, const float* __restrict__ galpha,
                      const unsigned char* __restrict__ covered_in, float* __restrict__ gface, RasterParams rp) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  const TileLists tl = tile_lists(s_dyn, rp.knum);
  const int b = blockIdx.z, tid = threadIdx.x, lane = tid & 31, wbase = tid & ~31;
  int px, py; tile_px(tid, px, py);
  const int w = blockIdx.x * kTile + px, h = blockIdx.y * kTile + py;
  const bool in_img = (w < rp.W && h < rp.H);
  const FaceRec* rec = rec_all + (size_t)b * rp.F;
  float X, Y; pixel_coords(rp, min(w, rp.W - 1), min(h, rp.H - 1), X, Y);
  float wxL, wxR, wyT, wyB;
  pixel_coords(rp, min(w - (px & 7), rp.W - 1), min(h - (py & 3), rp.H - 1), wxL, wyT);
  pixel_coords(rp, min(w - (px & 7) + 7, rp.W - 1), min(h - (py & 3) + 3, rp.H - 1), wxR, wyB);
  const float em = __fmul_rn(rp.expand, rp.mult);
  float g = 0.f; bool active = false;
  if (in_img) {
    size_t o = ((size_t)b * rp.H + h) * rp.W + w;
    g = galpha[o];
    active = (covered_in[o] == 0) && (g != 0.f);
  }
  if (!__any_sync(0xffffffffu, active)) return;         // blocks without an uncovered pixel that has a gradient do nothing
  int cnt = 0;
  const float4* boxes = box_all + (size_t)b * ((rp.F + kRThreads - 1) / kRThreads) * 8;
  walk_warp_faces(rec, boxes, rp.F, wxL, wxR, wyB, wyT, em, rp.cull_soft, [&](int f, const FaceRec& r, const float4& tb) {
    if (!active || cnt >= rp.knum) return;
    const float txmin = tb.x, txmax = tb.y, tymin = tb.z, tymax = tb.w;
    if (!(X >= __fsub_rn(txmin, em) && X < __fadd_rn(txmax, em) && Y >= __fsub_rn(tymin, em) && Y < __fadd_rn(tymax, em))) return;
    tl.cand[cnt * kRThreads + tid] = (unsigned short)f; ++cnt;
  });
  int total;
  const int off = warp_offsets(cnt, &total);
  if (total == 0) return;
  __syncwarp();
  const int padded = (total + 31) & ~31;
  for (int it = lane; it < padded; it += 32) {
    const bool on = it < total;
    const int pl = item_lane(off, on ? it : 0);
    const int k = it - __shfl_sync(0xffffffffu, off, pl);
    const float PX = __shfl_sync(0xffffffffu, X, pl), PY = __shfl_sync(0xffffffffu, Y, pl);
    if (on) {
      const FaceRec r = rec[tl.cand[k * kRThreads + wbase + pl]];
      int which;
      const float d2 = tri_dist2(r, PX, PY, rp.mult, rp.eps, which);
      const float z = __fdiv_rn(__fdiv_rn(__fmul_rn(rp.delta, d2), rp.mult), rp.mult);
      tl.fac[k * kRThreads + wbase + pl] = expf(-z);
      tl.which[k * kRThreads + wbase + pl] = (unsigned char)which;
    }
  }
  __syncwarp();
  for (int it = lane; it < padded; it += 32) {
    const bool on = it < total;
    const int pl = item_lane(off, on ? it : 0);
    const int offp = __shfl_sync(0xffffffffu, off, pl), n = __shfl_sync(0xffffffffu, cnt, pl);
    const float PX = __shfl_sync(0xffffffffu, X, pl), PY = __shfl_sync(0xffffffffu, Y, pl), gp = __shfl_sync(0xffffffffu, g, pl);
    if (!on) continue;
    const int k = it - offp, p = wbase + pl;
    // alpha = 1 - prod_j (1 - p_j);  d alpha / d p_k = prod_{j != k} (1 - p_j), multiplied in the order prefix * suffix
    float prefix = 1.0f, suffix = 1.0f;
    for (int j = 0; j < k; ++j) prefix *= (1.0f - tl.fac[j * kRThreads + p]);
    for (int j = n - 1; j > k; --j) suffix *= (1.0f - tl.fac[j * kRThreads + p]);
    const float dadp = prefix * suffix;
    const float prob = tl.fac[k * kRThreads + p];
    const int which = tl.which[k * kRThreads + p];
    const int f = tl.cand[k * kRThreads + p];
    const FaceRec r = rec[f];
    // p = exp(-delta d2 / mult^2)  ->  dp/dd2 = -p delta / mult^2
    const float gd2 = gp * dadp * (-prob) * rp.delta / (rp.mult * rp.mult);
    float gr[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float vx[3] = {r.ax, r.bx, r.cx}, vy[3] = {r.ay, r.by, r.cy};
    if (which < 3) {
      const int i1 = which, i2 = (which + 1) % 3;
      const float x1 = vx[i1], y1 = vy[i1], x2 = vx[i2], y2 = vy[i2];
      const float A = y2 - y1, Bc = x1 - x2, C = x2 * y1 - x1 * y2;
      const float up = A * PX + Bc * PY + C, de = A * A + Bc * Bc + rp.eps;
      const float gU = gd2 * 2.0f * up / de, gD = -gd2 * up * up / (de * de);
      const float gA = gU * PX + gD * 2.0f * A, gB = gU * PY + gD * 2.0f * Bc, gC = gU;
      gr[2 * i1] += gB - gC * y2;  gr[2 * i1 + 1] += -gA + gC * x2;
      gr[2 * i2] += -gB + gC * y1; gr[2 * i2 + 1] += gA - gC * x1;
    } else {
      const int i = which - 3;
      gr[2 * i] = gd2 * 2.0f * (vx[i] - PX);
      gr[2 * i + 1] = gd2 * 2.0f * (vy[i] - PY);
    }
    float* o = gface + 6 * ((size_t)b * rp.F + f);
#pragma unroll
    for (int c = 0; c < 6; ++c) if (gr[c] != 0.f) atomicAdd(o + c, gr[c]);
  }
}

// Per face: chain the 6 screen-space gradients through  s = mult * xy,  xy = cam.xy*proj.xy/(cam.z*proj.z),
// cam = rot (v - pos)  and scatter into the vertex gradients.
__global__ void sil_face_to_vertex_kernel(const float* __restrict__ gface, const int* __restrict__ faces,
                                          const float* __restrict__ cam, const float* __restrict__ rot,
                                          float px, float py, float pz, float mult,
                                          float* __restrict__ gverts, int V, int F) {
  const int b = blockIdx.y;
  int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const float* g = gface + 6 * ((size_t)b * F + f);
  const float* r = rot + 9 * (size_t)b;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float gx = g[2 * k] * mult, gy = g[2 * k + 1] * mult;
    if (gx == 0.f && gy == 0.f) continue;
    int vi = faces[3 * f + k];
    const float* c = cam + 3 * ((size_t)b * V + vi);
    float zz = c[2] * pz;
    float x = c[0] * px / zz, y = c[1] * py / zz;
    float gcx = gx * px / zz, gcy = gy * py / zz;
    float gcz = -(gx * x + gy * y) / c[2];
    float* o = gverts + 3 * ((size_t)b * V + vi);
    atomicAdd(o + 0, r[0] * gcx + r[3] * gcy + r[6] * gcz);
    atomicAdd(o + 1, r[1] * gcx + r[4] * gcy + r[7] * gcz);
    atomicAdd(o + 2, r[2] * gcx + r[5] * gcy + r[8] * gcz);
  }
}

static size_t al256s(size_t x) { return (x + 255) & ~(size_t)255; }
struct SilWs { size_t cam, xy, rec, gface, box, total; };
static SilWs sil_layout(int B, int V, int F) {
  SilWs w; size_t o = 0;
  w.cam = o; o += al256s((size_t)B * V * 3 * 4);
  w.xy = o; o += al256s((size_t)B * V * 2 * 4);
  w.rec = o; o += al256s((size_t)B * F * sizeof(FaceRec));
  w.gface = o; o += al256s((size_t)B * F * 6 * 4);
  w.box = o; o += al256s((size_t)B * ((F + kRThreads - 1) / kRThreads) * 8 * sizeof(float4));
  w.total = o;
  return w;
}

}  // namespace vpn

using namespace vpn;

extern "C" int vpn_silhouette_workspace_bytes(int B, int V, int F, size_t* bytes) {
  if (B < 0 || V <= 0 || F <= 0 || !bytes) { vpn_set_error("silhouette workspace: bad arguments"); return VPN_ERR_ARG; }
  *bytes = sil_layout(B, V, F).total;
  return VPN_OK;
}

static int sil_check(int B, int V, int F, int H, int W, int knum) {
  if (B < 0 || V <= 0 || F <= 0 || H <= 0 || W <= 0) { vpn_set_error("silhouette: bad shape"); return VPN_ERR_SHAPE; }
  if (B > 65535) { vpn_set_error("silhouette: batch > 65535 unsupported"); return VPN_ERR_SHAPE; }
  if (knum < 1 || knum > kKnumMax) { vpn_set_error("silhouette: knum must be in [1, %d]", kKnumMax); return VPN_ERR_ARG; }
  if (F > 65535) { vpn_set_error("silhouette: more than 65535 faces per mesh unsupported (16-bit candidate lists)"); return VPN_ERR_SHAPE; }
  return VPN_OK;
}

// verts (B,V,3); faces (F,3) int32 shared by all samples; cam_rot (B,3,3); cam_pos (B,3); proj (px,py,pz).
// Outputs: alpha (B,H,W), covered (B,H,W) u8 (1 where a front face covers the pixel centre),
// normals (B,F,3) or NULL.  The workspace keeps the projected state for the backward call.
extern "C" int vpn_silhouette_fwd(const float* verts, const int* faces, const float* cam_rot, const float* cam_pos,
                                  float proj_x, float proj_y, float proj_z, float expand, int knum, float multiplier,
                                  float delta, int soft_cull_backfaces, float* alpha, unsigned char* covered, float* normals,
                                  void* workspace, size_t workspace_bytes, int B, int V, int F, int H, int W, void* stream) {
  int rc = sil_check(B, V, F, H, W, knum);
  if (rc) return rc;
  if (B == 0) return VPN_OK;
  if (!verts || !faces || !cam_rot || !cam_pos || !alpha || !covered || !workspace) { vpn_set_error("silhouette fwd: null pointer"); return VPN_ERR_ARG; }
  SilWs wl = sil_layout(B, V, F);
  if (workspace_bytes < wl.total) { vpn_set_error("silhouette fwd: workspace too small"); return VPN_ERR_WORKSPACE; }
  char* ws = reinterpret_cast<char*>(workspace);
  float* cam = reinterpret_cast<float*>(ws + wl.cam);
  float* xy = reinterpret_cast<float*>(ws + wl.xy);
  FaceRec* rec = reinterpret_cast<FaceRec*>(ws + wl.rec);
  cudaStream_t s = (cudaStream_t)stream;
  sil_project_kernel<<<dim3((V + 255) / 256, B), 256, 0, s>>>(verts, cam_rot, cam_pos, proj_x, proj_y, proj_z, cam, xy, V);
  if ((rc = vpn_check_launch("sil_project_kernel"))) return rc;
  float4* boxes = reinterpret_cast<float4*>(ws + wl.box);
  sil_faces_kernel<<<dim3((F + kRThreads - 1) / kRThreads, B), kRThreads, 0, s>>>(cam, xy, faces, rec, normals, boxes, V, F, multiplier,
                                                                                  expand * multiplier, soft_cull_backfaces ? 1 : 0);
  if ((rc = vpn_check_launch("sil_faces_kernel"))) return rc;
  RasterParams rp{H, W, F, knum, expand, multiplier, delta, 1e-15f, soft_cull_backfaces ? 1 : 0};
  dim3 grid((W + kTile - 1) / kTile, (H + kTile - 1) / kTile, B);
  static DeviceOnce once_fwd;
  if (set_dyn_smem(sil_raster_fwd_kernel, (int)tile_list_bytes_fwd(kKnumMax), once_fwd) != cudaSuccess) {
    vpn_set_error("silhouette fwd: smem attribute"); return VPN_ERR_CUDA;
  }
  sil_raster_fwd_kernel<<<grid, kRThreads, tile_list_bytes_fwd(knum), s>>>(rec, boxes, alpha, covered, rp);
  return vpn_check_launch("sil_raster_fwd_kernel");
}

// Needs the workspace exactly as vpn_silhouette_fwd left it.  grad_verts (B,V,3) is overwritten.
extern "C" int vpn_silhouette_bwd(const int* faces, const float* cam_rot, float proj_x, float proj_y, float proj_z,
                                  float expand, int knum, float multiplier, float delta, int soft_cull_backfaces,
                                  const float* grad_alpha,
                                  const unsigned char* covered, float* grad_verts, void* workspace, size_t workspace_bytes,
                                  int B, int V, int F, int H, int W, void* stream) {
  int rc = sil_check(B, V, F, H, W, knum);
  if (rc) return rc;
  if (B == 0) return VPN_OK;
  if (!faces || !cam_rot || !grad_alpha || !covered || !grad_verts || !workspace) { vpn_set_error("silhouette bwd: null pointer"); return VPN_ERR_ARG; }
  SilWs wl = sil_layout(B, V, F);
  if (workspace_bytes < wl.total) { vpn_set_error("silhouette bwd: workspace too small"); return VPN_ERR_WORKSPACE; }
  char* ws = reinterpret_cast<char*>(workspace);
  float* cam = reinterpret_cast<float*>(ws + wl.cam);
  FaceRec* rec = reinterpret_cast<FaceRec*>(ws + wl.rec);
  float* gface = reinterpret_cast<float*>(ws + wl.gface);
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(gface, 0, (size_t)B * F * 6 * 4, s) != cudaSuccess ||
      cudaMemsetAsync(grad_verts, 0, (size_t)B * V * 3 * 4, s) != cudaSuccess) {
    vpn_set_error("silhouette bwd: memset failed"); return VPN_ERR_CUDA;
  }
  RasterParams rp{H, W, F, knum, expand, multiplier, delta, 1e-15f, soft_cull_backfaces ? 1 : 0};
  dim3 grid((W + kTile - 1) / kTile, (H + kTile - 1) / kTile, B);
  static DeviceOnce once_bwd;
  if (set_dyn_smem(sil_raster_bwd_kernel, (int)tile_list_bytes_bwd(kKnumMax), once_bwd) != cudaSuccess) {
    vpn_set_error("silhouette bwd: smem attribute"); return VPN_ERR_CUDA;
  }
  sil_raster_bwd_kernel<<<grid, kRThreads, tile_list_bytes_bwd(knum), s>>>(rec, reinterpret_cast<const float4*>(ws + wl.box), grad_alpha, covered, gface, rp);
  if ((rc = vpn_check_launch("sil_raster_bwd_kernel"))) return rc;
  sil_face_to_vertex_kernel<<<dim3((F + 255) / 256, B), 256, 0, s>>>(gface, faces, cam, cam_rot, proj_x, proj_y, proj_z,
                                                                      multiplier, grad_verts, V, F);
  return vpn_check_launch("sil_face_to_vertex_kernel");
}
