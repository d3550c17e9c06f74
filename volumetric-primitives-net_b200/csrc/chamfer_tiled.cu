// Chamfer nearest-neighbour search, tiled FP32 path for sm_100a.
//
// One pass over the (P x M) distance matrix serves BOTH directions of
// modules/loss/chamfer_distance.py:14-23 (row minima over the targets, column minima over the
// predicted points), with O(P + M) memory instead of the reference's dense (B,P,M,3) temporary.
//
// Structure
//   main kernel   : CTA = 256 threads; each thread owns R rows of cloud 1 held as packed f32x2
//                   register pairs (FADD2/FMUL2/FFMA2: two pairs per issue slot); the columns of cloud 2
//                   are staged through shared memory in chunks of kCW and broadcast to all lanes.
//                   The hot loop is branch free and only tracks VALUES: per-row running minima
//                   (FMNMX3) and per-column warp minima (FMNMX3 + CREDUX.MIN.F32).  At the end of each
//                   chunk they are folded into a tiny candidate record: best value + bit mask of the
//                   chunks (rows) / warps (columns) that can still hold the arg-min.
//   recovery      : warp-cooperative kernels re-evaluate only the candidate chunks with the
//                   reference's exact arithmetic and pick (min sqrt(d), first index) - torch.min's
//                   tie rule - so min and arg-min are bit-exact whatever arithmetic the hot loop used.
//
// Arithmetic modes of the hot loop (recovery is always exact):
//   MODE_EXACT  : d = fl(fl(fl(dx*dx)+fl(dy*dy))+fl(dz*dz)), the reference's own rounding sequence
//                 (8 pipe ops per pair).  Candidate slack: the sqrt rounding class only (2^-20 relative).
//   MODE_DIFF   : same differences, FMA-accumulated squares (6 pipe ops per pair).  Differs from the
//                 reference by <= ~7 ulp; slack 2^-18 relative.
//   MODE_EXPAND : |p-t|^2 = |p|^2 + |t|^2 - 2 p.t on coordinates centred on the tile's centroid
//                 (4 pipe ops per pair: 3 FFMA2 + 1 FADD2 per two pairs).  With rho = tile radius the
//                 error vs the reference is <= max(384 u rho^2, 96 u d) (u = 2^-24; derivation in
//                 DESIGN.md), absorbed by the slack 2.5 * 2^-15 rho^2 + 2^-15 |x|.  Inputs whose centred
//                 magnitudes overflow the analysis raise a per-sample flag and that sample is redone
//                 by a MODE_DIFF launch (all other CTAs of that launch exit immediately).
//
// NOTE on ptxas: mul.rn.f32x2 followed by add.rn.f32x2 IS contracted into FFMA2 by ptxas 12.9 even
// with --fmad=false (the scalar .rn forms are not).  The exact mode therefore performs its two
// additions as fma(x, 1.0, y) with the 1.0 passed as a kernel argument, which rounds exactly like
// an add and cannot be contracted.
#include <cstdlib>
#include <mutex>
#include <type_traits>
#include "common.cuh"

namespace vpn {

enum { MODE_EXACT = 0, MODE_DIFF = 1, MODE_EXPAND = 2, MODE_TC = 3 };

constexpr int kTThreads = 256;
constexpr int kTWarps = kTThreads / 32;
constexpr int kCW = 128;                  // columns per chunk (candidate granularity for rows)
constexpr int kMaxChunksPerSplit = 64;    // bits in the row candidate mask
constexpr float kBig = 1.0e30f;           // centred magnitudes^2 above this fall back to MODE_DIFF

__device__ __forceinline__ u64 pk(float a, float b) { u64 r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk(u64 v, float& a, float& b) { asm("mov.b64 {%0,%1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ float min3f(float a, float b, float c) { float r; asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }
__device__ __forceinline__ float warp_min_f32(float a) { float r; asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(a)); return r; }
__device__ __forceinline__ float inf_f() { return __int_as_float(0x7f800000); }

// Upper bound of the hot-loop values that may still belong to the arg-min when the smallest hot-loop
// value seen is x: x + rel |x| + abs, rounded up.
__device__ __forceinline__ float thr_of(float x, float rel, float abs_) {
  return __fadd_ru(__fmaf_ru(fabsf(x), rel, x), abs_);
}
__device__ __forceinline__ float mode_rel(int mode) {
  return mode == MODE_EXACT ? 9.5367431640625e-07f /* 2^-20 */
       : mode == MODE_DIFF ? 3.814697265625e-06f   /* 2^-18 */
                           : 3.0517578125e-05f;     /* 2^-15 */
}

__device__ __forceinline__ float exact_d2s(float ax, float ay, float az, float bx, float by, float bz) {
  float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

template <int R>
struct TiledSmem {
  float4 tile[2][kCW];
  float colw[2][kTWarps][kCW];
  float rs_best[R][kTThreads];
  float rs_thr[R][kTThreads];
  u64 rs_mask[R][kTThreads];
  float red[kTWarps][4];
  float ctr[4];
};

// Row constants held per packed row pair.
//   EXACT / DIFF : c0,c1,c2 = (px,py,pz)
//   EXPAND       : c0,c1,c2 = -2 (px,py,pz) centred, c3 = |p|^2 centred
template <int MODE>
__device__ __forceinline__ u64 pair_val(u64 c0, u64 c1, u64 c2, u64 c3, const float4& col, float one) {
  if (MODE == MODE_EXPAND) {
    u64 e = fma2(c0, pk(col.x, col.x), c3);
    e = fma2(c1, pk(col.y, col.y), e);
    e = fma2(c2, pk(col.z, col.z), e);
    return add2(e, pk(col.w, col.w));
  }
  u64 dx = sub2(c0, pk(col.x, col.x)), dy = sub2(c1, pk(col.y, col.y)), dz = sub2(c2, pk(col.z, col.z));
  if (MODE == MODE_EXACT) {
    u64 xx = mul2(dx, dx), yy = mul2(dy, dy), zz = mul2(dz, dz);
    u64 o2 = pk(one, one);
    return fma2(fma2(xx, o2, yy), o2, zz);          // fl(fl(xx + yy) + zz), never contracted
  }
  return fma2(dz, dz, fma2(dy, dy, mul2(dx, dx)));
}

// grid: x = row tile, y = column split, z = sample
template <int R, int MODE>
__global__ void __launch_bounds__(kTThreads, (R <= 8 ? 2 : 1))
chamfer_tiled_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                     float* __restrict__ rbest, u64* __restrict__ rmask,
                     float* __restrict__ cbest, unsigned* __restrict__ cmask,
                     float2* __restrict__ tslack, int* __restrict__ fallback,
                     int P, int M, int nchunks, int cps, float one, int only_flagged) {
  constexpr int TM = kTThreads * R;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TiledSmem<R>& sm = *reinterpret_cast<TiledSmem<R>*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tile_i = blockIdx.x, split = blockIdx.y, b = blockIdx.z;
  const int ntiles = gridDim.x, nsplit = gridDim.y;
  if (only_flagged && fallback[b] == 0) return;
  const float* A = p1 + (size_t)b * P * 3;
  const float* T = p2 + (size_t)b * M * 3;

  u64 c0[R / 2], c1[R / 2], c2[R / 2], c3[R / 2];
  float rm[R];
  float cx = 0.f, cy = 0.f, cz = 0.f;
  float slack_rel = mode_rel(MODE), slack_abs = 1e-36f;
  {
    float x[R], y[R], z[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      int i = min(tile_i * TM + r * kTThreads + tid, P - 1);
      x[r] = A[3 * (size_t)i]; y[r] = A[3 * (size_t)i + 1]; z[r] = A[3 * (size_t)i + 2];
    }
    if (MODE == MODE_EXPAND) {
      // tile centroid (any centre is valid; the centroid keeps the radius, hence the slack, small)
      float sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
      for (int r = 0; r < R; ++r) { sx += x[r]; sy += y[r]; sz += z[r]; }
      sx = warp_sum(sx); sy = warp_sum(sy); sz = warp_sum(sz);
      if (lane == 0) { sm.red[warp][0] = sx; sm.red[warp][1] = sy; sm.red[warp][2] = sz; }
      __syncthreads();
      if (tid < 3) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kTWarps; ++w) s += sm.red[w][tid];
        sm.ctr[tid] = s / (float)TM;
      }
      __syncthreads();
      cx = sm.ctr[0]; cy = sm.ctr[1]; cz = sm.ctr[2];
      float rho2 = 0.f;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        x[r] = __fsub_rn(x[r], cx); y[r] = __fsub_rn(y[r], cy); z[r] = __fsub_rn(z[r], cz);
        rho2 = fmaxf(rho2, fmaf(z[r], z[r], fmaf(y[r], y[r], x[r] * x[r])));
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rho2 = fmaxf(rho2, __shfl_xor_sync(0xffffffffu, rho2, o));
      __syncthreads();
      if (lane == 0) sm.red[warp][3] = rho2;
      __syncthreads();
      rho2 = sm.red[0][3];
#pragma unroll
      for (int w = 1; w < kTWarps; ++w) rho2 = fmaxf(rho2, sm.red[w][3]);
      if (!(rho2 < kBig)) { if (tid == 0) atomicOr(&fallback[b], 1); rho2 = 0.f; }
      slack_abs = __fmaf_ru(8.0e-5f, rho2, 1e-36f);          // 2.5 * 2^-15 rho^2 (+ margin), see header
    }
#pragma unroll
    for (int rp = 0; rp < R / 2; ++rp) {
      const int r0 = 2 * rp, r1 = 2 * rp + 1;
      if (MODE == MODE_EXPAND) {
        c0[rp] = pk(-2.f * x[r0], -2.f * x[r1]); c1[rp] = pk(-2.f * y[r0], -2.f * y[r1]); c2[rp] = pk(-2.f * z[r0], -2.f * z[r1]);
        c3[rp] = pk(fmaf(z[r0], z[r0], fmaf(y[r0], y[r0], x[r0] * x[r0])), fmaf(z[r1], z[r1], fmaf(y[r1], y[r1], x[r1] * x[r1])));
      } else {
        c0[rp] = pk(x[r0], x[r1]); c1[rp] = pk(y[r0], y[r1]); c2[rp] = pk(z[r0], z[r1]); c3[rp] = 0ull;
      }
    }
  }
  if (tid == 0 && split == 0) tslack[(size_t)b * ntiles + tile_i] = make_float2(slack_rel, slack_abs);
#pragma unroll
  for (int r = 0; r < R; ++r) {
    rm[r] = inf_f();
    sm.rs_best[r][tid] = inf_f(); sm.rs_thr[r][tid] = inf_f(); sm.rs_mask[r][tid] = 0ull;
  }
  const int c_first = split * cps;
  const int c_last = min(nchunks, c_first + cps);

  auto make_col = [&](float tx, float ty, float tz) -> float4 {
    if (MODE == MODE_EXPAND) {
      float x = __fsub_rn(tx, cx), y = __fsub_rn(ty, cy), z = __fsub_rn(tz, cz);
      float c = fmaf(z, z, fmaf(y, y, x * x));
      if (!(c < kBig)) atomicOr(&fallback[b], 1);
      return make_float4(x, y, z, c);
    }
    return make_float4(tx, ty, tz, 0.f);
  };

  if (tid < kCW) {
    int col = min(c_first * kCW + tid, M - 1);
    sm.tile[0][tid] = make_col(T[3 * (size_t)col], T[3 * (size_t)col + 1], T[3 * (size_t)col + 2]);
  }
  __syncthreads();

  for (int c = c_first; c < c_last; ++c) {
    const int buf = (c - c_first) & 1;
    // prefetch the next chunk into registers while this one is being consumed
    float nx = 0.f, ny = 0.f, nz = 0.f;
    const bool has_next = (c + 1 < c_last) && (tid < kCW);
    if (has_next) {
      int col = min((c + 1) * kCW + tid, M - 1);
      nx = T[3 * (size_t)col]; ny = T[3 * (size_t)col + 1]; nz = T[3 * (size_t)col + 2];
    }
    const float4* tl = sm.tile[buf];
    float* cw = sm.colw[buf][warp];
#pragma unroll 2
    for (int k = 0; k < kCW; k += 2) {
      const float4 q0 = tl[k], q1 = tl[k + 1];
      float cm0 = inf_f(), cm1 = inf_f();
#pragma unroll
      for (int rp = 0; rp < R / 2; ++rp) {
        u64 d0 = pair_val<MODE>(c0[rp], c1[rp], c2[rp], c3[rp], q0, one);
        u64 d1 = pair_val<MODE>(c0[rp], c1[rp], c2[rp], c3[rp], q1, one);
        float a0, b0, a1, b1;
        upk(d0, a0, b0); upk(d1, a1, b1);
        rm[2 * rp] = min3f(rm[2 * rp], a0, a1);
        rm[2 * rp + 1] = min3f(rm[2 * rp + 1], b0, b1);
        cm0 = min3f(cm0, a0, b0);
        cm1 = min3f(cm1, a1, b1);
      }
      float w0 = warp_min_f32(cm0), w1 = warp_min_f32(cm1);
      if (lane == 0) *reinterpret_cast<float2*>(cw + k) = make_float2(w0, w1);
    }
    // fold this chunk's row minima into the per-row candidate record
    const u64 bit = 1ull << (c - c_first);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float m = rm[r];
      rm[r] = inf_f();
      if (m <= sm.rs_thr[r][tid]) {
        const float best = sm.rs_best[r][tid];
        const float tm = thr_of(m, slack_rel, slack_abs);
        u64 mask = (tm < best) ? 0ull : sm.rs_mask[r][tid];
        sm.rs_mask[r][tid] = mask | bit;
        if (m < best) { sm.rs_best[r][tid] = m; sm.rs_thr[r][tid] = tm; }
      }
    }
    if (has_next) sm.tile[buf ^ 1][tid] = make_col(nx, ny, nz);
    __syncthreads();
    // per-column candidate record of this tile: best warp minimum + mask of warps within slack
    if (tid < kCW) {
      const int col = c * kCW + tid;
      if (col < M) {
        float w[kTWarps];
        float best = inf_f();
#pragma unroll
        for (int i = 0; i < kTWarps; ++i) { w[i] = sm.colw[buf][i][tid]; best = fminf(best, w[i]); }
        const float t = thr_of(best, slack_rel, slack_abs);
        unsigned mask = 0;
#pragma unroll
        for (int i = 0; i < kTWarps; ++i) mask |= (w[i] <= t) ? (1u << i) : 0u;
        size_t o = ((size_t)b * ntiles + tile_i) * M + col;
        cbest[o] = best; cmask[o] = mask;
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    int row = tile_i * TM + r * kTThreads + tid;
    if (row < P) {
      size_t o = ((size_t)b * nsplit + split) * P + row;
      rbest[o] = sm.rs_best[r][tid]; rmask[o] = sm.rs_mask[r][tid];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// recovery: exact (min sqrt(d), first index) over the candidate chunks only.
// Work items (row, column chunk) / (column, warp block) are compacted per CTA and split into sub-units so
// that all threads stay busy; the scanned cloud (the sample's targets, or the tile's rows) sits in shared
// memory and every lane walks it with a lane-rotated start, which makes the float4 reads conflict free.
// Results are merged with a 64-bit atomicMin on (float_bits(v) << 32 | index): value, then lowest index.
// ---------------------------------------------------------------------------------------------
constexpr int kRecThreads = 1024;
constexpr int kSegChunks = 64;                       // column chunks resident in shared memory per segment
constexpr int kItemCap = 4096;                      // work items per round: (row, 32-column unit) / (column, row block)

struct ExactBest {
  float d, hi, v; int i;
  __device__ __forceinline__ void init() { d = inf_f(); hi = inf_f(); v = inf_f(); i = 0x7fffffff; }
  // dd = exact squared distance (NaN for padding: never accepted).  Any visiting order is allowed.
  __device__ __forceinline__ void offer(float dd, int idx) {
    if (dd <= hi) {
      float vv = sqrtf(dd);
      if (vv < v || (vv == v && idx < i)) { v = vv; i = idx; }
      if (dd < d) { d = dd; hi = thr_of(dd, 9.5367431640625e-07f, 1e-36f); }   // covers dd's sqrt rounding class
    }
  }
  __device__ __forceinline__ u64 key() const { return ((u64)__float_as_uint(v) << 32) | (unsigned)i; }
};

// Scan of 32 squared distances held in registers (d[kk] belongs to position (kk + rot) & 31 of the unit).
// Phase 1 found dm = min d.  One more pass counts the values within dm's sqrt rounding class and sums their
// positions (two predicated integer adds per value).  Returns 1 with *at = the winner's position when the count is 1
// (v = sqrt(dm), no index bookkeeping per value), 2 when several values share the class (ties / near ties, rare: the
// caller takes the out-of-line exact walk), 0 when the unit holds no valid point.
__device__ __forceinline__ int unit_scan(const float (&d)[32], float dm, int rot, int* at) {
  if (!(dm < inf_f())) {                       // all padding, or genuinely infinite distances
    bool any = false;
#pragma unroll
    for (int kk = 0; kk < 32; ++kk) any |= (d[kk] == inf_f());
    if (!any) return 0;
    return 2;
  }
  const float hi = thr_of(dm, 9.5367431640625e-07f, 1e-36f);
  int cnt = 0, pos = 0;
#pragma unroll
  for (int kk = 0; kk < 32; ++kk) {
    const bool in = d[kk] <= hi;               // NaN padding compares false
    cnt += in ? 1 : 0;
    pos += in ? kk : 0;
  }
  *at = (pos + rot) & 31;
  return cnt == 1 ? 1 : 2;
}

// Out-of-line exact walk over a unit's 32 points (rare path: kept out of the scan's register budget).  pts: the 32
// staged points; index of point k = w-component as int bits (use_w: original index of a permuted cloud) or idx0 + k.
__device__ __noinline__ u64 unit_exact_walk(float ax, float ay, float az, const float4* __restrict__ pts, int idx0, int use_w) {
  ExactBest eb; eb.init();
  for (int k = 0; k < 32; ++k) {
    const float4 q = pts[k];
    eb.offer(exact_d2s(ax, ay, az, q.x, q.y, q.z), use_w ? __float_as_int(q.w) : idx0 + k);
  }
  return eb.i != 0x7fffffff ? eb.key() : ~0ull;
}

// exclusive prefix sum of `cnt` over the CTA (NT threads, NT / 32 <= 32 warps); returns the offset, *total gets the sum
template <int NT>
__device__ __forceinline__ int block_exclusive_scan(int cnt, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = lane < NT / 32 ? warp_sums[lane] : 0;
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += t; }
    warp_sums[lane] = winc - w;
    if (lane == 31) warp_sums[32] = winc;
  }
  __syncthreads();
  int off = warp_sums[warp] + inc - cnt;
  *total = warp_sums[32];
  __syncthreads();
  return off;
}

// 16 chunk bits -> 64 unit bits (bit k -> bits 4k..4k+3): a chunk-granular record names all four units of the chunk
__device__ __forceinline__ u64 expand_chunk_bits16(unsigned v) {
  u64 x = v & 0xffffu;
  x = (x | (x << 24)) & 0x000000ff000000ffull;
  x = (x | (x << 12)) & 0x000f000f000f000full;
  x = (x | (x << 6)) & 0x0303030303030303ull;
  x = (x | (x << 3)) & 0x1111111111111111ull;
  return x * 0xfull;
}
// seg |= w << base over a 256-bit mask held in four words (base may be negative or past the end)
__device__ __forceinline__ void or_shifted256(u64 (&seg)[4], u64 w, int base) {
  if (w == 0ull || base >= 256 || base <= -64) return;
  const int k = base >> 6, sh = base & 63;                     // floor division: base = 64 k + sh
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    if (kk == k) seg[kk] |= w << sh;
    if (sh != 0 && kk == k + 1) seg[kk] |= w >> (64 - sh);
  }
}

// exclusive prefix sum of `cnt` over one half of the CTA (kRowGroup threads, named barrier `bar`); *total gets the sum
constexpr int kRowGroup = kRecThreads / 2;            // the CTA works as two independent groups of 512 threads
constexpr int kRowItemCap = kItemCap / 2;
constexpr size_t kRowsFixedSmem = (size_t)kRecThreads * (16 + 8 + 32 + 4 + 12 + 4) + (size_t)kItemCap * 4;    // row recovery: everything but the targets
__device__ __forceinline__ void group_sync(int bar) { asm volatile("bar.sync %0, %1;" :: "r"(bar), "n"(kRowGroup) : "memory"); }
__device__ __forceinline__ int group_exclusive_scan(int cnt, int* warp_sums, int* total, int gt, int bar) {
  const int lane = gt & 31, warp = gt >> 5;                           // 16 warps
  int inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) warp_sums[warp] = inc;
  group_sync(bar);
  if (warp == 0) {
    int w = lane < kRowGroup / 32 ? warp_sums[lane] : 0;
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += t; }
    if (lane < kRowGroup / 32) warp_sums[lane] = winc - w;
    if (lane == 31) warp_sums[kRowGroup / 32] = winc;
  }
  group_sync(bar);
  int off = warp_sums[warp] + inc - cnt;
  *total = warp_sums[kRowGroup / 32];
  group_sync(bar);
  return off;
}

// Persistent: grid x = min(#SMs, B * nblk) CTAs; CTA k takes the work items (sample, block of kRowGroup rows)
// [k per, (k + 1) per) - consecutive items belong to the same sample, whose targets are staged in shared memory ONCE
// (one CTA per item re-staged 131 KB per 1024 rows: a fifth of the kernel).  The two halves of the CTA take alternate
// items and meet only when the staged targets change: while one half waits for its rows' records (a DRAM round trip per
// item, nothing else to run on an SM that holds a single CTA) the other evaluates units.  dynamic smem: kRowsFixedSmem
// bytes + float4 cols[min(nchunks,64)*128].  Clouds of more than 64 chunks are swept in segments; the running best of a row then
// passes from one segment to the next through min1 / idx1.
// Candidate records: planes == 4: four u64 planes (plane_stride apart) of 32-column UNIT bits (tensor-core filter),
// planes == 1: one u64 of 128-column chunk bits (CUDA-core filters), expanded to unit bits here.
// p2v != NULL: the targets as float4 (x, y, z, original index) padded with NaN to whole chunks (stride mpad per sample).
__global__ void __launch_bounds__(kRecThreads, 1)
chamfer_recover_rows_kernel(const float* __restrict__ p1, const float* __restrict__ p2, const float4* __restrict__ p2v, int mpad,
                            const float* __restrict__ rbest, const u64* __restrict__ rmask, int planes, size_t plane_stride,
                            const float2* __restrict__ tslack, float* __restrict__ min1, int* __restrict__ idx1,
                            int P, int M, int nchunks, int nsplit, int cps, int TM, int ntiles,
                            const int* __restrict__ skip, int nblk, int nitems, const int* __restrict__ rperm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // dynamic shared memory: [rowc | key | pre_mask | items | pre_rb | pre_p1 | pre_perm] (kRowsFixedSmem bytes) then cols[]
  float4* rowc_ = reinterpret_cast<float4*>(smem_raw);
  u64* key_ = reinterpret_cast<u64*>(rowc_ + kRecThreads);
  u64 (*pre_mask)[kRecThreads] = reinterpret_cast<u64 (*)[kRecThreads]>(key_ + kRecThreads);
  unsigned* items_ = reinterpret_cast<unsigned*>(pre_mask + 4);
  float* pre_rb = reinterpret_cast<float*>(items_ + kItemCap);
  float* pre_p1 = pre_rb + kRecThreads;
  int* pre_perm = reinterpret_cast<int*>(pre_p1 + 3 * kRecThreads);
  float4* cols = reinterpret_cast<float4*>(smem_raw + kRowsFixedSmem);
  __shared__ int warp_sums_[2][kRowGroup / 32 + 1];
  // records of the group's NEXT item, fetched with cp.async while the current item's units are evaluated (one record per
  // row, i.e. nsplit == 1; a thread only ever touches its own slots, so no barrier is involved)
  const int tid = threadIdx.x, lane = tid & 31, grp = tid / kRowGroup, gt = tid % kRowGroup, bar = 1 + grp;
  const bool use_pre = (nsplit == 1) && (planes == 4);
  auto prefetch = [&](int b_, int wi_) {
    const int row_ = (wi_ - b_ * nblk) * kRowGroup + gt;
    if (row_ < P) {
      const size_t o_ = (size_t)b_ * P + row_;
      cp_async4(&pre_rb[tid], rbest + o_);
#pragma unroll
      for (int w = 0; w < 4; ++w) cp_async8(&pre_mask[w][tid], rmask + o_ + w * plane_stride);
#pragma unroll
      for (int k = 0; k < 3; ++k) cp_async4(&pre_p1[tid * 3 + k], p1 + 3 * o_ + k);
      if (rperm) cp_async4(&pre_perm[tid], rperm + o_);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  float4* rowc = rowc_ + grp * kRowGroup; u64* key = key_ + grp * kRowGroup;
  unsigned* items = items_ + grp * kRowItemCap; int* warp_sums = warp_sums_[grp];
  const int per = (nitems + gridDim.x - 1) / gridDim.x;
  const int w0 = blockIdx.x * per, w1 = min(nitems, w0 + per);
  const int nseg = (nchunks + kSegChunks - 1) / kSegChunks;
  const float qnan = __int_as_float(0x7fc00000);
  for (int b = w0 / nblk; b * nblk < w1; ++b) {
    if (skip && skip[b]) continue;                       // sample redone by chamfer_flagged_kernel
    const int i0 = max(w0, b * nblk), i1 = min(w1, (b + 1) * nblk);      // this CTA's items of sample b
    for (int seg = 0; seg < nseg; ++seg) {
      const int seg_chunks = min(kSegChunks, nchunks - seg * kSegChunks);
      __syncthreads();                                   // both groups are done with the previous contents
      if (p2v) {
        const float4* src = p2v + (size_t)b * mpad + (size_t)seg * kSegChunks * kCW;
        for (int i = tid; i < seg_chunks * kCW; i += kRecThreads) cols[i] = src[i];
      } else {
        const float* T = p2 + (size_t)b * M * 3;
        for (int i = tid; i < seg_chunks * kCW; i += kRecThreads) {
          const int col = seg * kSegChunks * kCW + i;
          cols[i] = col < M ? make_float4(T[3 * (size_t)col], T[3 * (size_t)col + 1], T[3 * (size_t)col + 2], __int_as_float(col))
                            : make_float4(qnan, qnan, qnan, __int_as_float(0x7fffffff));
        }
      }
      __syncthreads();
      if (use_pre && i0 + grp < i1) prefetch(b, i0 + grp);
      for (int wi = i0 + grp; wi < i1; wi += 2) {
        const int row = (wi - b * nblk) * kRowGroup + gt;
        const bool valid = row < P;
        // p1 is the spatially sorted copy when rperm != NULL: the results go to the row's original position (looked up where
        // it is needed: kept live across the item it costs two registers the kernel does not have)
        // (prefetched with the records and parked in the unused .w of the row's staged coordinates: loaded just before the
        // final stores it was 6 % of the kernel's stalls)
        auto orow_of = [&]() { return (size_t)b * P + (use_pre ? __float_as_int(rowc[gt].w) : (rperm ? rperm[(size_t)b * P + row] : row)); };
        float g = inf_f(), gthr = inf_f();
        u64 kinit = ~0ull;
        // this row's candidate units of the segment: 256 bits, unit u of the segment = columns [32 u, 32 u + 32) of cols[]
        u64 sg[4] = {0ull, 0ull, 0ull, 0ull};
        if (use_pre) {
          asm volatile("cp.async.wait_all;" ::: "memory");
          if (valid) {
            rowc[gt] = make_float4(pre_p1[tid * 3], pre_p1[tid * 3 + 1], pre_p1[tid * 3 + 2], __int_as_float(rperm ? pre_perm[tid] : row));
            g = pre_rb[tid];
            if (seg > 0) { const size_t orow = orow_of(); kinit = ((u64)__float_as_uint(min1[orow]) << 32) | (unsigned)idx1[orow]; }
            const int rel = -seg * kSegChunks * 4;                               // first unit of the record, relative to the segment
            if (rel == 0) {
#pragma unroll
              for (int w = 0; w < 4; ++w) sg[w] = pre_mask[w][tid];
            } else {
#pragma unroll
              for (int w = 0; w < 4; ++w) or_shifted256(sg, pre_mask[w][tid], rel + 64 * w);
            }
          }
          if (wi + 2 < i1) prefetch(b, wi + 2);            // my slots are free again: the next item's records start moving
          if (valid && seg_chunks < kSegChunks) {                                // units past the end of the cloud
            const int nu = seg_chunks * 4;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              const int left = nu - 64 * w;
              if (left <= 0) sg[w] = 0ull; else if (left < 64) sg[w] &= (1ull << left) - 1ull;
            }
          }
        } else if (valid) {
          const float* a = p1 + 3 * ((size_t)b * P + row);
          rowc[gt] = make_float4(a[0], a[1], a[2], 0.f);
          for (int s = 0; s < nsplit; ++s) g = fminf(g, rbest[((size_t)b * nsplit + s) * P + row]);
          const float2 sl = tslack[(size_t)b * ntiles + row / TM];
          gthr = thr_of(g, sl.x, sl.y);
          if (seg > 0) { const size_t orow = orow_of(); kinit = ((u64)__float_as_uint(min1[orow]) << 32) | (unsigned)idx1[orow]; }
          for (int s = 0; s < nsplit; ++s) {
            const size_t o = ((size_t)b * nsplit + s) * P + row;
            if (!(rbest[o] <= gthr)) continue;
            const int rel = (s * cps - seg * kSegChunks) * 4;                    // first unit of the split, relative to the segment
            if (planes == 4) {
#pragma unroll
              for (int w = 0; w < 4; ++w) or_shifted256(sg, rmask[o + w * plane_stride], rel + 64 * w);
            } else {
              const u64 m = rmask[o];
#pragma unroll
              for (int w = 0; w < 4; ++w) or_shifted256(sg, expand_chunk_bits16((unsigned)(m >> (16 * w))), rel + 64 * w);
            }
          }
          if (seg_chunks < kSegChunks) {                                         // units past the end of the cloud
            const int nu = seg_chunks * 4;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              const int left = nu - 64 * w;
              if (left <= 0) sg[w] = 0ull; else if (left < 64) sg[w] &= (1ull << left) - 1ull;
            }
          }
        }
        key[gt] = kinit;
        int total;
        const int cnt = __popcll(sg[0]) + __popcll(sg[1]) + __popcll(sg[2]) + __popcll(sg[3]);
        const int off = group_exclusive_scan(cnt, warp_sums, &total, gt, bar);   // syncs the group: rowc / key are written
        for (int base = 0; base < total; base += kRowItemCap) {
          int j = off;
#pragma unroll
          for (int w = 0; w < 4; ++w)
            for (u64 mm = sg[w]; mm; mm &= mm - 1, ++j)
              if (j >= base && j < base + kRowItemCap) items[j - base] = ((unsigned)gt << 8) | (unsigned)(64 * w + __ffsll((long long)mm) - 1);
          group_sync(bar);
          const int units = min(kRowItemCap, total - base);
          for (int it = gt; it < units; it += kRowGroup) {
            const unsigned item = items[it];
            const int r = item >> 8, u = item & 255;
            const float4 rc = rowc[r];
            const float4* src = cols + u * 32;
            float d[32], dm = inf_f();
#pragma unroll
            for (int kk = 0; kk < 32; ++kk) {
              const float4 q = src[(kk + lane) & 31];
              d[kk] = exact_d2s(rc.x, rc.y, rc.z, q.x, q.y, q.z);
              dm = fminf(dm, d[kk]);
            }
            int at;
            const int st = unit_scan(d, dm, lane, &at);
            if (st == 1) atomicMin(&key[r], ((u64)__float_as_uint(sqrtf(dm)) << 32) | (unsigned)__float_as_int(src[at].w));
            else if (st == 2) { const u64 kv = unit_exact_walk(rc.x, rc.y, rc.z, src, 0, 1); if (kv != ~0ull) atomicMin(&key[r], kv); }
          }
          group_sync(bar);
        }
        if (valid) {
          const u64 kv = key[gt];
          const size_t orow = orow_of();
          min1[orow] = __uint_as_float((unsigned)(kv >> 32));
          idx1[orow] = (int)(unsigned)(kv & 0xffffffffu);
        }
        group_sync(bar);                                 // the next item overwrites rowc / key
      }
    }
  }
}

// per column: threshold over all tiles' records
__global__ void chamfer_col_thr_kernel(const float* __restrict__ cbest, const float2* __restrict__ tslack,
                                       float* __restrict__ cthr, int M, int ntiles) {
  const int b = blockIdx.y;
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= M) return;
  float g = inf_f(), rel = 0.f, ab = 0.f;
  for (int ti = 0; ti < ntiles; ++ti) {
    g = fminf(g, cbest[((size_t)b * ntiles + ti) * M + col]);
    const float2 sl = tslack[(size_t)b * ntiles + ti];
    rel = fmaxf(rel, sl.x); ab = fmaxf(ab, sl.y);
  }
  cthr[(size_t)b * M + col] = thr_of(g, rel, ab);
}

// grid: x = row tile, y = sample.  dynamic smem: float4 rows[TM].  key2 (B,M) u64 pre-filled with 0xFF.
// Candidate records of a (tile, column):
//   TC == false : `unsigned`, bit k = rows rr * 256 + k * 32 + [0,32), rr = 0..R-1  (warp k of chamfer_tiled_kernel<R>, TM = 256 R)
//   TC == true  : u64, bit k = rows 32 k + [0,32) of the tile                        (32-row UNITS, chamfer_tc_kernel, TM = 128 R)
// NT threads per CTA: 512 for the tensor-core records (two CTAs per SM: the kernel is a chain of short latency-bound phases -
// record loads, scan, a few hundred unit evaluations per tile - and a single 1024-thread CTA per SM left the SM idle
// between them), 1024 otherwise.
template <int R, bool TC, int NT>
__global__ void __launch_bounds__(NT, 1024 / NT)
chamfer_recover_cols_kernel(const float* __restrict__ p1, const float* __restrict__ p2,
                            const float* __restrict__ cbest, const void* __restrict__ cmask_,
                            const float* __restrict__ cthr, u64* __restrict__ key2, int P, int M, int ntiles,
                            const int* __restrict__ skip, const int* __restrict__ rperm) {
  constexpr int TM = TC ? 128 * R : kTThreads * R;
  constexpr int kSub = TC ? 1 : ((R >= 4) ? 4 : R);      // sub-units per (column, bit) item
  constexpr int kRunsPerSub = TC ? 1 : R / kSub;
  constexpr int kPer = TC ? 4096 / NT : 8;               // columns per thread and slab (4096 columns per slab with the tensor-core records)
  constexpr int kBitBits = TC ? 6 : 4;
  using mask_t = typename std::conditional<TC, u64, unsigned>::type;
  const mask_t* __restrict__ cmask = reinterpret_cast<const mask_t*>(cmask_);
  const mask_t kBitMask = TC ? (mask_t)((4 * R >= 64) ? ~0ull : ((1ull << (4 * R)) - 1ull)) : (mask_t)0xffu;
  if (skip && skip[blockIdx.y]) return;                  // sample redone by chamfer_flagged_kernel
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* rows = reinterpret_cast<float4*>(smem_raw);
  __shared__ unsigned items[kItemCap];
  __shared__ int warp_sums[33];
  const int b = blockIdx.y, ti = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  const float* A = p1 + (size_t)b * P * 3;
  const float qnan = __int_as_float(0x7fc00000);
  for (int i = tid; i < TM; i += NT) {
    int rowi = ti * TM + i;
    // w = the row's ORIGINAL index (p1 is the spatially sorted copy when rperm != NULL): ties go to the first original row
    rows[i] = rowi < P ? make_float4(A[3 * (size_t)rowi], A[3 * (size_t)rowi + 1], A[3 * (size_t)rowi + 2],
                                     __int_as_float(rperm ? rperm[(size_t)b * P + rowi] : rowi))
                       : make_float4(qnan, qnan, qnan, __int_as_float(0x7fffffff));
  }
  const size_t rec0 = ((size_t)b * ntiles + ti) * M;
  // columns are visited in slabs of NT * kPer so that one slab's items normally fit the list
  for (int slab = 0; slab < M; slab += NT * kPer) {
    mask_t mk[kPer];
    int cnt = 0;
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int col = slab + u * NT + tid;
      mk[u] = 0;
      if (col < M && cbest[rec0 + col] <= cthr[(size_t)b * M + col]) mk[u] = cmask[rec0 + col] & kBitMask;
      cnt += TC ? __popcll((u64)mk[u]) : __popc((unsigned)mk[u]);
    }
    int total;
    const int off = block_exclusive_scan<NT>(cnt, warp_sums, &total);
    for (int base = 0; base < total; base += kItemCap) {
      int j = off;
#pragma unroll
      for (int u = 0; u < kPer; ++u)
        for (mask_t mm = mk[u]; mm; mm &= mm - 1, ++j)
          if (j >= base && j < base + kItemCap)
            items[j - base] = ((unsigned)(u * NT + tid) << kBitBits) |
                              (unsigned)((TC ? __ffsll((long long)mm) : __ffs((int)mm)) - 1);
      __syncthreads();
      const int units = min(kItemCap, total - base) * kSub;
      for (int it = tid; it < units; it += NT) {
        const unsigned item = items[it / kSub];
        const int col = slab + (int)(item >> kBitBits), w = item & ((1u << kBitBits) - 1u), sub = it % kSub;
        const float* t = p2 + 3 * ((size_t)b * M + col);
        const float tx = __ldg(t), ty = __ldg(t + 1), tz = __ldg(t + 2);
        u64 best = ~0ull;
#pragma unroll 1
        for (int rr = sub * kRunsPerSub; rr < (sub + 1) * kRunsPerSub; ++rr) {
          const int base_row = TC ? (w * 32) : (rr * kTThreads + w * 32);
          float d[32], dm = inf_f();
#pragma unroll
          for (int kk = 0; kk < 32; ++kk) {
            const float4 a = rows[base_row + ((kk + lane) & 31)];
            d[kk] = exact_d2s(a.x, a.y, a.z, tx, ty, tz);
            dm = fminf(dm, d[kk]);
          }
          int at;
          const int st = unit_scan(d, dm, lane, &at);
          u64 kv = ~0ull;
          if (st == 1) kv = ((u64)__float_as_uint(sqrtf(dm)) << 32) | (unsigned)__float_as_int(rows[base_row + at].w);
          else if (st == 2) kv = unit_exact_walk(tx, ty, tz, rows + base_row, 0, 1);
          best = kv < best ? kv : best;
        }
        if (best != ~0ull) atomicMin(&key2[(size_t)b * M + col], best);
      }
      __syncthreads();
    }
  }
}

// perm (optional): key[i] belongs to sorted position i of its sample; the outputs are indexed by the original position
__global__ void chamfer_unpack_key_kernel(const u64* __restrict__ key, float* __restrict__ mn, int* __restrict__ idx, size_t n,
                                          const int* __restrict__ skip, int per_sample, const int* __restrict__ perm) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t smp = i / (size_t)per_sample;
  if (skip && skip[smp]) return;
  u64 k = key[i];
  const size_t o = perm ? smp * (size_t)per_sample + (size_t)perm[i] : i;
  mn[o] = __uint_as_float((unsigned)(k >> 32));
  idx[o] = (int)(unsigned)(k & 0xffffffffu);
}

// ---------------------------------------------------------------------------------------------
// row recovery over spatially sorted clouds (pruned tensor-core filter).  A CTA owns one 128-row block of the sorted
// predicted points, the block the filter's MMAs used.  Sorted rows share most of their candidate 32-column units, so the
// CTA ORs its rows' units into one bit set and stages only that set in shared memory, kStageUnits units per page.  A
// sorted block's set is a few units and fits one page; lattices, duplicates and tie-heavy scenes take several pages,
// each staged and evaluated in turn.  Every (row, unit) item of a page is listed, evaluated with the exact unit code
// above and merged into the row's key with a shared atomicMin, so the result is (min sqrt(d), first original index) over
// the candidate units whatever the order.  The CTAs are small and eight share an SM, so one CTA's record and target
// loads overlap another's evaluation; units index p2v directly, so there is no segment loop for any M.
// ---------------------------------------------------------------------------------------------
constexpr int kOwn = 128;                            // rows per CTA
constexpr int kStageUnits = 32;                      // units staged per page (16 KB)
constexpr int kOwnItemCap = 1024;                    // listed (row, unit) items per round
constexpr int kOwnCtasPerSm = 8;                     // resident CTAs per SM (__launch_bounds__ below)

struct OwnedSmem {
  float4 pts[kStageUnits * 32];                      // the page's units: (x, y, z, original index as int bits)
  float4 own[kOwn];                                  // the rows' coordinates
  u64 key[kOwn];
  unsigned items[kOwnItemCap];                       // row << 8 | slot in the page
  int sunit[kStageUnits];                            // slot in the page -> unit
  int warp_sums[33];
};
// dynamic shared memory: OwnedSmem, then the union's bit words uni[nw] and their exclusive popcount prefix wpre[nw + 1]
constexpr size_t kMaxOwnedSmem = 96 * 1024;         // union words of target clouds up to ~9 M points
static size_t owned_smem_bytes(int nunits) { const size_t nw = ((size_t)nunits + 31) / 32; return sizeof(OwnedSmem) + nw * 4 + (nw + 1) * 4; }

// Row tid's coordinates are in sm.own[tid] before the call.  for_each(f) calls f(unit) for every candidate unit of the
// thread's row (nothing for a row past the end of the cloud).  load(unit, k) returns point k of a unit.  On return
// sm.key[tid] holds the row's key (~0 without candidates).
template <class ForEach, class Load>
__device__ __forceinline__ void owned_recover(OwnedSmem& sm, unsigned* uni, int* wpre, int nw, const ForEach& for_each, const Load& load) {
  const int tid = threadIdx.x, lane = tid & 31;
  for (int i = tid; i < nw; i += kOwn) uni[i] = 0u;
  sm.key[tid] = ~0ull;
  __syncthreads();
  int cnt_all = 0;
  for_each([&](int u) { atomicOr(&uni[u >> 5], 1u << (u & 31)); ++cnt_all; });
  __syncthreads();
  if (tid < 32) {                                    // slot of the union's first unit in each word
    int carry = 0;
    for (int w0 = 0; w0 < nw; w0 += 32) {
      const int w = w0 + lane;
      const int c = w < nw ? __popc(uni[w]) : 0;
      int inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
      if (w < nw) wpre[w] = carry + inc - c;
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) wpre[nw] = carry;
  }
  __syncthreads();
  const int nu = wpre[nw];
  auto slot_of = [&](int u) { return wpre[u >> 5] + __popc(uni[u >> 5] & ((1u << (u & 31)) - 1u)); };
  for (int p0 = 0; p0 < nu; p0 += kStageUnits) {
    const int p1 = min(nu, p0 + kStageUnits);
    if (tid < 32) {
      for (int w = lane; w < nw; w += 32) {
        if (wpre[w] >= p1 || wpre[w + 1] <= p0) continue;
        int s = wpre[w];
        for (unsigned m = uni[w]; m; m &= m - 1u, ++s)
          if (s >= p0 && s < p1) sm.sunit[s - p0] = 32 * w + __ffs((int)m) - 1;
      }
    }
    __syncthreads();
    for (int i = tid; i < (p1 - p0) * 32; i += kOwn) sm.pts[i] = load(sm.sunit[i >> 5], i & 31);
    int cnt = cnt_all;
    if (nu > kStageUnits) {                          // several pages: this page's share of the row's units
      cnt = 0;
      for_each([&](int u) { const int s = slot_of(u); cnt += (s >= p0 && s < p1) ? 1 : 0; });
    }
    int total;
    const int off = block_exclusive_scan<kOwn>(cnt, sm.warp_sums, &total);      // also publishes the staged page
    for (int base = 0; base < total; base += kOwnItemCap) {
      int j = off;
      for_each([&](int u) {
        const int s = slot_of(u);
        if (s >= p0 && s < p1) {
          if (j >= base && j < base + kOwnItemCap) sm.items[j - base] = ((unsigned)tid << 8) | (unsigned)(s - p0);
          ++j;
        }
      });
      __syncthreads();
      const int n = min(kOwnItemCap, total - base);
      for (int it = tid; it < n; it += kOwn) {
        const unsigned item = sm.items[it];
        const int r = item >> 8;
        const float4 rc = sm.own[r];
        const float4* src = sm.pts + (item & 255u) * 32;
        float d[32], dm = inf_f();
#pragma unroll
        for (int kk = 0; kk < 32; ++kk) {
          const float4 q = src[(kk + lane) & 31];
          d[kk] = exact_d2s(rc.x, rc.y, rc.z, q.x, q.y, q.z);
          dm = fminf(dm, d[kk]);
        }
        int at;
        const int st = unit_scan(d, dm, lane, &at);
        if (st == 1) atomicMin(&sm.key[r], ((u64)__float_as_uint(sqrtf(dm)) << 32) | (unsigned)__float_as_int(src[at].w));
        else if (st == 2) { const u64 kv = unit_exact_walk(rc.x, rc.y, rc.z, src, 0, 1); if (kv != ~0ull) atomicMin(&sm.key[r], kv); }
      }
      __syncthreads();                               // the next round or page overwrites items / pts
    }
  }
}

// grid: x = 128-row block of the sorted rows, y = sample.  Records: four u64 planes (plane_stride apart) of 32-column unit
// bits per (split, row), unit 4 c + u of the split = unit 4 (split * cps + c) + u of p2v.  With nsplit > 1 a split's
// record counts only when its best is within the row's threshold (tslack of the row's tile).
// p2v: the sorted targets as (x, y, z, original index), NaN-padded to whole chunks (stride mpad per sample).
__global__ void __launch_bounds__(kOwn, kOwnCtasPerSm)
chamfer_recover_rows_sorted_kernel(const float* __restrict__ p1s, const float4* __restrict__ p2v, int mpad,
                                   const float* __restrict__ rbest, const u64* __restrict__ rmask, size_t plane_stride,
                                   const float2* __restrict__ tslack, float* __restrict__ min1, int* __restrict__ idx1,
                                   int P, int nunits, int nsplit, int cps, int TM, int ntiles,
                                   const int* __restrict__ skip, const int* __restrict__ rperm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  OwnedSmem& sm = *reinterpret_cast<OwnedSmem*>(smem_raw);
  const int nw = (nunits + 31) >> 5;
  unsigned* uni = reinterpret_cast<unsigned*>(smem_raw + sizeof(OwnedSmem));
  int* wpre = reinterpret_cast<int*>(uni + nw);
  const int b = blockIdx.y, tid = threadIdx.x, row = blockIdx.x * kOwn + tid;
  if (skip && skip[b]) return;                       // sample redone by chamfer_flagged_kernel
  const bool valid = row < P;
  const size_t orow = (size_t)b * P + row;
  float gthr = inf_f();
  u64 m1[4] = {0ull, 0ull, 0ull, 0ull};              // the record when there is one split
  if (valid) {
    sm.own[tid] = make_float4(p1s[3 * orow], p1s[3 * orow + 1], p1s[3 * orow + 2], 0.f);
    if (nsplit == 1) {
#pragma unroll
      for (int w = 0; w < 4; ++w) m1[w] = rmask[orow + w * plane_stride];
    } else {
      float g = inf_f();
      for (int s = 0; s < nsplit; ++s) g = fminf(g, rbest[((size_t)b * nsplit + s) * P + row]);
      const float2 sl = tslack[(size_t)b * ntiles + row / TM];
      gthr = thr_of(g, sl.x, sl.y);
    }
  }
  auto for_each = [&](auto&& f) {
    if (!valid) return;
    if (nsplit == 1) {
#pragma unroll
      for (int w = 0; w < 4; ++w)
        for (u64 m = m1[w]; m; m &= m - 1) { const int u = 64 * w + __ffsll((long long)m) - 1; if (u < nunits) f(u); }
      return;
    }
    for (int s = 0; s < nsplit; ++s) {
      const size_t o = ((size_t)b * nsplit + s) * P + row;
      if (!(rbest[o] <= gthr)) continue;
      for (int w = 0; w < 4; ++w) {
        const int u0 = s * cps * 4 + 64 * w;
        for (u64 m = rmask[o + w * plane_stride]; m; m &= m - 1) { const int u = u0 + __ffsll((long long)m) - 1; if (u < nunits) f(u); }
      }
    }
  };
  const float4* tv = p2v + (size_t)b * mpad;
  owned_recover(sm, uni, wpre, nw, for_each, [&](int u, int k) { return __ldg(tv + (size_t)u * 32 + k); });
  if (valid) {
    const u64 kv = sm.key[tid];
    const size_t o = (size_t)b * P + rperm[orow];
    min1[o] = __uint_as_float((unsigned)(kv >> 32));
    idx1[o] = (int)(unsigned)(kv & 0xffffffffu);
  }
}


// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct TiledPlan { int R, ntiles, nchunks, nsplit, cps, tc, TM; };

// chamfer_tc.cu
size_t chamfer_tc_smem_bytes(int NB);
int chamfer_tc_plan_words();
int chamfer_tc_launch(const float* p1, const float* p2, float* rbest, u64* rmask, float* cbest, u64* cmask,
                      float2* tslack, int* fallback, float* tmax, const float* cbox, const float* rbox, const float* rthr,
                      const float* cub, u64* stats, unsigned* plan_masks, int* plan_work, int* plan_order, int with_bounds,
                      int B, int P, int M, int NB, int ntiles, int nsplit, int nchunks, int cps, cudaStream_t s);
// chamfer_prep.cu
int chamfer_prep_launch(const float* p1, const float* p2, float* p2s, float4* p2v, int* perm, float* cbox, float* rbox, float* rthr,
                        float* cub, float* tmax, float* p1s, int* rperm, unsigned long long* stats, int B, int P, int M, cudaStream_t s);
int chamfer_flagged_launch(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                           const int* fallback, int B, int P, int M, cudaStream_t s);

static void finish_plan(TiledPlan& pl, int B, long long slots, int min_cps) {
  long long base = (long long)pl.ntiles * B;
  long long s = (4 * slots + base - 1) / base;
  long long smin = (pl.nchunks + kMaxChunksPerSplit - 1) / kMaxChunksPerSplit;
  long long smax = pl.nchunks / min_cps;
  if (s > smax) s = smax;
  if (s < smin) s = smin;
  if (s > pl.nchunks) s = pl.nchunks;
  if (s < 1) s = 1;
  pl.cps = (int)((pl.nchunks + s - 1) / s);
  pl.nsplit = (pl.nchunks + pl.cps - 1) / pl.cps;
}

// CUDA-core kernel: tile = 256 R rows (R rows per thread)
static bool make_plan(int B, int P, int M, int sm_count, TiledPlan& pl) {
  if (P < 1024 || M < kCW || B < 1) return false;
  pl.tc = 0;
  pl.nchunks = (M + kCW - 1) / kCW;
  const int rs[3] = {16, 8, 4};
  int pick = 4;
  for (int k = 0; k < 3; ++k) {
    int R = rs[k], tm = kTThreads * R;
    long long nt = (P + tm - 1) / tm;
    double waste = (double)(nt * tm) / P;
    long long slots = (long long)sm_count * (R <= 8 ? 2 : 1);
    if (waste <= 1.26 && nt * B * pl.nchunks >= 2 * slots) { pick = R; break; }
  }
  { int r = tuning_value(kTuneTiledR); if (r == 4 || r == 8 || r == 16) pick = r; }   // vpn_set_tuning("tiled_r")
  pl.R = pick;
  pl.TM = kTThreads * pl.R;
  pl.ntiles = (P + pl.TM - 1) / pl.TM;
  finish_plan(pl, B, (long long)sm_count * (pl.R <= 8 ? 2 : 1), 1);
  return pl.nsplit <= 65535;
}

// tensor-core kernel: tile = 128 NB rows (NB row blocks), one CTA per SM; R holds NB
static bool make_plan_tc(int B, int P, int M, int sm_count, TiledPlan& pl) {
  if (P < 512 || M < kCW || B < 1) return false;
  pl.tc = 1;
  pl.nchunks = (M + kCW - 1) / kCW;
  const int nbs[3] = {16, 8, 4};
  int pick = 4;
  for (int k = 0; k < 3; ++k) {
    int nb = nbs[k], tm = 128 * nb;
    long long nt = (P + tm - 1) / tm;
    double waste = (double)(nt * tm) / P;
    if (waste <= 1.26 && nt * B * pl.nchunks >= 2LL * sm_count * 8) { pick = nb; break; }
  }
  { int r = tuning_value(kTuneTcNb); if (r == 4 || r == 8 || r == 16) pick = r; }      // vpn_set_tuning("tc_nb")
  pl.R = pick;
  pl.TM = 128 * pl.R;
  pl.ntiles = (P + pl.TM - 1) / pl.TM;
  // every CTA first builds its row operands: keep >= 4 column chunks per CTA so that this is amortised
  finish_plan(pl, B, sm_count, 4);
  return pl.nsplit <= 65535;
}

static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

struct TiledWs { size_t rbest, rmask, cbest, cmask, tslack, fallback, tmax, cthr, key2, p2s, p2v, perm, cbox, rbox, rthr, cub, pmask, pwork, porder, p1s, rperm, total; };
static TiledWs ws_layout(int B, int P, int M, const TiledPlan& pl) {
  TiledWs w; size_t o = 0;
  w.rbest = o; o += al256((size_t)B * pl.nsplit * P * 4);
  w.rmask = o; o += al256((size_t)B * pl.nsplit * P * 8 * (pl.tc ? 4 : 1));      // tensor-core filter: four planes of unit bits
  w.cbest = o; o += al256((size_t)B * pl.ntiles * M * 4);
  w.cmask = o; o += al256((size_t)B * pl.ntiles * M * (pl.tc ? 8 : 4));          // tensor-core filter: 64 unit bits
  w.tslack = o; o += al256((size_t)B * pl.ntiles * 8);
  w.fallback = o; o += al256((size_t)B * 4 + 8 + 128);     // + 16 x u64 statistics / cycle counters of the tensor-core filter, zeroed with the flags
  w.tmax = o; o += al256((size_t)B * 4);
  w.cthr = o; o += al256((size_t)B * M * 4);
  w.key2 = o; o += al256((size_t)B * M * 8);
  w.p2s = w.p2v = w.perm = w.cbox = w.rbox = w.rthr = w.cub = w.pmask = w.pwork = w.porder = w.p1s = w.rperm = 0;
  if (pl.tc) {                                             // spatial preparation of the pruned tensor-core filter (chamfer_prep.cu)
    const size_t nrb = (size_t)(P + 127) / 128;
    w.p2s = o; o += al256((size_t)B * M * 12);
    w.p2v = o; o += al256((size_t)B * pl.nchunks * kCW * 16);     // (x, y, z, original index), NaN-padded to whole chunks
    w.perm = o; o += al256((size_t)B * M * 4);
    w.cbox = o; o += al256((size_t)B * pl.nchunks * 32);
    w.rbox = o; o += al256((size_t)B * nrb * 32);
    w.rthr = o; o += al256((size_t)B * nrb * 4);
    w.cub = o; o += al256((size_t)B * pl.nchunks * 4);
    const size_t ncta = (size_t)pl.ntiles * pl.nsplit * B;         // tiles of the filter: skip masks, work, run order
    w.pmask = o; o += al256(ncta * (size_t)chamfer_tc_plan_words() * 4);
    w.pwork = o; o += al256(ncta * 4);
    w.porder = o; o += al256(ncta * 4);
    w.p1s = o; o += al256((size_t)B * P * 12);                     // predicted points, Morton-sorted inside 4096-row segments
    w.rperm = o; o += al256((size_t)B * P * 4);                    // sorted row -> original row
  }
  w.total = o;
  return w;
}

// mode: -1 auto, MODE_*.  Auto prefers the tensor-core filter.  The plan depends on the SM count of the current
// device: the workspace query and the launch must be made with the same device current (they are: same thread).
static bool plan_for(int mode, int B, int P, int M, TiledPlan& pl) {
  const int kPlanSms = device_sm_count();
  if (mode == MODE_TC) return make_plan_tc(B, P, M, kPlanSms, pl);
  if (mode >= 0) return make_plan(B, P, M, kPlanSms, pl);
  return make_plan_tc(B, P, M, kPlanSms, pl) || make_plan(B, P, M, kPlanSms, pl);
}

int chamfer_tiled_supported(int B, int P, int M, int mode) {
  TiledPlan pl;
  return plan_for(mode, B, P, M, pl) ? 1 : 0;
}

int chamfer_tiled_uses_tc(int B, int P, int M, int mode) {
  TiledPlan pl;
  return (plan_for(mode, B, P, M, pl) && pl.tc) ? 1 : 0;
}

size_t chamfer_tiled_workspace_bytes(int B, int P, int M, int mode) {
  TiledPlan pl;
  if (!plan_for(mode, B, P, M, pl)) return 0;
  return ws_layout(B, P, M, pl).total;
}

// Statistics of the last tensor-core forward that used this workspace: out[0] = 128 x 256 stages in the sweep,
// out[1] = stages skipped, out[2..9] = cycle / work counters (chamfer_tc.cu), out[10..15] = 0.  Synchronises the stream.
int chamfer_tiled_stats(int B, int P, int M, int mode, const void* ws_, unsigned long long* out, cudaStream_t s) {
  TiledPlan pl;
  for (int i = 0; i < 16; ++i) out[i] = 0;
  if (!plan_for(mode, B, P, M, pl) || !pl.tc) return VPN_OK;
  TiledWs wl = ws_layout(B, P, M, pl);
  const char* src = reinterpret_cast<const char*>(ws_) + wl.fallback + (((size_t)B * 4 + 7) & ~(size_t)7);
  if (cudaMemcpyAsync(out, src, 128, cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
    vpn_set_error("chamfer stats: copy failed"); return VPN_ERR_CUDA;
  }
  return VPN_OK;
}

template <int R, int MODE>
static int launch_main(const float* p1, const float* p2, char* ws, const TiledWs& wl, const TiledPlan& pl,
                       int B, int P, int M, int only_flagged, cudaStream_t s) {
  static DeviceOnce once;
  size_t smem = sizeof(TiledSmem<R>);
  {
    cudaError_t e = set_dyn_smem(chamfer_tiled_kernel<R, MODE>, (int)smem, once);
    if (e != cudaSuccess) { vpn_set_error("chamfer tiled: smem attribute: %s", cudaGetErrorString(e)); return VPN_ERR_CUDA; }
  }
  dim3 grid(pl.ntiles, pl.nsplit, B);
  chamfer_tiled_kernel<R, MODE><<<grid, kTThreads, smem, s>>>(
      p1, p2, reinterpret_cast<float*>(ws + wl.rbest), reinterpret_cast<u64*>(ws + wl.rmask),
      reinterpret_cast<float*>(ws + wl.cbest), reinterpret_cast<unsigned*>(ws + wl.cmask),
      reinterpret_cast<float2*>(ws + wl.tslack), reinterpret_cast<int*>(ws + wl.fallback),
      P, M, pl.nchunks, pl.cps, 1.0f, only_flagged);
  return vpn_check_launch("chamfer_tiled_kernel");
}

template <int R>
static int launch_main_mode(int mode, const float* p1, const float* p2, char* ws, const TiledWs& wl, const TiledPlan& pl,
                            int B, int P, int M, int only_flagged, cudaStream_t s) {
  switch (mode) {
    case MODE_EXACT: return launch_main<R, MODE_EXACT>(p1, p2, ws, wl, pl, B, P, M, only_flagged, s);
    case MODE_DIFF:  return launch_main<R, MODE_DIFF>(p1, p2, ws, wl, pl, B, P, M, only_flagged, s);
    default:         return launch_main<R, MODE_EXPAND>(p1, p2, ws, wl, pl, B, P, M, only_flagged, s);
  }
}

static int launch_any(int mode, const float* p1, const float* p2, char* ws, const TiledWs& wl, const TiledPlan& pl,
                      int B, int P, int M, int only_flagged, cudaStream_t s) {
  switch (pl.R) {
    case 16: return launch_main_mode<16>(mode, p1, p2, ws, wl, pl, B, P, M, only_flagged, s);
    case 8:  return launch_main_mode<8>(mode, p1, p2, ws, wl, pl, B, P, M, only_flagged, s);
    default: return launch_main_mode<4>(mode, p1, p2, ws, wl, pl, B, P, M, only_flagged, s);
  }
}

template <int R, bool TC>
static int launch_recover_cols(const float* p1, const float* p2, const float* cb, const void* cmk, const float* cthr,
                               u64* key2, int B, int P, int M, int ntiles, const int* skip, const int* rperm, cudaStream_t s) {
  static DeviceOnce once, once_half;
  const size_t smem = (size_t)(TC ? 128 * R : kTThreads * R) * sizeof(float4);
  // 512-thread CTAs, two per SM, once the grid fills the machine twice (C2: 1024 CTAs, 79 -> 73 us); a grid below that (C5:
  // 64 CTAs) is faster with all 1024 threads on its few CTAs
  if (TC && (long long)ntiles * B >= 2LL * device_sm_count()) {
    if (set_dyn_smem(chamfer_recover_cols_kernel<R, TC, 512>, (int)smem, once_half) != cudaSuccess) {
      vpn_set_error("chamfer tiled: smem attribute (cols recovery)"); return VPN_ERR_CUDA;
    }
    chamfer_recover_cols_kernel<R, TC, 512><<<dim3(ntiles, B), 512, smem, s>>>(p1, p2, cb, cmk, cthr, key2, P, M, ntiles, skip, rperm);
    return vpn_check_launch("chamfer_recover_cols_kernel");
  }
  if (set_dyn_smem(chamfer_recover_cols_kernel<R, TC, kRecThreads>, (int)smem, once) != cudaSuccess) {
    vpn_set_error("chamfer tiled: smem attribute (cols recovery)"); return VPN_ERR_CUDA;
  }
  chamfer_recover_cols_kernel<R, TC, kRecThreads><<<dim3(ntiles, B), kRecThreads, smem, s>>>(p1, p2, cb, cmk, cthr, key2, P, M, ntiles, skip, rperm);
  return vpn_check_launch("chamfer_recover_cols_kernel");
}

// The row recovery and the column recovery chain (threshold, recovery, unpack) are independent and each leaves most of
// an SM idle (ncu: 60 % / 28 % issue utilisation; a 131 KB and a 33 KB CTA fit one SM together), so the column chain is
// forked onto a per-device side stream and joined before the call returns control of `s` - under CUDA-graph capture
// the fork / join becomes two parallel branches.  The side stream and its two events are created on first use outside
// a capture (never during one: the call then runs the chain serially) and the enqueue section is serialised per
// device, so concurrent host threads cannot interleave their event records.
struct SideStream { cudaStream_t s = nullptr; cudaEvent_t fork = nullptr, join = nullptr; bool ok = false; std::mutex mu; };
static SideStream g_side[64];
static SideStream* side_stream_for(cudaStream_t s) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SideStream& ss = g_side[dev];
  if (ss.ok) return &ss;
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) { cudaGetLastError(); return nullptr; }
  std::lock_guard<std::mutex> lock(ss.mu);
  if (!ss.ok) {
    if (cudaStreamCreateWithFlags(&ss.s, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    ss.ok = true;
  }
  return &ss;
}

// mode: -1 auto, 0 exact, 1 diff, 2 expand, 3 tensor-core filter.  events (optional, 5 entries) bracket the stages.
int chamfer_tiled_fwd(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                      int B, int P, int M, void* ws_, size_t ws_bytes, int mode, cudaStream_t s, cudaEvent_t* ev) {
  TiledPlan pl;
  if (!plan_for(mode, B, P, M, pl)) { vpn_set_error("chamfer tiled: unsupported shape"); return VPN_ERR_SHAPE; }
  if (mode < 0) mode = pl.tc ? MODE_TC : MODE_EXPAND;
  TiledWs wl = ws_layout(B, P, M, pl);
  if (ws_bytes < wl.total) { vpn_set_error("chamfer tiled: workspace too small (%zu < %zu)", ws_bytes, wl.total); return VPN_ERR_WORKSPACE; }
  char* ws = reinterpret_cast<char*>(ws_);
  int* fallback = reinterpret_cast<int*>(ws + wl.fallback);
  const int* skip = nullptr;
  int rc;
  if (ev) cudaEventRecord(ev[0], s);
  const size_t flag_bytes = (((size_t)B * 4 + 7) & ~(size_t)7) + 128;     // per-sample flags + the 16 u64 statistics words
  if (mode == MODE_EXPAND || mode == MODE_TC) {
    if (cudaMemsetAsync(fallback, 0, flag_bytes, s) != cudaSuccess) { vpn_set_error("chamfer tiled: memset failed"); return VPN_ERR_CUDA; }
  }
  const float* p2w = p2;                       // the targets the sweep and the recovery kernels read
  const int* perm = nullptr;                   // sorted position -> original index (tensor-core mode)
  const float4* p2v = nullptr;                 // the swept targets as (x, y, z, original index) (tensor-core mode, pruned)
  const float* p1w = p1;                       // the predicted points the sweep and the recovery kernels read
  const int* rperm = nullptr;                  // sorted row -> original row (tensor-core mode, pruned)
  if (mode == MODE_TC) {
    float* p2s = reinterpret_cast<float*>(ws + wl.p2s);
    int* pm = reinterpret_cast<int*>(ws + wl.perm);
    float* cbox = reinterpret_cast<float*>(ws + wl.cbox); float* rbox = reinterpret_cast<float*>(ws + wl.rbox);
    float* rthr = reinterpret_cast<float*>(ws + wl.rthr); float* cub = reinterpret_cast<float*>(ws + wl.cub);
    float* tmax = reinterpret_cast<float*>(ws + wl.tmax);
    u64* stats = reinterpret_cast<u64*>(ws + wl.fallback + (((size_t)B * 4 + 7) & ~(size_t)7));
    const bool prune = tuning_value(kTuneTcPrune) != 2;                      // vpn_set_tuning("tc_prune", 2): unpruned sweep
    if (prune) {
      float4* pv = reinterpret_cast<float4*>(ws + wl.p2v);
      float* p1s = reinterpret_cast<float*>(ws + wl.p1s);
      int* rp = reinterpret_cast<int*>(ws + wl.rperm);
      if ((rc = chamfer_prep_launch(p1, p2, p2s, pv, pm, cbox, rbox, rthr, cub, tmax, p1s, rp, stats, B, P, M, s))) return rc;
      p2w = p2s; perm = pm; p2v = pv; p1w = p1s; rperm = rp;
    }
    rc = chamfer_tc_launch(p1w, p2w, reinterpret_cast<float*>(ws + wl.rbest), reinterpret_cast<u64*>(ws + wl.rmask),
                           reinterpret_cast<float*>(ws + wl.cbest), reinterpret_cast<u64*>(ws + wl.cmask),
                           reinterpret_cast<float2*>(ws + wl.tslack), fallback, tmax, prune ? cbox : nullptr, rbox, rthr, cub, stats,
                           reinterpret_cast<unsigned*>(ws + wl.pmask), reinterpret_cast<int*>(ws + wl.pwork),
                           reinterpret_cast<int*>(ws + wl.porder), prune ? 0 : 1, B, P, M, pl.R, pl.ntiles, pl.nsplit, pl.nchunks,
                           pl.cps, s);
    if (rc) return rc;
    if (ev) cudaEventRecord(ev[1], s);
    // samples outside the filter's validity range (non-finite / huge coordinates): exact brute force, recovery skips them
    if ((rc = chamfer_flagged_launch(p1, p2, min1, idx1, min2, idx2, fallback, B, P, M, s))) return rc;
    skip = fallback;
  } else {
    if ((rc = launch_any(mode, p1, p2, ws, wl, pl, B, P, M, 0, s))) return rc;
    if (ev) cudaEventRecord(ev[1], s);
    if (mode == MODE_EXPAND) {
      if ((rc = launch_any(MODE_DIFF, p1, p2, ws, wl, pl, B, P, M, 1, s))) return rc;
    }
  }
  if (ev) cudaEventRecord(ev[2], s);
  // fork: the column chain runs on the side stream `sc`, the row recovery on `s`
  SideStream* side = tuning_value(kTuneSerialRecovery) ? nullptr : side_stream_for(s);
  std::unique_lock<std::mutex> side_lock;
  cudaStream_t sc = s;
  if (side) {
    side_lock = std::unique_lock<std::mutex>(side->mu);
    if (cudaEventRecord(side->fork, s) == cudaSuccess && cudaStreamWaitEvent(side->s, side->fork, 0) == cudaSuccess) sc = side->s;
    else { cudaGetLastError(); side = nullptr; side_lock.unlock(); }
  }
  // Sorted clouds take the per-block row recovery when its grid fills the machine at least once; a smaller grid (C5:
  // 1024 blocks, 0.078 against 0.047 ms on one B200) leaves each block's chain of dependent loads and barriers exposed,
  // and the persistent kernel below is faster there.
  const long long sorted_blocks = (long long)B * ((P + kOwn - 1) / kOwn);
  if (p2v && sorted_blocks >= (long long)kOwnCtasPerSm * device_sm_count()) {
    static DeviceOnce once_rows_sorted;
    const int nunits = pl.nchunks * 4;
    const size_t smem = owned_smem_bytes(nunits);
    if (smem > kMaxOwnedSmem) { vpn_set_error("chamfer tiled: target cloud too large for the row recovery"); return VPN_ERR_SHAPE; }
    if (set_dyn_smem(chamfer_recover_rows_sorted_kernel, (int)kMaxOwnedSmem, once_rows_sorted) != cudaSuccess) {
      vpn_set_error("chamfer tiled: smem attribute (rows recovery)"); return VPN_ERR_CUDA;
    }
    chamfer_recover_rows_sorted_kernel<<<dim3((P + kOwn - 1) / kOwn, B), kOwn, smem, s>>>(
        p1w, p2v, pl.nchunks * kCW, reinterpret_cast<const float*>(ws + wl.rbest), reinterpret_cast<const u64*>(ws + wl.rmask),
        (size_t)B * pl.nsplit * P, reinterpret_cast<const float2*>(ws + wl.tslack), min1, idx1, P, nunits, pl.nsplit, pl.cps,
        pl.TM, pl.ntiles, skip, rperm);
    if ((rc = vpn_check_launch("chamfer_recover_rows_sorted_kernel"))) return rc;
  } else {
    static DeviceOnce once_rows;
    const size_t smem_rows = kRowsFixedSmem + (size_t)(pl.nchunks < kSegChunks ? pl.nchunks : kSegChunks) * kCW * sizeof(float4);
    if (set_dyn_smem(chamfer_recover_rows_kernel, (int)(kRowsFixedSmem + kSegChunks * kCW * sizeof(float4)), once_rows) != cudaSuccess) {
      vpn_set_error("chamfer tiled: smem attribute (rows recovery)"); return VPN_ERR_CUDA;
    }
    const int nblk = (P + kRowGroup - 1) / kRowGroup;
    const long long nitems = (long long)nblk * B;
    if (nitems > 0x7fffffffLL) { vpn_set_error("chamfer tiled: too many row blocks"); return VPN_ERR_SHAPE; }
    const int sms = device_sm_count();
    chamfer_recover_rows_kernel<<<(unsigned)(nitems < sms ? nitems : sms), kRecThreads, smem_rows, s>>>(
        p1w, p2w, p2v, pl.nchunks * kCW, reinterpret_cast<const float*>(ws + wl.rbest), reinterpret_cast<const u64*>(ws + wl.rmask),
        pl.tc ? 4 : 1, (size_t)B * pl.nsplit * P, reinterpret_cast<const float2*>(ws + wl.tslack), min1, idx1, P, M, pl.nchunks,
        pl.nsplit, pl.cps, pl.TM, pl.ntiles, skip, nblk, (int)nitems, rperm);
    if ((rc = vpn_check_launch("chamfer_recover_rows_kernel"))) return rc;
  }
  if (ev) cudaEventRecord(ev[3], s);          // with the fork: end of the row recovery; [3]..[4] = what the column chain adds after it
  const float* cb = reinterpret_cast<const float*>(ws + wl.cbest);
  const void* cmk = ws + wl.cmask;
  const float2* tsl = reinterpret_cast<const float2*>(ws + wl.tslack);
  float* cthr = reinterpret_cast<float*>(ws + wl.cthr);
  u64* key2 = reinterpret_cast<u64*>(ws + wl.key2);
  if (cudaMemsetAsync(key2, 0xFF, (size_t)B * M * 8, sc) != cudaSuccess) { vpn_set_error("chamfer tiled: memset failed"); return VPN_ERR_CUDA; }
  chamfer_col_thr_kernel<<<dim3((M + 255) / 256, B), 256, 0, sc>>>(cb, tsl, cthr, M, pl.ntiles);
  if ((rc = vpn_check_launch("chamfer_col_thr_kernel"))) return rc;
  if (pl.tc) {
    switch (pl.R) {
      case 16: rc = launch_recover_cols<16, true>(p1w, p2w, cb, cmk, cthr, key2, B, P, M, pl.ntiles, skip, rperm, sc); break;
      case 8:  rc = launch_recover_cols<8, true>(p1w, p2w, cb, cmk, cthr, key2, B, P, M, pl.ntiles, skip, rperm, sc); break;
      default: rc = launch_recover_cols<4, true>(p1w, p2w, cb, cmk, cthr, key2, B, P, M, pl.ntiles, skip, rperm, sc); break;
    }
  } else {
    switch (pl.R) {
      case 16: rc = launch_recover_cols<16, false>(p1, p2, cb, cmk, cthr, key2, B, P, M, pl.ntiles, skip, nullptr, sc); break;
      case 8:  rc = launch_recover_cols<8, false>(p1, p2, cb, cmk, cthr, key2, B, P, M, pl.ntiles, skip, nullptr, sc); break;
      default: rc = launch_recover_cols<4, false>(p1, p2, cb, cmk, cthr, key2, B, P, M, pl.ntiles, skip, nullptr, sc); break;
    }
  }
  if (rc) return rc;
  {
    size_t n = (size_t)B * M;
    chamfer_unpack_key_kernel<<<(unsigned)((n + 255) / 256), 256, 0, sc>>>(key2, min2, idx2, n, skip, M, perm);
  }
  rc = vpn_check_launch("chamfer_unpack_key_kernel");
  if (side) {                                  // join
    if (cudaEventRecord(side->join, sc) != cudaSuccess || cudaStreamWaitEvent(s, side->join, 0) != cudaSuccess) {
      vpn_set_error("chamfer tiled: stream join failed"); rc = VPN_ERR_CUDA;
    }
  }
  if (ev) cudaEventRecord(ev[4], s);
  return rc;
}

}  // namespace vpn
