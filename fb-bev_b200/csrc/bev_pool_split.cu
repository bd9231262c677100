// bev_pool_split.cu -- dense lift-splat pooling as two lean kernels.
//
// Evidence behind the structure (profiles/, DESIGN.md section 5):
//  * tools/micro/store_pattern.cu: writing the (B,C,Z,Y,X) volume as per-tile
//    channel rows (128-bit stores, 512 B per row and tile) runs at memset speed
//    on B200 (35 us for 204.8 MB) -- the output pattern is not the limit;
//  * every fused single-kernel variant measured (one tile per CTA, persistent,
//    cp.async-pipelined, TMA-store) stayed at 60-100 us with the SM issue slots
//    ~55 % busy (37-51 M warp instructions) and long-scoreboard / barrier stalls:
//    index chasing (tile table -> index words -> depth / feat rows) inside the
//    CTA that owns the 40 KB output tile starves the store stream.
// So the index chasing is moved out of the CTA that owns an output tile:
//
//  K1 "interval sums": warp w folds the 32 kept points [32w, 32w+32) --
//      perfectly balanced, so the dense voxels next to a camera (up to 63
//      points on the 200x200x16 grid, thousands on the 1-camera 128x128 grid:
//      the reference kernel's and every tile-owning kernel's tail) are spread
//      over many warps.  Coalesced index loads; a 4-lane group owns 4
//      consecutive points (128-bit feat loads that depend only on the index
//      words, one FMA per point and channel in point order,
//      bev_pool_cuda.cu:36-40) and runs of equal voxel rank are stitched
//      across groups through shared memory.  Interval sums go to compact rows
//      V[interval][C] (43 MB for the 200x200x16 grid; they stay in L2), the
//      part of an interval that spills into later slices to carry rows
//      X[slice][C].
//  K2 "dense write": a CTA owns T consecutive voxel ranks x all C channels.
//      Empty tiles stream zeros at once; the others copy the rows of their
//      contiguous intervals V[i0:i1] into shared memory with cp.async, add
//      carry rows in slice order, and stream the tile out channel row by channel
//      row with 128-bit evict-first stores.
//  Every output element and every V / X row is written exactly once; no
//  atomics; results are deterministic.
//
// Requires C % 4 == 0 and (Z*Y*X) % 4 == 0, 16-byte aligned out.
#include <algorithm>
#include <cstdlib>

#include "bev_pool_split.h"
#include "bulk.cuh"

namespace fbbev {

#ifndef FBBEV_SUM_THREADS
#define FBBEV_SUM_THREADS 128
#endif
#ifndef FBBEV_SUM_MINB
#define FBBEV_SUM_MINB 6
#endif
constexpr int kSumThreads = FBBEV_SUM_THREADS;  // interval-sum CTAs

// ------------------------------- plan --------------------------------------
// tile_first[t] = first interval of tile t (tile_first[n_tiles] = n);
// seg_rank[i]   = voxel rank of interval i;
// warp_first[w] = first interval starting at or after point 32*w: K1's warp w
//                 owns intervals [warp_first[w], warp_first[w+1]) -- whole
//                 intervals only, about kPtsPerWarp points each, so a dense
//                 region near a camera is spread over many warps instead of
//                 serialising one (the reference kernel's and every
//                 tile-owning kernel's tail, see profiles/);
// meta = {n_intervals, n_kept_points, n_warps}.
constexpr int kPtsPerWarp = 32;

__global__ void split_plan_kernel(
    const int* __restrict__ ranks_bev, const int* __restrict__ interval_starts,
    const int* __restrict__ interval_lengths, int n_intervals_max,
    const int* __restrict__ n_intervals_dev, int n_warps_max, int64_t zyx,
    int tiles_per_b, int T, int64_t n_tiles, int* __restrict__ tile_first,
    int* __restrict__ seg_rank, int* __restrict__ warp_first,
    int* __restrict__ meta) {
  const int n = n_intervals_dev ? min(*n_intervals_dev, n_intervals_max)
                                : n_intervals_max;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t gsz = (int64_t)gridDim.x * blockDim.x;
  if (n <= 0) {
    if (gid == 0) meta[0] = meta[1] = meta[2] = 0;
    for (int64_t t = gid; t <= n_tiles; t += gsz) tile_first[t] = 0;
    return;
  }
  const int n_kept = interval_starts[n - 1] + interval_lengths[n - 1];
  const int n_warps = min((n_kept + kPtsPerWarp - 1) / kPtsPerWarp, n_warps_max);
  if (gid == 0) {
    meta[0] = n;
    meta[1] = n_kept;
    meta[2] = n_warps;
  }
  auto tile_of = [&](int64_t rank) {
    const int64_t b = rank / zyx;
    const int64_t t = b * tiles_per_b + (rank - b * zyx) / T;
    return max((int64_t)0, min(t, n_tiles - 1));
  };
  for (int64_t i = gid; i < n; i += gsz) {
    const int rank = ranks_bev[interval_starts[i]];
    seg_rank[i] = rank;
    const int64_t t = tile_of(rank);
    const int64_t tp =
        i > 0 ? tile_of(ranks_bev[interval_starts[i - 1]]) : (int64_t)-1;
    for (int64_t u = tp + 1; u <= t; ++u) tile_first[u] = (int)i;
    if (i == n - 1)
      for (int64_t u = t + 1; u <= n_tiles; ++u) tile_first[u] = n;
  }
  for (int64_t w = gid; w <= n_warps; w += gsz) {
    int lo = 0, hi = n;  // lower_bound(interval_starts, 32*w)
    const int key = (int)w * kPtsPerWarp;
    if (w == n_warps) lo = n;
    else
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (interval_starts[mid] < key) lo = mid + 1; else hi = mid;
      }
    warp_first[w] = lo;
  }
}

#ifdef POOL_TRACE
// -DPOOL_TRACE: timeline of lane 0 / warp 0 of two CTAs of interval_sums_kernel
// (the first one and one of the last wave), read back with
// fbbev_debug_pool_trace (tools/pool_trace.py).  `dep` ties the clock read to
// the value it follows, so a tag is taken when that value has arrived.
__device__ long long g_pool_trace[2][16];
__device__ __forceinline__ void pool_trace(int slot, int tag, unsigned dep) {
  long long t;
  asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) : "r"(dep) : "memory");
  if (slot >= 0 && (threadIdx.x == 0) && tag < 16) g_pool_trace[slot][tag] = t;
}
#define PTRACE(tag, dep) pool_trace(trace_slot, tag, (unsigned)(dep))
#else
#define PTRACE(tag, dep) do {} while (0)
#endif

// --------------------------- K1: interval sums -----------------------------
// Warp w folds exactly the 32 kept points [32w, 32w+32): perfectly balanced, so
// the dense voxels next to a camera (up to 63 points each on the 200x200x16
// grid, thousands on the 1-camera 128x128 grid) are spread over many warps.
// Two dependent loads reach the data (plan table -> index words, coalesced).
// An LG-lane group owns LG CONSECUTIVE points of the slice, whatever the run
// structure: its 128-bit feat loads (VPL per lane and point) depend only on the
// index words, so two points per lane are in flight and the load chain does not
// grow with the run lengths.  The group folds its points in point order (one
// FMA per point and channel, bev_pool_cuda.cu:36-40); a run of equal voxel rank
// that ends inside the group is flushed at once, a run that crosses into the
// following groups collects their leading partial sums ("heads") through shared
// memory, in point order.
// A run that STARTS in the slice is stored to its row V[interval]; the leading
// part of an interval that started in an earlier slice goes to the slice's
// carry row X[w] and is added, in slice order, by K2.  Every row is written
// exactly once; no atomics; deterministic.
template <int LG, int VPL>
__global__ void __launch_bounds__(kSumThreads, FBBEV_SUM_MINB)
    interval_sums_kernel(const float* __restrict__ depth,
                         const float* __restrict__ feat,
                         const int* __restrict__ ranks_depth,
                         const int* __restrict__ ranks_feat,
                         const int* __restrict__ ranks_bev,
                         const int* __restrict__ interval_starts,
                         const int* __restrict__ warp_first,
                         const int* __restrict__ meta, int c,
                         float* __restrict__ V, float* __restrict__ X) {
  constexpr int WPC = kSumThreads / kWarp;
  constexpr int GPW = kWarp / LG;  // groups per warp
  __shared__ float4 s_head[WPC][GPW][LG * VPL];
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int64_t w = (int64_t)blockIdx.x * WPC + wi;
#ifdef POOL_TRACE
  const int trace_slot = blockIdx.x == 0 ? 0 : (blockIdx.x == gridDim.x - 8 ? 1 : -1);
#endif
  PTRACE(0, 0);
  if (w >= meta[2]) return;
  PTRACE(1, meta[2]);
  const int n = meta[0];
  const int base = (int)w * kPtsPerWarp;
  const int cnt = min(kPtsPerWarp, meta[1] - base);
  const int lb = __ldg(warp_first + w);
  int rbL = -1, rfL = 0;
  float dL = 0.f;
  if (lane < cnt) {
    rbL = __ldg(ranks_bev + base + lane);
    rfL = __ldg(ranks_feat + base + lane);
    dL = __ldg(depth + __ldg(ranks_depth + base + lane));
  }
  PTRACE(2, rbL ^ rfL ^ lb);
  PTRACE(3, __float_as_uint(dL));
  // does the slice begin inside an interval that started earlier?
  const int carry = !(lb < n && __ldg(interval_starts + lb) == base);
  const int prev = __shfl_up_sync(kFull, rbL, 1);
  const unsigned starts =
      __ballot_sync(kFull, lane < cnt && (lane == 0 || rbL != prev));
  PTRACE(4, starts ^ carry);

  const int gl = lane % LG, g = lane / LG, p0 = g * LG;
  const int c4 = c >> 2;
  const float4* feat4 = reinterpret_cast<const float4*>(feat) + gl;
  float4* V4 = reinterpret_cast<float4*>(V) + gl;
  float4* X4 = reinterpret_cast<float4*>(X) + gl;
  float4* hd = &s_head[wi][g][gl];

  float4 acc[VPL];
#pragma unroll
  for (int q = 0; q < VPL; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  bool head = !((starts >> p0) & 1u);  // the group opens inside a run
  int cur = p0;                        // first point of the run being folded

  // store the finished run: a head goes to shared memory, a run that started
  // in this group to its own row
  auto flush = [&]() {
    float4* dst;
    if (head) {
      dst = hd;
    } else {
      const int j = __popc(starts & ((1u << cur) - 1u));
      dst = (j == 0 && carry) ? X4 + w * c4
                              : V4 + (int64_t)(lb + j - carry) * c4;
    }
#pragma unroll
    for (int q = 0; q < VPL; ++q)
      if (head || gl + LG * q < c4) dst[LG * q] = acc[q];
  };

#pragma unroll
  for (int k = 0; k < LG; k += 2) {
    const int pa = p0 + k, pb = pa + 1;
    const int rfa = __shfl_sync(kFull, rfL, pa), rfb = __shfl_sync(kFull, rfL, pb);
    const float da = __shfl_sync(kFull, dL, pa), db = __shfl_sync(kFull, dL, pb);
    float4 xa[VPL], xb[VPL];
    const float4* fa = feat4 + (int64_t)rfa * c4;
    const float4* fb = feat4 + (int64_t)rfb * c4;
#pragma unroll
    for (int q = 0; q < VPL; ++q) {
      const bool col = gl + LG * q < c4;
      xa[q] = (col && pa < cnt) ? __ldg(fa + LG * q)
                                : make_float4(0.f, 0.f, 0.f, 0.f);
      xb[q] = (col && pb < cnt) ? __ldg(fb + LG * q)
                                : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (pa < cnt) {
      if (k > 0 && ((starts >> pa) & 1u)) {
        flush();
#pragma unroll
        for (int q = 0; q < VPL; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        head = false;
        cur = pa;
      }
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        acc[q].x = fmaf(xa[q].x, da, acc[q].x);
        acc[q].y = fmaf(xa[q].y, da, acc[q].y);
        acc[q].z = fmaf(xa[q].z, da, acc[q].z);
        acc[q].w = fmaf(xa[q].w, da, acc[q].w);
      }
    }
    if (pb < cnt) {
      if ((starts >> pb) & 1u) {
        flush();
#pragma unroll
        for (int q = 0; q < VPL; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        head = false;
        cur = pb;
      }
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        acc[q].x = fmaf(xb[q].x, db, acc[q].x);
        acc[q].y = fmaf(xb[q].y, db, acc[q].y);
        acc[q].z = fmaf(xb[q].z, db, acc[q].z);
        acc[q].w = fmaf(xb[q].w, db, acc[q].w);
      }
    }
    PTRACE(5 + k / 2, __float_as_uint(acc[0].x));  // batch k / 2 folded
  }
  // the run that reaches the end of the group
  if (head) flush();  // the whole group continues an earlier run
  if (GPW > 1) __syncwarp();
  PTRACE(13, 0);
  if (!head && p0 < cnt) {
    for (int h = g + 1; h < GPW; ++h) {
      const int ph = h * LG;
      if (ph >= cnt || ((starts >> ph) & 1u)) break;
      const float4* src = &s_head[wi][h][gl];
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const float4 t = src[LG * q];
        acc[q].x += t.x; acc[q].y += t.y; acc[q].z += t.z; acc[q].w += t.w;
      }
      const unsigned later = LG == 32 ? starts : (starts >> ph) & ((1u << (LG & 31)) - 1u);
      if (later) break;  // the run ended inside group h
    }
    flush();
  }
  PTRACE(14, 0);
}

// ---------------------------- K2: dense write ------------------------------
// smem: rows[T + 1][c + 4] (row T stays zero: the row of an empty voxel)
//       | slot[T] (row of each voxel) | carry_lo[T], carry_n[T] (carry rows
//       X[lo+1 .. lo+n] of each interval)
template <int T>
__global__ void __launch_bounds__(2 * T, 1280 / (2 * T)) dense_write_kernel(
    const float* __restrict__ V, const float* __restrict__ X,
    const int* __restrict__ tile_first, const int* __restrict__ seg_rank,
    const int* __restrict__ interval_starts,
    const int* __restrict__ interval_lengths, int c, int zyx,
    const float* __restrict__ add, int yx_n, float* __restrict__ out, int part) {
  // `part`: 0 every tile; 1 only the EMPTY tiles (their zero / `add` stream
  // needs nothing but the plan, so it can run beside the interval sums); 2 only
  // the tiles that hold intervals.
  // `add` (may be null): a (B, C, Y*X) map added to every Z slice while the
  // tile streams out -- FBOCC's `bev_feat_refined[..., None] + bev_feat`
  // (fbocc.py:365-366) without a second pass over the volume
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int pitch = c + 4;  // 16-byte aligned rows, 4-way bank spread
  float* rows = reinterpret_cast<float*>(smem_raw);  // [T + 1][pitch]
  int* slot = reinterpret_cast<int*>(rows + (size_t)(T + 1) * pitch);  // [T]
  int* carry_lo = slot + T;
  int* carry_n = carry_lo + T;

  constexpr int kWrThreads = 2 * T, kWrWarps = kWrThreads / kWarp;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y;
  const int tile = b * gridDim.x + blockIdx.x;
  const int v0 = blockIdx.x * T;
  const int nv = min(T, zyx - v0);
  const int i0 = __ldg(tile_first + tile);
  const int i1 = __ldg(tile_first + tile + 1);
  const int nrows = min(i1 - i0, T);
  if ((part == 1 && nrows > 0) || (part == 2 && nrows <= 0)) return;
  const int c4 = c >> 2;
  constexpr int LPR = T / 4;        // lanes per channel row
  constexpr int RPW = kWarp / LPR;  // rows per warp instruction
  const int g = lane % LPR;
  const int row0 = warp * RPW + lane / LPR;
  float* o = out + ((int64_t)b * c + row0) * zyx + v0 + 4 * g;
  const int64_t step = (int64_t)kWrWarps * RPW * zyx;
  const float* ap = nullptr;  // this lane's four voxels in the `add` map
  int64_t astep = 0;
  if (add) {
    ap = add + ((int64_t)b * c + row0) * yx_n + (v0 + 4 * g) % yx_n;
    astep = (int64_t)kWrWarps * RPW * yx_n;
  }

  if (nrows <= 0) {  // empty tile: pure zero (or `add`) stream
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    if (4 * g < nv)
      for (int row = row0; row < c; row += kWrWarps * RPW, o += step) {
        st_stream(reinterpret_cast<float4*>(o),
                  ap ? __ldg(reinterpret_cast<const float4*>(ap)) : z);
        if (ap) ap += astep;
      }
    return;
  }
  // rows of this tile's intervals: contiguous in V, copied asynchronously,
  // one warp per row
  {
    const float4* src = reinterpret_cast<const float4*>(V) + (int64_t)i0 * c4;
    for (int r = warp; r < nrows; r += kWrWarps)
      for (int v = lane; v < c4; v += kWarp)
        cp_async16(smem_u32(rows + (size_t)r * pitch + 4 * v),
                   src + (size_t)r * c4 + v);
  }
  for (int q = tid; q < T; q += kWrThreads) slot[q] = T;
  for (int q = tid; q < pitch; q += kWrThreads) rows[(size_t)T * pitch + q] = 0.f;
  __syncthreads();
  const int64_t rank0 = (int64_t)b * zyx + v0;
  int any_carry = 0;
  for (int r = tid; r < nrows; r += kWrThreads) {
    const int64_t vl = (int64_t)__ldg(seg_rank + i0 + r) - rank0;
    if (vl >= 0 && vl < nv) slot[vl] = r;
    const int st = __ldg(interval_starts + i0 + r);
    const int ln = __ldg(interval_lengths + i0 + r);
    const int lo = st / kPtsPerWarp;
    const int nx = (st + ln - 1) / kPtsPerWarp - lo;  // carry rows to add
    carry_lo[r] = lo;
    carry_n[r] = nx;
    any_carry |= nx > 0;
  }
  cp_async_commit();
  cp_async_wait0();
  if (__syncthreads_or(any_carry)) {
    // add the carry rows of intervals that span several K1 slices, in slice
    // order (deterministic); one warp per row, 8 loads in flight per lane
    const float4* X4 = reinterpret_cast<const float4*>(X);
    for (int r = warp; r < nrows; r += kWrWarps) {
      const int nx = carry_n[r];
      if (nx == 0) continue;
      for (int v = lane; v < c4; v += kWarp) {
        float4* dst = reinterpret_cast<float4*>(rows + (size_t)r * pitch + 4 * v);
        float4 a = *dst;
        const float4* src = X4 + (int64_t)(carry_lo[r] + 1) * c4 + v;
        for (int k = 0; k < nx; k += 8) {
          float4 t[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            t[j] = (k + j < nx) ? __ldcg(src + (int64_t)(k + j) * c4)
                                : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (k + j < nx) {
              a.x += t[j].x; a.y += t[j].y; a.z += t[j].z; a.w += t[j].w;
            }
          }
        }
        *dst = a;
      }
    }
    __syncthreads();
  }

  if (4 * g < nv) {
    // four consecutive voxels of one channel per lane; an empty voxel reads the
    // zero row, so the loop is branch-free: 4 LDS + 1 STG.128 per 16 bytes
    const int4 s4 = *reinterpret_cast<const int4*>(slot + 4 * g);
    const float* rx = rows + (size_t)s4.x * pitch;
    const float* ry = rows + (size_t)s4.y * pitch;
    const float* rz = rows + (size_t)s4.z * pitch;
    const float* rw = rows + (size_t)s4.w * pitch;
#pragma unroll 5
    for (int row = row0; row < c; row += kWrWarps * RPW, o += step) {
      float4 v;
      v.x = rx[row];
      v.y = ry[row];
      v.z = rz[row];
      v.w = rw[row];
      if (ap) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(ap));
        v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
        ap += astep;
      }
      st_stream(reinterpret_cast<float4*>(o), v);
    }
  }
}

// ------------------------ Z-mean of the pooled volume ----------------------
// lss[b][y*X + x][:] += (1/Z) * (sum of interval i) for every interval: the
// `bev_feat.mean(-1)` FBOCC feeds to the backward projection (fbocc.py:359),
// computed from the ~n_int interval sums instead of the dense volume (one read
// of V instead of one read of B*C*Z*Y*X).  Token-major output (B, Y*X, C): the
// layout the BEV queries use.  One warp per interval; an interval that spans
// several K1 slices adds its carry rows first (as K2 does); red.global.add.v4
// into the zero-filled map (<= Z contributions per element, order not fixed).
__global__ void __launch_bounds__(256) zmean_kernel(
    const float* __restrict__ V, const float* __restrict__ X,
    const int* __restrict__ seg_rank, const int* __restrict__ interval_starts,
    const int* __restrict__ interval_lengths, const int* __restrict__ meta,
    int c, int zyx, int yx_n, float inv_z, float* __restrict__ lss) {
  const int lane = threadIdx.x & 31;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= meta[0]) return;
  const int rank = __ldg(seg_rank + i);
  const int b = rank / zyx, yx = (rank - b * zyx) % yx_n;
  const int st = __ldg(interval_starts + i), ln = __ldg(interval_lengths + i);
  const int lo = st / kPtsPerWarp;
  const int nx = (st + ln - 1) / kPtsPerWarp - lo;
  const int c4 = c >> 2;
  const float4* V4 = reinterpret_cast<const float4*>(V) + i * c4;
  const float4* X4 = reinterpret_cast<const float4*>(X) + (int64_t)(lo + 1) * c4;
  float4* dst = reinterpret_cast<float4*>(lss) + ((int64_t)b * yx_n + yx) * c4;
  for (int v = lane; v < c4; v += kWarp) {
    float4 a = __ldg(V4 + v);
    for (int k = 0; k < nx; ++k) {
      const float4 t = __ldg(X4 + (int64_t)k * c4 + v);
      a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
    }
    a.x *= inv_z; a.y *= inv_z; a.z *= inv_z; a.w *= inv_z;
    atomicAdd(dst + v, a);
  }
}

static inline size_t write_smem_bytes(int T, int c) {
  return (size_t)(T + 1) * (c + 4) * 4 + (size_t)3 * T * 4;
}

// FBBEV_POOL_TILE overrides the tile size (32 / 64 / 128 voxels) for tuning.
static int split_pick_tile(int c) {
  static const char* env = getenv("FBBEV_POOL_TILE");
  if (env) {
    const int t = atoi(env);
    if (t == 32 || t == 64 || t == 128) return t;
  }
  // measured on B200 (DESIGN.md section 5): 128-voxel tiles while five or more
  // CTAs fit an SM (C <= 64), 64-voxel tiles above (C = 80: 9 CTAs of 128
  // threads instead of 5 of 256, 3-5 % faster), 32 for very wide C
  if (write_smem_bytes(128, c) <= 40 * 1024) return 128;
  if (write_smem_bytes(64, c) <= 45 * 1024) return 64;
  return 32;
}

bool split_supported(int c, int64_t zyx) {
  return c % 4 == 0 && zyx % 4 == 0 && zyx < (1ll << 31) && c >= 4 &&
         c <= 1024 &&
         write_smem_bytes(32, c) <= 200 * 1024;
}

static inline size_t up256(size_t x) { return (x + 255) & ~(size_t)255; }

struct SplitWs {
  int* tile_first;
  int* seg_rank;
  int* warp_first;
  int* meta;
  float* V;    // [n_intervals_max][c]  interval sums
  float* X;    // [n_warps_max][c]      carry rows of producer slices
  int n_warps_max, n_sum_ctas;
  size_t bytes;
};

static SplitWs split_layout(void* ws, int batch, int64_t zyx,
                            int n_intervals_max, int n_points_max, int c) {
  const int64_t tiles = (int64_t)batch * ceil_div64(zyx, 32);
  char* p = static_cast<char*>(ws);
  SplitWs w;
  size_t off = 0;
  w.tile_first = reinterpret_cast<int*>(p + off);
  off += up256((size_t)(tiles + 1) * 4);
  w.seg_rank = reinterpret_cast<int*>(p + off);
  off += up256((size_t)std::max(n_intervals_max, 1) * 4);
  w.n_warps_max = (int)ceil_div64(std::max(n_points_max, 1), kPtsPerWarp);
  w.n_sum_ctas = (int)ceil_div64(w.n_warps_max, kSumThreads / kWarp);
  w.warp_first = reinterpret_cast<int*>(p + off);
  off += up256((size_t)(w.n_warps_max + 1) * 4);
  w.meta = reinterpret_cast<int*>(p + off);
  off += 256;
  w.V = reinterpret_cast<float*>(p + off);
  off += up256((size_t)std::max(n_intervals_max, 1) * c * 4);
  w.X = reinterpret_cast<float*>(p + off);
  off += up256((size_t)w.n_warps_max * c * 4);
  w.bytes = off;
  return w;
}

size_t split_workspace_bytes(int batch, int64_t zyx, int n_intervals_max,
                             int n_points_max, int c) {
  return split_layout(nullptr, batch, zyx, n_intervals_max, n_points_max, c)
      .bytes;
}

SplitPlanPtrs split_plan_ptrs(void* workspace, int batch, int64_t zyx,
                              int n_intervals_max, int n_points_max, int c) {
  const SplitWs w =
      split_layout(workspace, batch, zyx, n_intervals_max, n_points_max, c);
  SplitPlanPtrs p;
  p.tile_first = w.tile_first; p.seg_rank = w.seg_rank;
  p.warp_first = w.warp_first; p.meta = w.meta;
  p.T = split_pick_tile(c);
  p.tiles_per_b = (int)ceil_div64(zyx, p.T);
  p.n_tiles = (int64_t)batch * p.tiles_per_b;
  p.n_warps_max = w.n_warps_max;
  return p;
}

int split_plan(const int* ranks_bev, const int* interval_starts,
               const int* interval_lengths, int n_intervals_max,
               const int* n_intervals_dev, int n_points_max, int c, int batch,
               int64_t zyx, void* workspace, cudaStream_t st) {
  const SplitWs w =
      split_layout(workspace, batch, zyx, n_intervals_max, n_points_max, c);
  const int T = split_pick_tile(c);
  const int tiles_per_b = (int)ceil_div64(zyx, T);
  const int64_t n_tiles = (int64_t)batch * tiles_per_b;
  const int threads = 256;
  const int64_t work = n_intervals_max > 0
                           ? std::max<int64_t>(n_intervals_max, w.n_warps_max + 1)
                           : n_tiles + 1;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div64(work, threads),
                                                    (int64_t)1 << 20);
  count_launch();
  split_plan_kernel<<<grid, threads, 0, st>>>(
      ranks_bev, interval_starts, interval_lengths, n_intervals_max,
      n_intervals_dev, w.n_warps_max, zyx, tiles_per_b, T, n_tiles,
      w.tile_first, w.seg_rank, w.warp_first, w.meta);
  return launch_status();
}

template <int T>
static int launch_write(const SplitWs& w, const int* interval_starts,
                        const int* interval_lengths, int c, int64_t zyx,
                        int tiles_per_b, int batch, const float* add, int yx_n,
                        float* out, cudaStream_t st, int part = 0) {
  const size_t smem = write_smem_bytes(T, c);
  auto k = dense_write_kernel<T>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(
        k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  k<<<dim3((unsigned)tiles_per_b, (unsigned)batch), 2 * T, smem, st>>>(
      w.V, w.X, w.tile_first, w.seg_rank, interval_starts, interval_lengths, c,
      (int)zyx, add, yx_n, out, part);
  return launch_status();
}

static int launch_write_any(int T, const SplitWs& w, const int* interval_starts,
                            const int* interval_lengths, int c, int64_t zyx,
                            int tiles_per_b, int batch, const float* add,
                            int yx_n, float* out, cudaStream_t st, int part) {
  switch (T) {
    case 128:
      return launch_write<128>(w, interval_starts, interval_lengths, c, zyx,
                               tiles_per_b, batch, add, yx_n, out, st, part);
    case 64:
      return launch_write<64>(w, interval_starts, interval_lengths, c, zyx,
                              tiles_per_b, batch, add, yx_n, out, st, part);
    default:
      return launch_write<32>(w, interval_starts, interval_lengths, c, zyx,
                              tiles_per_b, batch, add, yx_n, out, st, part);
  }
}

// Side stream for the zero stream of the empty tiles (one per host thread,
// created on first use -- warm up once before capturing a CUDA graph).
struct PoolSide {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  int device = -1;
};
static PoolSide* pool_side() {
  static thread_local PoolSide s;
  int dev = 0;
  cudaGetDevice(&dev);
  if (s.stream && s.device == dev) return &s;
  if (s.stream) return nullptr;   // another device on this thread: no overlap
  if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) {
    s.stream = nullptr;
    cudaGetLastError();
    return nullptr;
  }
  s.device = dev;
  return &s;
}

int split_launch(const float* depth, const float* feat, const int* ranks_depth,
                 const int* ranks_feat, const int* ranks_bev,
                 const int* interval_starts, const int* interval_lengths,
                 int n_intervals_max, int n_points_max, int c, int batch,
                 int64_t zyx, float* out, void* workspace, cudaStream_t st,
                 int stages, const float* add, int yx_n) {
  const bool do_sums = (stages & kSplitSums) != 0;
  const bool do_write = (stages & kSplitWrite) != 0;
  if (do_write && (reinterpret_cast<uintptr_t>(out) & 15))
    return FBBEV_ERR_INVALID_ARGUMENT;
  if (add && ((reinterpret_cast<uintptr_t>(add) & 15) || yx_n <= 0 ||
              yx_n % 4 || zyx % yx_n))
    return FBBEV_ERR_INVALID_ARGUMENT;
  const SplitWs w =
      split_layout(workspace, batch, zyx, n_intervals_max, n_points_max, c);
  const int T = split_pick_tile(c);
  const int tiles_per_b = (int)ceil_div64(zyx, T);
  // One-shot op (sums + write): the empty tiles' zero stream -- 79 % of the
  // 200x200x16 volume -- depends on the plan only, so it is launched on a side
  // stream beside the interval sums (latency-bound, 18 us, few bytes) and the
  // tiles that hold intervals follow the sums (FBBEV_POOL_OVERLAP=0: serial).
  static const bool overlap_on = [] {
    const char* e = getenv("FBBEV_POOL_OVERLAP");
    return !(e && e[0] == '0');
  }();
  PoolSide* side = (do_sums && do_write && n_intervals_max > 0 && overlap_on)
                       ? pool_side() : nullptr;
  if (side) {
    if (cudaEventRecord(side->fork, st) != cudaSuccess ||
        cudaStreamWaitEvent(side->stream, side->fork, 0) != cudaSuccess) {
      cudaGetLastError();
      side = nullptr;
    }
  }
  if (do_sums && n_intervals_max > 0) {
    count_launch();
    const unsigned grid = (unsigned)w.n_sum_ctas;
    const int c4 = c / 4;
#define FBBEV_SUM_CASE(LGV, VPLV)                                             \
  interval_sums_kernel<LGV, VPLV><<<grid, kSumThreads, 0, st>>>(              \
      depth, feat, ranks_depth, ranks_feat, ranks_bev, interval_starts,       \
      w.warp_first, w.meta, c, w.V, w.X)
    // group width LG and float4 columns per lane VPL with LG * VPL >= C / 4
    if (c4 <= 4) FBBEV_SUM_CASE(4, 1);
    else if (c4 <= 8) FBBEV_SUM_CASE(4, 2);
    else if (c4 <= 16) FBBEV_SUM_CASE(4, 4);
    else if (c4 <= 20) FBBEV_SUM_CASE(4, 5);
    else if (c4 <= 32) FBBEV_SUM_CASE(4, 8);
    else if (c4 <= 64) FBBEV_SUM_CASE(8, 8);
    else if (c4 <= 128) FBBEV_SUM_CASE(16, 8);
    else FBBEV_SUM_CASE(32, 8);
#undef FBBEV_SUM_CASE
    int rc = launch_status();
    if (rc) return rc;
  }
  if (side) {   // after the sums: their CTAs take their SM slots first
    count_launch();
    int rc = launch_write_any(T, w, interval_starts, interval_lengths, c, zyx,
                              tiles_per_b, batch, add, yx_n, out, side->stream, 1);
    if (rc) return rc;
  }
  if (!do_write) return FBBEV_OK;
  count_launch();
  int rc = launch_write_any(T, w, interval_starts, interval_lengths, c, zyx,
                            tiles_per_b, batch, add, yx_n, out, st, side ? 2 : 0);
  if (side) {
    if (cudaEventRecord(side->join, side->stream) != cudaSuccess ||
        cudaStreamWaitEvent(st, side->join, 0) != cudaSuccess)
      return (int)cudaGetLastError();
  }
  return rc;
}

int split_zmean(const int* interval_starts, const int* interval_lengths,
                int n_intervals_max, int n_points_max, int c, int batch,
                int64_t zyx, int yx_n, float* lss, void* workspace,
                cudaStream_t st) {
  if (yx_n <= 0 || zyx % yx_n || (reinterpret_cast<uintptr_t>(lss) & 15))
    return FBBEV_ERR_INVALID_ARGUMENT;
  const SplitWs w =
      split_layout(workspace, batch, zyx, n_intervals_max, n_points_max, c);
  cudaError_t e =
      cudaMemsetAsync(lss, 0, (size_t)batch * yx_n * c * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  count_launch();
  if (n_intervals_max <= 0) return FBBEV_OK;
  const float inv_z = 1.0f / (float)(zyx / yx_n);
  const unsigned grid = (unsigned)ceil_div64((int64_t)n_intervals_max * 32, 256);
  count_launch();
  zmean_kernel<<<grid, 256, 0, st>>>(w.V, w.X, w.seg_rank, interval_starts,
                                     interval_lengths, w.meta, c, (int)zyx, yx_n,
                                     inv_z, lss);
  return launch_status();
}

}  // namespace fbbev

#ifdef POOL_TRACE
FBBEV_API int fbbev_debug_pool_trace(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, fbbev::g_pool_trace,
                                   sizeof(long long) * 32);
}
#endif
