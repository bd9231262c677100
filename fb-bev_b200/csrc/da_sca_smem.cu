// da_sca_smem.cu -- depth-aware spatial cross-attention with the camera's value
// map resident in shared memory (sm_100a).
//
// Same arithmetic and contract as da_sca_fwd_kernel (msda_fwd.cu; reference
// spatial_cross_attention_depth.py:156-216, 540-595).  What changes is where
// the gathers go.  The thread-per-(query, head) kernel loops over cameras per
// query and gathers from global memory: ncu showed it bound by L1 wavefronts
// (one per distinct 128-byte line per load: 2.9 M corner gathers of 40 bytes ->
// 83 us at 200x200 queries, 0.11 of the HBM roofline of its operands).
// Here the roles are swapped:
//
//   * a CTA owns ONE camera of one sample and stages that camera's projected
//     value map -- contiguous n_value x E floats, 225 KB for the 16x44 x 80 map
//     of FB-OCC -- into shared memory with 1-D TMA bulk copies (cp.async.bulk +
//     mbarrier), once;
//   * its warps then walk the BEV queries in batches of 32, keep the ones the
//     camera sees (ballot compaction into a per-warp ring, no block barrier) and
//     process them four at a time: lane = (query slot, head), so the eight
//     heads of a query share the mask / reference-point / depth words
//     (broadcast loads) and the four queries of a warp -- neighbours in the BEV
//     row -- mostly hit the same pixels (shared-memory broadcast);
//   * every gather is an LDS.64 at 128 B/clk/SM; with E = 80 the head chunks of
//     one pixel fall into disjoint banks (10 m mod 32 distinct for m = 0..7, and
//     odd / even pixels are 16 banks apart), so a warp's load is conflict-free
//     unless two of its queries hit different pixels of the same parity;
//   * CTAs are shared out over the (sample, camera) pairs in proportion to the
//     number of queries each camera sees (counted on the device by the
//     prologue kernel, which also zero-fills the output), each CTA taking an
//     interleaved subset of the 32-query batches: balanced without any host
//     synchronisation;
//   * a query seen by several cameras receives one contribution per camera:
//     red.global.add.v2.f32 of acc / count into the zero-filled output (the
//     reference forms (sum of cameras) / count; the two differ by one rounding).
//
// Used when the whole map fits (n_value * E * 4 <= ~220 KB) for the head layout
// the bank analysis holds for (8 heads x 10 channels, 1 level, 8 points, 4
// anchors); every other shape keeps the global-memory kernel.
#include <stdlib.h>

#include "bulk.cuh"
#include "common.cuh"
#include "da_sca_smem.h"
#include "msda_common.cuh"

namespace fbbev {

constexpr int kScaMaxWarps = 24;
constexpr int kRoundBatches = 64;   // 32-query batches scanned per round
constexpr int kListCap = kRoundBatches * 32;   // visible-query codes (uint16)
constexpr int kListBytes = kListCap * 2;
constexpr int kCH = 10, kHeads = 8, kE = 80, kZ = 4, kPts = 8;

struct ScaSmemParams {
  const float *value, *depth_prob, *ref_cam, *ref_depth, *offsets, *logits;
  const uint32_t* mask32;  // (n_cams, bs, nq) words of 4 mask bytes (Z = 4)
  const int* counts;       // [bs * n_cams][kCountChunks] partial counts of the
                           // queries each (sample, camera) pair sees
  const int64_t* shapes;   // device (levels, 2) = [[H, W]]
  float* out;
  float d_min, d_step;
  int bs, n_cams, nq, n_value, DC, n_pairs;
};

// ---- prologue: per-(sample, camera) visible-query counts + zero-fill --------
// Blocks [0, n_pairs * kCountChunks) each count one chunk of one pair's mask
// words into partial[pair][chunk] (plain stores: no atomics, nothing to
// pre-zero); the remaining blocks zero-fill the output.
constexpr int kCountChunks = 16;

__global__ void __launch_bounds__(256) da_sca_prologue_kernel(
    const uint32_t* __restrict__ mask32, int bs, int n_cams, int nq,
    int* __restrict__ partial, float4* __restrict__ out4, int64_t n_out4) {
  const int n_count = bs * n_cams * kCountChunks;
  if ((int)blockIdx.x < n_count) {
    // pair index in the kernel's (b, n) order; mask is laid out (n, b, q)
    const int pair = blockIdx.x / kCountChunks, chunk = blockIdx.x % kCountChunks;
    const int b = pair / n_cams, n = pair % n_cams;
    const uint32_t* m = mask32 + ((int64_t)n * bs + b) * nq;
    const int per = (nq + kCountChunks - 1) / kCountChunks;
    const int q0 = chunk * per, q1 = min(nq, q0 + per);
    int c = 0;
    for (int q = q0 + threadIdx.x; q < q1; q += blockDim.x) c += __ldg(m + q) != 0;
    __shared__ int red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFull, c, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int i = 0; i < 8; ++i) t += red[i];
      partial[blockIdx.x] = t;
    }
    return;
  }
  const int64_t stride = (int64_t)(gridDim.x - n_count) * blockDim.x;
  for (int64_t i = (int64_t)(blockIdx.x - n_count) * blockDim.x + threadIdx.x;
       i < n_out4; i += stride)
    out4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// acc[0..10) += wgt * bilinear(map, h_im, w_im); `map` points at channel 0 of
// the lane's head in pixel 0 of the value map ([pixel][80] floats) -- the
// shared-memory copy (SMEM, LDS.64) or, while the bulk copies are still in
// flight, the global original (LDG.64)
template <bool SMEM>
__device__ __forceinline__ float2 ld2(const float* p) {
  if (SMEM) {
    float2 v;
    asm("ld.shared.v2.f32 {%0, %1}, [%2];"
        : "=f"(v.x), "=f"(v.y)
        : "r"(smem_u32(p)));
    return v;
  }
  return __ldg(reinterpret_cast<const float2*>(p));
}

template <bool SMEM>
__device__ __forceinline__ void sample_map(const float* map, int H, int W,
                                           float h_im, float w_im, float wgt,
                                           float (&acc)[kCH]) {
  if (!(h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W))
    return;
  const int h_low = (int)floorf(h_im), w_low = (int)floorf(w_im);
  const float lh = h_im - (float)h_low, lw = w_im - (float)w_low;
  const float hh = 1.f - lh, hw = 1.f - lw;
  const bool t = h_low >= 0, btm = h_low + 1 <= H - 1;
  const bool l = w_low >= 0, r = w_low + 1 <= W - 1;
  // absent corners weigh 0 and read the (always valid) clamped address instead
  // of branching
  const float w1 = (t && l) ? hh * hw : 0.f, w2 = (t && r) ? hh * lw : 0.f;
  const float w3 = (btm && l) ? lh * hw : 0.f, w4 = (btm && r) ? lh * lw : 0.f;
  const int h0 = max(h_low, 0), h1 = min(h_low + 1, H - 1);
  const int x0 = max(w_low, 0), x1 = min(w_low + 1, W - 1);
  const float* p1 = map + (h0 * W + x0) * kE;
  const float* p2 = map + (h0 * W + x1) * kE;
  const float* p3 = map + (h1 * W + x0) * kE;
  const float* p4 = map + (h1 * W + x1) * kE;
#pragma unroll
  for (int c = 0; c < kCH / 2; ++c) {
    const float2 v1 = ld2<SMEM>(p1 + 2 * c), v2 = ld2<SMEM>(p2 + 2 * c);
    const float2 v3 = ld2<SMEM>(p3 + 2 * c), v4 = ld2<SMEM>(p4 + 2 * c);
    // same association as sample_accum: (w1 v1 + w2 v2 + w3 v3 + w4 v4) * wgt
    const float sx = w1 * v1.x + w2 * v2.x + w3 * v3.x + w4 * v4.x;
    const float sy = w1 * v1.y + w2 * v2.y + w3 * v3.y + w4 * v4.y;
    acc[2 * c] += sx * wgt;
    acc[2 * c + 1] += sy * wgt;
  }
}

// One pass of a warp: up to four queries (lane = (slot, head)) of camera `n` of
// sample `b`, sampled from the shared-memory map and added to the output.
struct ScaCtx {
  const float* tile;      // shared-memory value map of the CTA's camera
  const float* gmap;      // the same map in global memory
  const float* dp;        // depth_prob of the camera
  const uint32_t* bar;    // (address of) the TMA barrier, as a shared address
  int64_t rbase_pair;     // (n * bs + b) * nq
  int b, H, W;
  float inv_W, inv_H;
};

__device__ __forceinline__ void sca_pass(const ScaSmemParams& P, const ScaCtx& C,
                                         int q, bool active, int lane,
                                         bool& tile_ready) {
  const int slot = lane >> 3, m = lane & 7;
  const int64_t bq = (int64_t)C.b * P.nq + q;
  // cameras that see this query (:213-216): lane m asks for camera m
  const bool cam_sees =
      active && m < P.n_cams &&
      (__ldg(P.mask32 + ((int64_t)m * P.bs + C.b) * P.nq + q) & 0x01010101u) != 0;
  const unsigned cb = __ballot_sync(kFull, cam_sees);
  const float cnt = (float)max(1, __popc((cb >> (slot * 8)) & 0xffu));

  float acc[kCH];
#pragma unroll
  for (int c = 0; c < kCH; ++c) acc[c] = 0.f;
  float2 rxy[kZ];
  float w[kPts];
  float4 off4[4];
  float dwz = 0.f;
  if (active) {
    const int64_t rb = (C.rbase_pair + q) * kZ;
    const float4* r4 = reinterpret_cast<const float4*>(P.ref_cam + rb * 2);
    const float4 ra = __ldg(r4), rbv = __ldg(r4 + 1);
    rxy[0] = make_float2(ra.x, ra.y); rxy[1] = make_float2(ra.z, ra.w);
    rxy[2] = make_float2(rbv.x, rbv.y); rxy[3] = make_float2(rbv.z, rbv.w);
    const float4* l4 = reinterpret_cast<const float4*>(
        P.logits + (bq * kHeads + m) * kPts);
    const float4 la = __ldg(l4), lb = __ldg(l4 + 1);
    const float4* o4 = reinterpret_cast<const float4*>(
        P.offsets + (bq * kHeads + m) * kPts * 2);
#pragma unroll
    for (int i = 0; i < 4; ++i) off4[i] = __ldg(o4 + i);
    // depth weight of anchor z = m & 3, shared out below (:196-199, :584-591)
    const int z = m & 3;
    const float d = __ldg(P.ref_depth + rb + z);
    float fb = floorf(__fdiv_rn(__fsub_rn(d, P.d_min), P.d_step));
    fb = fminf(fmaxf(fb, 0.f), (float)(P.DC - 1));
    const float2 rz = z == 0 ? rxy[0] : z == 1 ? rxy[1] : z == 2 ? rxy[2]
                                                                 : rxy[3];
    dwz = sample_scalar(C.dp + (int)fb, C.H, C.W, P.DC, pix(rz.y, C.H),
                        pix(rz.x, C.W));
    // softmax over the head's 8 logits (:540)
    w[0] = la.x; w[1] = la.y; w[2] = la.z; w[3] = la.w;
    w[4] = lb.x; w[5] = lb.y; w[6] = lb.z; w[7] = lb.w;
    float mx = w[0];
#pragma unroll
    for (int p = 1; p < kPts; ++p) mx = fmaxf(mx, w[p]);
    float s = 0.f;
#pragma unroll
    for (int p = 0; p < kPts; ++p) {
      w[p] = __expf(w[p] - mx);
      s += w[p];
    }
    const float inv = __fdividef(1.f, s);
#pragma unroll
    for (int p = 0; p < kPts; ++p) w[p] *= inv;
  }
  float dw[kZ];
#pragma unroll
  for (int z = 0; z < kZ; ++z) dw[z] = __shfl_sync(kFull, dwz, (lane & ~7) | z);
  // the staged map is used as soon as its bulk copies have landed; until then
  // (the first ~10 us of the CTA) the same gathers go to the global original
  if (!tile_ready) tile_ready = mbar_test(smem_u32(C.bar), 0);
  if (active) {
#pragma unroll
    for (int p = 0; p < kPts; ++p) {          // point index = pp * Z + z (:563-570)
      const int z = p & (kZ - 1);
      const float ox = (p & 1) ? off4[p >> 1].z : off4[p >> 1].x;
      const float oy = (p & 1) ? off4[p >> 1].w : off4[p >> 1].y;
      // offsets / (W, H) as a multiplication by the reciprocal (<= 1 ulp from
      // the reference's division; the sampled value is continuous in it)
      const float lx = rxy[z].x + ox * C.inv_W;
      const float ly = rxy[z].y + oy * C.inv_H;
      // attention weight * depth weight, no renormalisation (:592)
      if (tile_ready)
        sample_map<true>(C.tile + m * kCH, C.H, C.W, pix(ly, C.H), pix(lx, C.W),
                         w[p] * dw[z], acc);
      else
        sample_map<false>(C.gmap + m * kCH, C.H, C.W, pix(ly, C.H),
                          pix(lx, C.W), w[p] * dw[z], acc);
    }
    float2* o = reinterpret_cast<float2*>(P.out + bq * kE + m * kCH);
    const float inv_cnt = 1.f / cnt;   // exact for 1, 2, 4 cameras
#pragma unroll
    for (int c = 0; c < kCH / 2; ++c)
      atomicAdd(o + c, make_float2(acc[2 * c] * inv_cnt,
                                   acc[2 * c + 1] * inv_cnt));
  }
}

template <int kScaThreads>
__global__ void __launch_bounds__(kScaThreads, 1) da_sca_smem_kernel(
    ScaSmemParams P) {
  constexpr int kScaWarps = kScaThreads / 32;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* tile = reinterpret_cast<float*>(smem_raw);
  const int tile_bytes = P.n_value * kE * 4;
  unsigned char* ring = smem_raw + tile_bytes;               // the CTA's list
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + tile_bytes +
                                              kListBytes);
  __shared__ int s_pair, s_k, s_K, s_next, s_left_n;
  __shared__ int s_left[4];
  __shared__ int s_cnt[64];   // per-pair counts (chunked when n_pairs > 64)
  __shared__ long long s_total;

  // ---- which (sample, camera) pair, and which share of it, is this CTA's ----
  // pair i gets K_i = 1 + floor(spare * count_i / total) CTAs
  const long long spare = (long long)gridDim.x - P.n_pairs;
  if (threadIdx.x == 0) {
    s_total = 0; s_next = 0; s_left_n = 0; s_pair = -1;
    mbar_init(smem_u32(bar), 1);
    fence_mbar_init();
  }
  __syncthreads();
  {  // total of all partial counts
    long long t = 0;
    for (int i = threadIdx.x; i < P.n_pairs * kCountChunks; i += kScaThreads)
      t += P.counts[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(kFull, t, o);
    if ((threadIdx.x & 31) == 0 && t) atomicAdd((unsigned long long*)&s_total,
                                                (unsigned long long)t);
  }
  __syncthreads();
  const long long total = s_total;
  int my_count = 0;
  for (int base = 0, cum = 0; base < P.n_pairs && s_pair < 0; base += 64) {
    const int n_here = min(64, P.n_pairs - base);
    if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n_here * kCountChunks; i += kScaThreads)
      atomicAdd(&s_cnt[i / kCountChunks], P.counts[base * kCountChunks + i]);
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 0; i < n_here; ++i) {
        const int Ki =
            1 + (total > 0 ? (int)(spare * s_cnt[i] / total) : 0);
        if ((int)blockIdx.x < cum + Ki) {
          s_pair = base + i; s_k = blockIdx.x - cum; s_K = Ki;
          s_left[0] = s_cnt[i];
          break;
        }
        cum += Ki;
      }
      if (s_pair < 0) s_left[1] = cum;
    }
    __syncthreads();
    if (s_pair < 0) cum = s_left[1];
    else my_count = s_left[0];
    __syncthreads();
  }
  const int pair = s_pair;
  if (pair < 0 || my_count == 0) return;      // spare CTA / camera sees nothing
  const int b = pair / P.n_cams, n = pair % P.n_cams;
  const int bn = pair;                        // value / depth are (b, n) major

  if (threadIdx.x == 0) {
    const uint32_t barrier = smem_u32(bar);
    mbar_arrive_expect_tx(barrier, (uint32_t)tile_bytes);
    const char* src = reinterpret_cast<const char*>(
        P.value + (int64_t)bn * P.n_value * kE);
    const uint32_t dst = smem_u32(tile);
    // the K CTAs of a camera all pull the same 225 KB: start each one at a
    // different chunk so that they do not queue on the same L2 lines
    constexpr int kChunk = 8192;
    const int n_chunks = (tile_bytes + kChunk - 1) / kChunk;
    const int start = (int)(((long long)s_k * n_chunks) / max(s_K, 1));
    for (int c = 0; c < n_chunks; ++c) {
      const int off = ((start + c) % n_chunks) * kChunk;
      const int nb = min(kChunk, tile_bytes - off);
      bulk_g2s(dst + off, src + off, (uint32_t)nb, barrier);
    }
  }

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = lane >> 3;
  uint16_t* list = reinterpret_cast<uint16_t*>(ring);   // [kListCap] codes
  const uint32_t* mask_pair = P.mask32 + ((int64_t)n * P.bs + b) * P.nq;
  ScaCtx C;
  C.tile = tile;
  C.gmap = P.value + (int64_t)bn * P.n_value * kE;
  C.H = (int)__ldg(P.shapes); C.W = (int)__ldg(P.shapes + 1);
  C.dp = P.depth_prob + (int64_t)bn * C.H * C.W * P.DC;
  C.bar = reinterpret_cast<const uint32_t*>(bar);
  C.rbase_pair = ((int64_t)n * P.bs + b) * P.nq;
  C.b = b;
  C.inv_W = 1.f / (float)C.W; C.inv_H = 1.f / (float)C.H;
  const int n_batches = (P.nq + 31) / 32;
  const int k = s_k, K = s_K;
  bool tile_ready = false;

  // CTA k of the pair owns the 32-query batches j = k (mod K) -- interleaved,
  // so every CTA samples the camera's visible wedge evenly.  Per round of up
  // to kRoundBatches batches: (A) the warps scan the batches and compact the
  // visible queries into ONE list for the CTA (16-bit codes: batch-in-round,
  // lane); (B) the warps pull groups of four queries from that list through a
  // shared counter.  The unit of scheduling is a pass, so the tail of a CTA is
  // at most one pass per warp (a whole batch of up to eight passes before:
  // 28 % of the warp time was spent waiting at the final barrier).
  for (int round = 0; k + (int64_t)round * K < n_batches;
       round += kRoundBatches) {
    if (threadIdx.x == 0) { s_next = 0; s_left_n = 0; }
    __syncthreads();
    for (int jl = warp; jl < kRoundBatches; jl += kScaWarps) {
      const int64_t j = k + (int64_t)(round + jl) * K;
      if (j >= n_batches) break;
      const int q = (int)j * 32 + lane;
      const bool seen = q < P.nq && __ldg(mask_pair + q) != 0;      // (:165)
      const unsigned bal = __ballot_sync(kFull, seen);
      int base = 0;
      if (lane == 0 && bal) base = atomicAdd(&s_left_n, __popc(bal));
      base = __shfl_sync(kFull, base, 0);
      if (seen)
        list[base + __popc(bal & ((1u << lane) - 1))] =
            (uint16_t)((jl << 5) | lane);
    }
    __syncthreads();
    const int n_vis = s_left_n;
    for (;;) {
      int p0 = 0;
      if (lane == 0) p0 = atomicAdd(&s_next, 4);
      p0 = __shfl_sync(kFull, p0, 0);
      if (p0 >= n_vis) break;
      const bool active = p0 + slot < n_vis;
      const int code = active ? (int)list[p0 + slot] : 0;
      const int q = (int)((k + (int64_t)(round + (code >> 5)) * K) * 32) +
                    (code & 31);
      sca_pass(P, C, q, active, lane, tile_ready);
    }
    __syncthreads();   // the list is rewritten by the next round
  }
  // the bulk copies must have landed before the CTA (and its shared memory)
  // goes away, also when this warp never touched the tile
  if (!tile_ready) mbar_wait(smem_u32(bar), 0);
}

size_t da_sca_smem_workspace_bytes(int bs, int n_cams) {
  return (size_t)bs * n_cams * kCountChunks * sizeof(int);
}

bool da_sca_smem_eligible(int n_cams, int n_value, int heads, int ch, int levels,
                          int points, int Z) {
  const size_t smem = (size_t)n_value * kE * 4 + kListBytes + 64;
  return heads == kHeads && ch == kCH && levels == 1 && points == kPts &&
         Z == kZ && n_cams <= 8 && smem <= 232448 - 1024 - 768;
}

int da_sca_smem_launch(const float* value, const float* depth_prob,
                       const float* ref_cam, const float* ref_depth,
                       const uint8_t* mask, const float* offsets,
                       const float* logits, const int64_t* shapes, float d_min,
                       float d_step, int bs, int n_cams, int nq, int n_value,
                       int DC, float* out, void* workspace, cudaStream_t st,
                       int stages) {
  ScaSmemParams P;
  P.value = value; P.depth_prob = depth_prob; P.ref_cam = ref_cam;
  P.ref_depth = ref_depth; P.offsets = offsets; P.logits = logits;
  P.mask32 = reinterpret_cast<const uint32_t*>(mask);
  P.counts = static_cast<const int*>(workspace);
  P.shapes = shapes;
  P.out = out;
  P.d_min = d_min; P.d_step = d_step;
  P.bs = bs; P.n_cams = n_cams; P.nq = nq; P.n_value = n_value;
  P.DC = DC; P.n_pairs = bs * n_cams;

  const int n_sm = sm_count();
  const int64_t n_out4 = (int64_t)bs * nq * kE / 4;
  const int zero_blocks = (int)std::min<int64_t>(ceil_div64(n_out4, 256 * 4),
                                                 (int64_t)n_sm * 16);
  if (stages & kScaPrologue) {
    count_launch();
    da_sca_prologue_kernel<<<P.n_pairs * kCountChunks + zero_blocks, 256, 0,
                             st>>>(P.mask32, bs, n_cams, nq,
                                   static_cast<int*>(workspace),
                                   reinterpret_cast<float4*>(out), n_out4);
    if (!(stages & kScaMain)) return launch_status();
  }
  count_launch();
  // 512 or 640 threads per CTA (FBBEV_SCA_THREADS: tuning aid)
  static int threads = 0;
  if (threads == 0) {
    const char* e = getenv("FBBEV_SCA_THREADS");
    threads = (e && atoi(e) == 640) ? 640 : 512;
    cudaFuncSetAttribute(da_sca_smem_kernel<512>,
                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                         232448 - 1024 - 768);
    cudaFuncSetAttribute(da_sca_smem_kernel<640>,
                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                         232448 - 1024 - 768);
  }
  const size_t smem = (size_t)n_value * kE * 4 + kListBytes + 64;
  // one CTA per SM; more waves when there are many (sample, camera) pairs so
  // that each pair still splits into several CTAs
  const int waves = std::max(1, (4 * P.n_pairs + n_sm - 1) / n_sm);
  if (threads == 640)
    da_sca_smem_kernel<640><<<n_sm * waves, 640, smem, st>>>(P);
  else
    da_sca_smem_kernel<512><<<n_sm * waves, 512, smem, st>>>(P);
  return launch_status();
}

}  // namespace fbbev
