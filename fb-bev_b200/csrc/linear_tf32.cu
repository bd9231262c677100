// linear_tf32.cu -- the row-wise Linears of the backward projection on the
// 5th-generation tensor cores (tcgen05, accumulators in TMEM), fp32 in / fp32 out.
//
// What it replaces: every nn.Linear of the BEVFormer encoder layer the reference
// builds for the backward projection -- sampling_offsets / attention_weights /
// value_proj / output_proj of the self- and cross-attention
// (spatial_cross_attention_depth.py:420-427, mmcv MultiScaleDeformableAttention)
// and the FFN (bevformer_encoder.py:251-377 op order) -- together with what
// follows each of them row by row: bias, ReLU, the residual add and the
// LayerNorm(embed_dims).  The reference runs them as cuBLAS fp32 GEMMs plus
// separate elementwise / LayerNorm kernels.
//
// Numerics: the 1e-4 parity bar excludes plain TF32 (10-bit mantissa), so every
// product is formed as 3xTF32:  x = x_hi + x_lo, w = w_hi + w_lo with *_hi the
// upper 19 bits and *_lo the exact fp32 remainder;
//     x.w ~= x_hi.w_hi + x_lo.w_hi + x_hi.w_lo        (error ~2^-21 relative)
// three tcgen05.mma.kind::tf32 per k-step into the same fp32 TMEM accumulator.
//
// Structure (one persistent CTA per SM owning a contiguous range of rows, cut
// into 128-row tiles; 14 warps):
//   warps 4-7   loaders: X rows -> registers (two K-blocks in flight per
//               thread) -> hi / lo split -> shared memory in the UMMA canonical
//               K-major layout (8x16-byte core matrices, no swizzle);
//   warp  13    one lane starts the 1-D bulk copy (TMA) of the pre-packed weight
//               block of a stage as soon as the stage is free;
//   warp  12    one lane issues the MMAs (M=128, N<=192, K=8 per instruction),
//               tcgen05.commit releases the stage / publishes the accumulator;
//   warps 0-3, 8-11  two epilogue groups, one per TMEM accumulator (even / odd
//               tiles): tcgen05.ld (lane == row), bias / ReLU / residual /
//               LayerNorm, rows staged through a shared-memory slab so that
//               global loads and stores are coalesced (optionally two outputs:
//               a column split, for two Linears that share their input).  The
//               epilogue is the longest stage per tile (one warp per scheduler,
//               dependent issue), hence two groups.
//   Ring of K-blocks of 40 floats (5 k-steps) between loaders and MMA, two
//   accumulators in TMEM between MMA and epilogue.
#include "tc5.cuh"

namespace fbbev {

constexpr int kLinThreads = 448;  // 14 warps, see the role table above
constexpr int kMaxN = 192;
constexpr int kSlabPitch = 20;  // floats: 16 columns + 4 (bank spread)
constexpr int kSlabBytes = 2 * kTileM * kSlabPitch * 4;  // both groups
// control area after the stages: mbarriers + TMEM slot (256 B), then bias /
// LayerNorm weight / LayerNorm bias staged once (the L1 left beside ~220 KB of
// shared memory is too small to keep them: a __ldg would be an L2 round trip)
constexpr int kCtrlBytes = 256 + 3 * kMaxN * 4;

// ------------------------------ weight packing -------------------------------
// W [N][K] row-major -> [k-block][hi, lo][chunk 0..9][Npad / 8][8 rows][4]:
// exactly the shared-memory image of one stage, so a stage's weights are one
// contiguous bulk copy.  Rows >= N and columns >= K are zero.
__global__ void linear_pack_kernel(const float* __restrict__ w, int n, int k,
                                   int npad, int n_kb, float* __restrict__ out) {
  const int64_t total = (int64_t)n_kb * kChunks * npad;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(i % npad);
    const int ch = (int)((i / npad) % kChunks);
    const int kb = (int)(i / ((int64_t)npad * kChunks));
    float hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = kb * kKB + ch * 4 + j;
      tf32_split((row < n && col < k) ? w[(int64_t)row * k + col] : 0.f, hi[j], lo[j]);
    }
    const int64_t part = (int64_t)kChunks * npad * 4;  // floats of one hi / lo part
    const int64_t off = (int64_t)kb * 2 * part + kmajor_off(row, ch, npad) / 4;
    *reinterpret_cast<float4*>(out + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<float4*>(out + off + part) =
        make_float4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// -------------------------------- the kernel ---------------------------------
struct LinearParams {
  const float* x;         // [M][K]
  const float* x_add;     // [M][K] or null: the GEMM input is x + x_add
  const float* wp;        // packed weights
  const float* bias;      // [N] or null
  const float* residual;  // [M][N] or null
  const float* gamma;     // LayerNorm weight [N] or null
  const float* beta;      // LayerNorm bias [N] or null
  float* y;               // [M][N]
  int M, K, N, npad, n_kb, relu, rows_per_cta, stages;
  int slab_pitch;  // floats per slab row: 20 (16-column chunks) or N + 4 (whole rows)
  int64_t ldx, ldr, ldy;  // row strides in floats
  int64_t ldxa;           // row stride of x_add
  // optional second output: columns [n_split, N) go to y2 (row stride ldy2)
  float* y2;
  int64_t ldy2;
  int n_split;
  float eps;
};

template <bool LN>
__global__ void __launch_bounds__(kLinThreads, 1)
    linear_tf32_kernel(const LinearParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  TRACE_DECL
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int npad = p.npad, S = p.stages;
  const uint32_t w_part = (uint32_t)npad * kKB * 4;        // bytes of W_hi
  const uint32_t stage_bytes = 2u * kAPart + 2u * w_part;
  unsigned char* ctrl = smem + (size_t)S * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ctrl);
  const uint32_t bar_full = smem_u32(bars);                // [S]
  const uint32_t bar_empty = bar_full + 8u * S;            // [S]
  const uint32_t bar_tfull = bar_empty + 8u * S;           // [2]
  const uint32_t bar_tempty = bar_tfull + 16u;             // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ctrl + 16 * S + 32);
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 12) {
    if (lane == 0) {
      for (int s = 0; s < S; ++s) {
        mbar_init(bar_full + 8u * s, 128 + 1);  // loader threads + expect_tx
        mbar_init(bar_empty + 8u * s, 1);       // tcgen05.commit
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(bar_tfull + 8u * a, 1);       // tcgen05.commit
        mbar_init(bar_tempty + 8u * a, 128);    // epilogue threads
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(smem_u32(tmem_slot));
  }
  float* s_bias = reinterpret_cast<float*>(ctrl + 256);
  float* s_gamma = s_bias + kMaxN;
  float* s_beta = s_gamma + kMaxN;
  for (int j = threadIdx.x; j < kMaxN; j += kLinThreads) {
    s_bias[j] = (p.bias && j < p.N) ? p.bias[j] : 0.f;
    s_gamma[j] = (p.gamma && j < p.N) ? p.gamma[j] : 1.f;
    s_beta[j] = (p.beta && j < p.N) ? p.beta[j] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) TRACE(3, 1);
  // this CTA's rows and 128-row tiles (the last one may be partial)
  const int row_begin = blockIdx.x * p.rows_per_cta;
  const int row_end = min(p.M, row_begin + p.rows_per_cta);
  const int n_my = row_end > row_begin ? (row_end - row_begin + kTileM - 1) / kTileM : 0;

  if (warp >= 4 && warp < 8) {
    // ================================ loaders ================================
    const int lw = warp - 4;
    const int total = n_my * p.n_kb;  // (tile, K-block) items, two per round
    for (int w0 = 0; w0 < total; w0 += 2) {
      float4 v[2][10];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int w = w0 + u;
        const int ti = w / p.n_kb, kb = w - ti * p.n_kb;
        gather_kblock(v[u], p.x, p.ldx, p.x_add, p.ldxa, p.K,
                      row_begin + ti * kTileM, row_end, kb, w < total, lw, lane);
      }
      if (threadIdx.x == 128) TRACE(1, 100 + w0);
      for (int u = 0; u < 2; ++u) {
        const uint32_t it = (uint32_t)(w0 + u);
        if ((int)it >= total) break;
        const uint32_t s = it % S, ph = (it / S) & 1u;
        mbar_wait(bar_empty + 8u * s, ph ^ 1u);
        if (threadIdx.x == 128) TRACE(1, 200 + it);
        store_kblock(smem + (size_t)s * stage_bytes, v[u], lw, lane);
        fence_proxy_async();
        mbar_arrive(bar_full + 8u * s);
        if (threadIdx.x == 128) TRACE(1, 300 + it);
      }
    }
  } else if (warp == 13) {
    // ============================ weight producer ============================
    if (lane == 0) {
      const uint32_t total = (uint32_t)(n_my * p.n_kb);
      for (uint32_t it = 0; it < total; ++it) {
        const uint32_t s = it % S, ph = (it / S) & 1u;
        mbar_wait(bar_empty + 8u * s, ph ^ 1u);
        mbar_arrive_expect_tx(bar_full + 8u * s, 2u * w_part);
        bulk_g2s(smem_base + s * stage_bytes + 2u * kAPart,
                 p.wp + (size_t)(it % p.n_kb) * (2u * w_part / 4u), 2u * w_part,
                 bar_full + 8u * s);
      }
    }
    __syncwarp();
  } else if (warp == 12) {
    // ================================ MMA issue ===============================
    // The whole warp walks the loop (all lanes poll the barriers) and ONE
    // elected lane issues: under a divergent `if (lane == 0)` the compiler
    // wraps every UTCHMMA in an ELECT / BRA.U.ANY serialisation loop (see
    // elect_one(), tc5.cuh) -- ~100 instead of ~52 cycles per MMA.
    const uint32_t idesc = idesc_tf32_m128(npad);
    const uint32_t lbo_b = (uint32_t)npad * 16u;
    uint32_t it = 0, tc = 0;
    for (int ti = 0; ti < n_my; ++ti, ++tc) {
      const uint32_t acc = tc & 1u, aph = (tc >> 1) & 1u;
      mbar_wait(bar_tempty + 8u * acc, aph ^ 1u);
      tc_fence_after();
      const uint32_t d = tmem_base + acc * (uint32_t)npad;
      for (int kb = 0; kb < p.n_kb; ++kb, ++it) {
        const uint32_t s = it % S, ph = (it / S) & 1u;
        mbar_wait(bar_full + 8u * s, ph);
        tc_fence_after();
        if (lane == 0) TRACE(2, 400 + it);
        const uint32_t a_hi = smem_base + s * stage_bytes;
        const uint32_t w_hi = a_hi + 2u * kAPart;
        if (elect_one()) {
          mma_kblock_ss(d, a_hi, w_hi, w_hi + w_part, lbo_b, idesc, kb);
          tc_commit(bar_empty + 8u * s);
          if (kb == p.n_kb - 1) tc_commit(bar_tfull + 8u * acc);
        }
        __syncwarp();
      }
      if (lane == 0) TRACE(2, 500 + tc);
    }
    __syncwarp();
  } else {
    // ================================ epilogue ================================
    // group 0 (warps 0-3) drains accumulator 0 = even tiles of this CTA, group 1
    // (warps 8-11) accumulator 1 = odd tiles; warp % 4 selects the TMEM lanes.
    // tcgen05.ld hands every thread one row, which is the wrong shape for
    // global memory (32 rows per request), so residual and output go through a
    // shared-memory slab per group: whole rows (pitch N + 4) for the LayerNorm
    // epilogue -- the row lives there between the passes, the residual is
    // prefetched into it with cp.async before the accumulator is ready, and the
    // result leaves it fully coalesced -- or 16 columns at a time (pitch 20)
    // otherwise.  Loops are kept rolled on purpose: straight-line code this
    // long ran at ~10 cycles per instruction on instruction fetch alone.
    const int N = p.N;
    const int nc16 = npad >> 4;
    const uint32_t grp = warp >> 3;
    const int q = warp & 3;
    const int gt = q * 32 + lane;  // thread within the group == row of the tile
    const int pitch = p.slab_pitch;
    float* slab = reinterpret_cast<float*>(ctrl + kCtrlBytes) +
                  (size_t)grp * kTileM * pitch;
    float* my_row = slab + (size_t)gt * pitch;
    const float4* bias4 = reinterpret_cast<const float4*>(s_bias);
    const int crow = gt >> 2, cq = gt & 3;  // cooperative mapping: 4 lanes per row
    const int bar_id = 1 + (int)grp;
    auto group_sync = [&]() {
      asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
    };
    uint32_t tc = 0;
    for (int ti = 0; ti < n_my; ++ti, ++tc) {
      if ((tc & 1u) != grp) continue;
      const uint32_t aph = (tc >> 1) & 1u;
      const int row0 = row_begin + ti * kTileM;
      const uint32_t taddr =
          tmem_base + ((uint32_t)(q * 32) << 16) + grp * (uint32_t)npad;
      if (LN) {
        bulk_wait_read0();  // this thread's row of the previous tile has left
        group_sync();       // ... and so have all the others
        if (p.residual)
          prefetch_rows(slab, pitch, p.residual, p.ldr, row0, row_end, row_begin,
                        N, nc16, gt);
        if (gt == 0) TRACE(3 + grp, 600 + tc);
        mbar_wait(bar_tfull + 8u * grp, aph);
        tc_fence_after();
        if (gt == 0) TRACE(3 + grp, 700 + tc);
        if (p.residual) {
          cp_async_wait0();
          group_sync();
        }
        const RowStats st = ln_pass1(taddr, nc16, N, s_bias, p.relu, p.residual,
                                     my_row, bar_tempty + 8u * grp);
        if (gt == 0) TRACE(3 + grp, 800 + tc);
        ln_normalise(my_row, N, st, p.eps, s_gamma, s_beta);
        if (gt == 0) TRACE(3 + grp, 900 + tc);
        store_row(p.y, p.ldy, row0 + gt, row_end, my_row, N);
        if (gt == 0) TRACE(3 + grp, 1000 + tc);
      } else {
        mbar_wait(bar_tfull + 8u * grp, aph);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < nc16; ++c) {
          float v[16];
          tmem_ld16(taddr + 16u * c, v);
          tmem_ld_wait();
          if (c == nc16 - 1) {
            tc_fence_before();
            mbar_arrive(bar_tempty + 8u * grp);
          }
          const int col = 16 * c + 4 * cq;
          if (p.residual) {  // 16 columns: global -> slab (64 B per row) -> row
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int r = crow + 32 * i;
              float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
              if (row0 + r < row_end && col < N)
                t = __ldg(reinterpret_cast<const float4*>(
                    p.residual + (size_t)(row0 + r) * p.ldr + col));
              *reinterpret_cast<float4*>(slab + (size_t)r * pitch + 4 * cq) = t;
            }
            group_sync();
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float4 t = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            if (16 * c + 4 * j < N) {
              const float4 bb = bias4[4 * c + j];
              t.x += bb.x; t.y += bb.y; t.z += bb.z; t.w += bb.w;
            }
            if (p.relu) {
              t.x = fmaxf(t.x, 0.f); t.y = fmaxf(t.y, 0.f);
              t.z = fmaxf(t.z, 0.f); t.w = fmaxf(t.w, 0.f);
            }
            float4* cell = reinterpret_cast<float4*>(my_row + 4 * j);
            if (p.residual) {
              const float4 r = *cell;
              t.x += r.x; t.y += r.y; t.z += r.z; t.w += r.w;
            }
            *cell = t;
          }
          group_sync();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = crow + 32 * i;
            if (row0 + r < row_end && col < N) {
              float* dst = col < p.n_split
                               ? p.y + (size_t)(row0 + r) * p.ldy + col
                               : p.y2 + (size_t)(row0 + r) * p.ldy2 + (col - p.n_split);
              *reinterpret_cast<float4*>(dst) =
                  *reinterpret_cast<const float4*>(slab + (size_t)r * pitch + 4 * cq);
            }
          }
          group_sync();
        }
      }
    }
  }

  if (LN) bulk_wait0();  // every row's bulk store has completed
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) TRACE(3, 2);
  if (warp == 12) {
    tc_fence_after();
    tmem_dealloc(tmem_base);
  }
}

static inline int n_kblocks(int k) { return (k + kKB - 1) / kKB; }

template <bool LN>
static int launch_linear(const LinearParams& p, size_t smem, int grid,
                         cudaStream_t st) {
  if (const int e = raise_smem_limit<linear_tf32_kernel<LN>>(smem)) return e;
  linear_tf32_kernel<LN><<<grid, kLinThreads, smem, st>>>(p);
  return launch_status();
}

}  // namespace fbbev

using namespace fbbev;

#ifdef TC_TRACE
// kernel 0: linear_tf32_kernel, 1: ffn_tf32_kernel (tools/tc_trace.py)
FBBEV_API int fbbev_debug_tc_trace(int kernel, long long* out, int* counts) {
  return kernel == 0 ? tc_trace_copy(out, counts) : ffn_trace_copy(out, counts);
}
#endif

FBBEV_API size_t fbbev_linear_packed_bytes(int32_t n, int32_t k) {
  if (n <= 0 || k <= 0) return 0;
  return (size_t)n_kblocks(k) * 2 * kKB * pad16(n) * sizeof(float);
}

FBBEV_API int fbbev_linear_pack(const float* weight, int32_t n, int32_t k,
                                float* packed, fbbev_stream_t stream) {
  if (!weight || !packed || n <= 0 || k <= 0) return FBBEV_ERR_INVALID_ARGUMENT;
  if (reinterpret_cast<uintptr_t>(packed) & 15) return FBBEV_ERR_INVALID_ARGUMENT;
  const int npad = pad16(n), nkb = n_kblocks(k);
  const int64_t total = (int64_t)nkb * kChunks * npad;
  count_launch();
  linear_pack_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0,
                       as_stream(stream)>>>(weight, n, k, npad, nkb, packed);
  return launch_status();
}

static int linear_run(const float* x, int64_t ldx, const float* x_add,
                      int64_t ldxa, const float* packed, const float* bias, const float* residual, int64_t ldr,
                      const float* ln_weight, const float* ln_bias, int64_t m,
                      int32_t k, int32_t n, int32_t relu, float ln_eps, float* y,
                      int64_t ldy, float* y2, int64_t ldy2, int32_t n_split,
                      fbbev_stream_t stream) {
  if (!x || !packed || !y || m < 0 || k <= 0 || n <= 0)
    return FBBEV_ERR_INVALID_ARGUMENT;
  if ((ln_weight == nullptr) != (ln_bias == nullptr))
    return FBBEV_ERR_INVALID_ARGUMENT;
  if (k % 4 != 0 || n % 4 != 0 || n > kMaxN || m > (int64_t)1 << 30)
    return FBBEV_ERR_UNSUPPORTED;
  if (ldx < k || ldy < n_split || (residual && ldr < n) || ldx % 4 || ldy % 4 ||
      (residual && ldr % 4))
    return FBBEV_ERR_INVALID_ARGUMENT;
  if (n_split < n &&
      (!y2 || n_split <= 0 || n_split % 4 || ldy2 < n - n_split || ldy2 % 4 ||
       ln_weight || (reinterpret_cast<uintptr_t>(y2) & 15)))
    return FBBEV_ERR_INVALID_ARGUMENT;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) |
       reinterpret_cast<uintptr_t>(packed) |
       reinterpret_cast<uintptr_t>(residual) |
       reinterpret_cast<uintptr_t>(x_add)) & 15)
    return FBBEV_ERR_INVALID_ARGUMENT;
  if (x_add && (ldxa < k || ldxa % 4)) return FBBEV_ERR_INVALID_ARGUMENT;
  if (m == 0) return FBBEV_OK;
  LinearParams p;
  p.x = x; p.x_add = x_add; p.ldxa = ldxa; p.wp = packed; p.bias = bias; p.residual = residual;
  p.gamma = ln_weight; p.beta = ln_bias; p.y = y;
  p.y2 = y2; p.ldy2 = ldy2; p.n_split = n_split;
  p.M = (int)m; p.K = k; p.N = n; p.npad = pad16(n); p.n_kb = n_kblocks(k);
  p.relu = relu; p.eps = ln_eps;
  p.ldx = ldx; p.ldr = ldr; p.ldy = ldy;
  const size_t stage = 2 * (size_t)kAPart + 2 * (size_t)p.npad * kKB * 4;
  // LayerNorm epilogue: whole-row slabs (residual prefetch, fully coalesced
  // stores) when they fit beside two pipeline stages, else 16-column chunks
  const bool ln = ln_weight != nullptr;
  size_t slab_bytes = kSlabBytes;
  p.slab_pitch = kSlabPitch;
  const size_t wide_bytes = 2 * (size_t)kTileM * (n + 4) * 4;
  if (ln) {
    if (2 * stage + kCtrlBytes + wide_bytes > (size_t)kSmemLimit)
      return FBBEV_ERR_UNSUPPORTED;  // n <= 80 with the 40-float K-block
    slab_bytes = wide_bytes;
    p.slab_pitch = n + 4;
  }
  int stages = (int)((kSmemLimit - kCtrlBytes - slab_bytes) / stage);
  stages = stages > 4 ? 4 : stages;
  if (stages < 2) return FBBEV_ERR_UNSUPPORTED;
  p.stages = stages;
  const size_t smem = stages * stage + kCtrlBytes + slab_bytes;
  const int n_sm = sm_count();
  // equal contiguous row ranges (multiples of 8 rows), one CTA per SM
  const int n_tiles = (int)ceil_div64(m, kTileM);
  int grid = n_tiles < n_sm ? n_tiles : n_sm;
  p.rows_per_cta = (int)(ceil_div64(ceil_div64(m, grid), 8) * 8);
  grid = (int)ceil_div64(m, p.rows_per_cta);
  cudaStream_t st = as_stream(stream);
  count_launch();
  return ln ? launch_linear<true>(p, smem, grid, st)
            : launch_linear<false>(p, smem, grid, st);
}

FBBEV_API int fbbev_linear_fwd(const float* x, int64_t ldx, const float* packed,
                               const float* bias, const float* residual,
                               int64_t ldr, const float* ln_weight,
                               const float* ln_bias, int64_t m, int32_t k,
                               int32_t n, int32_t relu, float ln_eps, float* y,
                               int64_t ldy, fbbev_stream_t stream) {
  return linear_run(x, ldx, nullptr, 0, packed, bias, residual, ldr, ln_weight,
                    ln_bias, m, k, n, relu, ln_eps, y, ldy, nullptr, 0, n, stream);
}

FBBEV_API int fbbev_linear_fwd_split(const float* x, int64_t ldx,
                                     const float* x_add, int64_t ldx_add,
                                     const float* packed, const float* bias,
                                     int64_t m, int32_t k, int32_t n,
                                     int32_t n_split, int32_t relu, float* y0,
                                     int64_t ldy0, float* y1, int64_t ldy1,
                                     fbbev_stream_t stream) {
  return linear_run(x, ldx, x_add, ldx_add, packed, bias, nullptr, 0, nullptr,
                    nullptr, m, k, n, relu, 0.f, y0, ldy0, y1, ldy1, n_split,
                    stream);
}
