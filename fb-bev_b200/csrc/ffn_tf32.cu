// ffn_tf32.cu -- the encoder layer's FFN as ONE tcgen05 kernel:
//
//     y = LayerNorm( x + W2 . relu(W1 . x + b1) + b2 )
//
// What it replaces: mmcv `FFN` (Linear -> ReLU -> Linear, identity add) and the
// `norm` that follows it in the reference's operation order
// (bevformer_encoder.py:251-377, config ffn_cfgs / operation_order).  The
// reference runs two cuBLAS GEMMs, three element-wise kernels and a LayerNorm
// kernel; rounds 1 / 2 of this repository ran three launches of
// linear_tf32_kernel (80 -> 192 + ReLU, 80 -> 128 + ReLU, 320 -> 80 + residual +
// LayerNorm) with the 40000 x 320 hidden activation (51 MB) written to and read
// back from HBM / L2 in between.  Here the hidden tile never leaves TENSOR
// MEMORY:
//
//   GEMM1   H[128 x hidden] = X[128 x E] . W1^T  in `hidden / 80` column chunks of
//           80 (A and B from shared memory), accumulators in TMEM columns
//           [0, hidden)
//   convert warps 8-11: tcgen05.ld a 40-column K-block of H (lane == row), add
//           b1, ReLU, split into hi / lo (3xTF32, see linear_tf32.cu); hi goes
//           back IN PLACE with tcgen05.st, lo into a two-stage ring of 40 TMEM
//           columns.  An fp32 accumulator tile (lane == row, column == n) is
//           already the layout tcgen05.mma wants for an A operand in tensor
//           memory (lane == row, column == k), so the second GEMM reads its A
//           operand where the first one left it: no shared-memory round trip
//   GEMM2   Y[128 x E] += H_kb . W2_kb^T per K-block, A from TMEM, B from shared
//           memory, accumulator in TMEM columns [hidden, hidden + E)
//   finish  warps 0-3: tcgen05.ld of Y, + b2 + residual, LayerNorm, row-wise TMA
//           bulk store (as the LayerNorm epilogue of linear_tf32_kernel), while
//           the tensor pipe is already on the next tile
//
// Roles (14 warps): 0-3 finish, 4-7 X loaders, 8-11 convert, 12 MMA issue (one
// elected lane) + TMEM allocation, 13 weight producer (one 1-D bulk copy per
// 25.6 KB stage: W1 chunk x K-block, then W2 K-blocks, in the order the MMA warp
// consumes them).  The weights do not fit beside the X tile, so they are streamed
// from L2 once per tile -- 410 KB -- and that stream bounds the kernel: ~0.72 us
// per stage against 0.40 us for the stage's 15 MMAs (tools/micro/mma_rate.cu:
// 52 / 40 cycles per MMA with A in shared / tensor memory), whether one thread
// issues bulk copies or 128 threads issue cp.async, and not improved by sending
// the weights unsplit and splitting them on the SM (68 us instead of 52: the
// split costs the loader warps more than the bytes saved; profiles/r02_notes.md).
// Hence the ring as deep as shared memory allows, and whole tiles per CTA.
// Shared memory: X tile hi / lo (80 KB) | LayerNorm slab (42 KB) | weight ring
// (4 x 25.6 KB) | barriers, biases, LayerNorm parameters.
// TMEM columns: H [0, hidden) | Y [hidden, hidden + pad16(E)) | lo ring 2 x 40.
//
// Shapes: E <= 80, E % 4 == 0; hidden % 80 == 0, hidden <= 320 (the b1 staged in
// shared memory), hidden + pad16(E) + 80 <= 512.
#include "tc5.cuh"

namespace fbbev {
namespace ffn {

constexpr int kABlock = 2 * kAPart;     // one K-block of X, hi + lo
constexpr int kThreads = 448;
constexpr int kHC = 80;                 // hidden columns per GEMM1 chunk
constexpr int kMaxE = 80;
constexpr int kMaxHidden = 320;
constexpr int kCtrlBytes = 512 + (kMaxHidden + 3 * kMaxE) * 4;
constexpr int kSlabBytes = kTileM * (kMaxE + 4) * 4;

struct Params {
  const float* x;         // [M][E]
  const float* w1p;       // hidden / 80 blocks, each fbbev_linear_pack(80 rows, E)
  const float* b1;        // [hidden] or null
  const float* w2p;       // fbbev_linear_pack(E rows, hidden)
  const float* b2;        // [E] or null
  const float* residual;  // [M][E] or null
  const float* gamma;     // [E] or null (no LayerNorm)
  const float* beta;
  float* y;               // [M][E]
  int M, E, hidden, npad, n_kb1, n_kb2, n_hc, rows_per_cta, wstages;
  int64_t ldx, ldr, ldy;
  float eps;
};

__global__ void __launch_bounds__(kThreads, 1) ffn_tf32_kernel(const Params p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  TRACE_DECL
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int npad = p.npad, S = p.wstages;
  const uint32_t w1_stage = 2u * kHC * kKB * 4;           // W1 chunk x K-block
  const uint32_t w2_stage = 2u * (uint32_t)npad * kKB * 4;  // W2 K-block
  const uint32_t wstage = w1_stage > w2_stage ? w1_stage : w2_stage;
  unsigned char* xa = smem;                               // [n_kb1 <= 2] K-blocks
  unsigned char* slab_raw = smem + 2 * kABlock;           // [128][E + 4] floats
  unsigned char* wr = slab_raw + kSlabBytes;              // [S] weight stages
  unsigned char* ctrl = wr + (size_t)S * wstage;
  const uint32_t bars = smem_u32(ctrl);
  const uint32_t bar_xfull = bars, bar_xempty = bars + 8;
  const uint32_t bar_yfull = bars + 16, bar_yempty = bars + 24;
  const uint32_t bar_hafull = bars + 32;    // [2]
  const uint32_t bar_haempty = bars + 48;   // [2]
  const uint32_t bar_hfull = bars + 64;     // [n_hc <= 5]
  const uint32_t bar_wfull = bars + 128;    // [S <= 4]
  const uint32_t bar_wempty = bars + 160;   // [S]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ctrl + 192);
  float* s_b1 = reinterpret_cast<float*>(ctrl + 512);
  float* s_b2 = s_b1 + kMaxHidden;
  float* s_gamma = s_b2 + kMaxE;
  float* s_beta = s_gamma + kMaxE;
  const uint32_t xa_base = smem_u32(xa), wr_base = smem_u32(wr);

  if (warp == 12) {
    if (lane == 0) {
      mbar_init(bar_xfull, 128);
      mbar_init(bar_xempty, 1);
      mbar_init(bar_yfull, 1);
      mbar_init(bar_yempty, 128);
      for (int g = 0; g < 2; ++g) {
        mbar_init(bar_hafull + 8u * g, 128);
        mbar_init(bar_haempty + 8u * g, 1);
      }
      for (int c = 0; c < p.n_hc; ++c) mbar_init(bar_hfull + 8u * c, 1);
      for (int s = 0; s < S; ++s) {
        mbar_init(bar_wfull + 8u * s, 1);     // expect_tx of the producer
        mbar_init(bar_wempty + 8u * s, 1);
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(smem_u32(tmem_slot));
  }
  for (int j = threadIdx.x; j < kMaxHidden; j += kThreads)
    s_b1[j] = (p.b1 && j < p.hidden) ? p.b1[j] : 0.f;
  for (int j = threadIdx.x; j < kMaxE; j += kThreads) {
    s_b2[j] = (p.b2 && j < p.E) ? p.b2[j] : 0.f;
    s_gamma[j] = (p.gamma && j < p.E) ? p.gamma[j] : 1.f;
    s_beta[j] = (p.beta && j < p.E) ? p.beta[j] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) TRACE(4, 1);
  const int row_begin = blockIdx.x * p.rows_per_cta;
  const int row_end = min(p.M, row_begin + p.rows_per_cta);
  const int n_my = row_end > row_begin ? (row_end - row_begin + kTileM - 1) / kTileM : 0;
  const int stages_per_tile = p.n_hc * p.n_kb1 + p.n_kb2;

  if (warp >= 4 && warp < 8) {
    // ============================== X loaders ================================
    // the whole K range of a 128-row tile per round, through registers (hi / lo
    // split)
    const int lw = warp - 4;
    auto load_x = [&](int ti) {
      float4 v[2][10];
#pragma unroll
      for (int u = 0; u < 2; ++u)
        gather_kblock(v[u], p.x, p.ldx, nullptr, 0, p.E, row_begin + ti * kTileM,
                      row_end, u, u < p.n_kb1, lw, lane);
      if (threadIdx.x == 128) TRACE(0, 100 + ti);
      mbar_wait(bar_xempty, (ti & 1) ^ 1);   // GEMM1 of the previous tile done
      if (threadIdx.x == 128) TRACE(0, 110 + ti);
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (u >= p.n_kb1) break;
        store_kblock(xa + (size_t)u * kABlock, v[u], lw, lane);
      }
      fence_proxy_async();
      mbar_arrive(bar_xfull);
      if (threadIdx.x == 128) TRACE(0, 120 + ti);
    };
    for (int ti = 0; ti < n_my; ++ti) load_x(ti);
  } else if (warp == 13) {
    // ============================ weight producer ============================
    // one 1-D bulk copy (TMA) per stage, issued by an elected lane as soon as
    // the stage is free; all lanes walk the loop (see elect_one())
    const int n_w1 = p.n_hc * p.n_kb1;
    uint32_t it = 0;
    for (int ti = 0; ti < n_my; ++ti) {
      for (int j = 0; j < stages_per_tile; ++j, ++it) {
        const uint32_t s = it % S, ph = (it / S) & 1u;
        const float* src;
        uint32_t bytes;
        if (j < n_w1) {   // W1: chunk c, K-block kb (j = c * n_kb1 + kb)
          src = p.w1p + (size_t)j * (w1_stage / 4u);
          bytes = w1_stage;
        } else {          // W2: K-block j - n_w1
          src = p.w2p + (size_t)(j - n_w1) * (w2_stage / 4u);
          bytes = w2_stage;
        }
        mbar_wait(bar_wempty + 8u * s, ph ^ 1u);
        if (lane == 0) TRACE(1, 1000 + it);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_wfull + 8u * s, bytes);
          bulk_g2s(wr_base + s * wstage, src, bytes, bar_wfull + 8u * s);
        }
        __syncwarp();
      }
    }
  } else if (warp == 12) {
    // =============================== MMA issue ===============================
    // the whole warp walks the loop (all lanes poll the barriers); one elected
    // lane issues -- see elect_one() for why not `if (lane == 0)`
    const uint32_t idesc1 = idesc_tf32_m128(kHC);
    const uint32_t idesc2 = idesc_tf32_m128(npad);
    const uint32_t lbo_b1 = (uint32_t)kHC * 16u, lbo_b2 = (uint32_t)npad * 16u;
    const uint32_t w1_part = (uint32_t)kHC * kKB * 4;
    const uint32_t w2_part = (uint32_t)npad * kKB * 4;
    const uint32_t d_y = tmem_base + (uint32_t)p.hidden;
    const uint32_t d_lo = d_y + (uint32_t)npad;
    uint32_t it = 0, hu = 0;   // weight stage counter, hidden K-block counter
    for (int ti = 0; ti < n_my; ++ti) {
      if (lane == 0) TRACE(2, 200 + ti);
      mbar_wait(bar_xfull, ti & 1);
      tc_fence_after();
      if (lane == 0) TRACE(2, 210 + ti);
      // ---- GEMM1: H chunk c = X . W1[80c : 80c + 80]^T ----
      for (int c = 0; c < p.n_hc; ++c) {
        const uint32_t d = tmem_base + (uint32_t)(c * kHC);
        for (int kb = 0; kb < p.n_kb1; ++kb, ++it) {
          const uint32_t s = it % S, ph = (it / S) & 1u;
          mbar_wait(bar_wfull + 8u * s, ph);
          tc_fence_after();
          if (lane == 0) TRACE(2, 2000 + it);
          const uint32_t w_hi = wr_base + s * wstage;
          if (elect_one()) {
            mma_kblock_ss(d, xa_base + (uint32_t)kb * kABlock, w_hi, w_hi + w1_part,
                          lbo_b1, idesc1, kb);
            tc_commit(bar_wempty + 8u * s);
            if (kb == p.n_kb1 - 1) {
              tc_commit(bar_hfull + 8u * c);    // chunk c can be converted
              if (c == p.n_hc - 1) tc_commit(bar_xempty);   // X tile consumed
            }
          }
          __syncwarp();
        }
      }
      // ---- GEMM2: Y += Hblk . W2blk^T ----
      mbar_wait(bar_yempty, (ti & 1) ^ 1);    // Y of the previous tile drained
      tc_fence_after();
      for (int kb = 0; kb < p.n_kb2; ++kb, ++it, ++hu) {
        const uint32_t s = it % S, ph = (it / S) & 1u;
        const uint32_t g = (uint32_t)kb & 1u, hph = (hu >> 1) & 1u;
        mbar_wait(bar_wfull + 8u * s, ph);
        if (lane == 0) TRACE(2, 2000 + it);
        mbar_wait(bar_hafull + 8u * g, hph);
        tc_fence_after();
        if (lane == 0) TRACE(2, 3000 + it);
        // A from tensor memory: hi where GEMM1 left the K-block (converted
        // in place), lo in ring stage g
        const uint32_t w_hi = wr_base + s * wstage;
        if (elect_one()) {
          mma_kblock_ts(d_y, tmem_base + (uint32_t)(kb * kKB), d_lo + g * (uint32_t)kKB,
                        w_hi, w_hi + w2_part, lbo_b2, idesc2, kb);
          tc_commit(bar_wempty + 8u * s);
          tc_commit(bar_haempty + 8u * g);
          if (kb == p.n_kb2 - 1) tc_commit(bar_yfull);
        }
        __syncwarp();
      }
      if (lane == 0) TRACE(2, 220 + ti);
    }
    __syncwarp();
  } else if (warp != 13) {
    // ===================== convert (warps 8-11) / finish (0-3) ===============
    const uint32_t grp = warp >> 3;          // 0: finish, 1: convert
    const int q = warp & 3;
    const int gt = q * 32 + lane;            // row of the tile == TMEM lane
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    const int E = p.E;
    if (grp == 1) {
      const uint32_t t_lo = lane_base + (uint32_t)(p.hidden + npad);
      uint32_t use = 0;                      // K-blocks converted so far
      for (int ti = 0; ti < n_my; ++ti) {
        for (int kb = 0; kb < p.n_kb2; ++kb, ++use) {
          const uint32_t g = use & 1u;       // == kb & 1 (n_kb2 is even)
          mbar_wait(bar_hfull + 8u * (kb / (kHC / kKB)), ti & 1);
          if (threadIdx.x == 256) TRACE(3, 4000 + use);
          mbar_wait(bar_haempty + 8u * g, ((use >> 1) & 1u) ^ 1u);
          tc_fence_after();
          if (threadIdx.x == 256) TRACE(3, 5000 + use);
          const uint32_t taddr = lane_base + (uint32_t)(kb * kKB);
          float v[kKB], lo[kKB];
          tmem_ld16(taddr, v);
          tmem_ld16(taddr + 16u, v + 16);
          tmem_ld8(taddr + 32u, v + 32);
          tmem_ld_wait();
          const float* bias = s_b1 + kb * kKB;
#pragma unroll
          for (int c = 0; c < kKB; ++c) tf32_split(fmaxf(v[c] + bias[c], 0.f), v[c], lo[c]);
          tmem_st16(taddr, v);
          tmem_st16(taddr + 16u, v + 16);
          tmem_st8(taddr + 32u, v + 32);
          const uint32_t tl = t_lo + g * (uint32_t)kKB;
          tmem_st16(tl, lo);
          tmem_st16(tl + 16u, lo + 16);
          tmem_st8(tl + 32u, lo + 32);
          tmem_st_wait();
          tc_fence_before();
          mbar_arrive(bar_hafull + 8u * g);
          if (threadIdx.x == 256) TRACE(3, 6000 + use);
        }
      }
    } else {
      // ---- finish: Y + b2 + residual -> LayerNorm -> bulk store ----
      const int pitch = E + 4;
      float* slab = reinterpret_cast<float*>(slab_raw);
      float* my_row = slab + (size_t)gt * pitch;
      const uint32_t ty = lane_base + (uint32_t)p.hidden;
      const int nc16 = npad >> 4;
      for (int ti = 0; ti < n_my; ++ti) {
        const int row0 = row_begin + ti * kTileM;
        bulk_wait_read0();   // my row of the previous tile has left the slab
        asm volatile("bar.sync 1, 128;" ::: "memory");   // ... and everybody's
        // residual rows of this tile -> slab with cp.async while the tensor
        // pipe is still on the tile (4 lanes per row, 64 contiguous bytes per
        // row and round: coalesced; a load per thread and row inside the pass
        // below cost a full L2 round trip each: 6 us per tile)
        if (p.residual)
          prefetch_rows(slab, pitch, p.residual, p.ldr, row0, row_end, row_begin,
                        E, nc16, gt);
        if (threadIdx.x == 0) TRACE(4, 300 + ti);
        mbar_wait(bar_yfull, ti & 1);
        tc_fence_after();
        if (threadIdx.x == 0) TRACE(4, 310 + ti);
        if (p.residual) {
          cp_async_wait0();
          asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        const RowStats st =
            ln_pass1(ty, nc16, E, s_b2, false, p.residual, my_row, bar_yempty);
        if (p.gamma) ln_normalise(my_row, E, st, p.eps, s_gamma, s_beta);
        store_row(p.y, p.ldy, row0 + gt, row_end, my_row, E);
        if (threadIdx.x == 0) TRACE(4, 320 + ti);
      }
      bulk_wait0();
      if (threadIdx.x == 0) TRACE(4, 330);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 12) {
    tc_fence_after();
    tmem_dealloc(tmem_base);
  }
}

}  // namespace ffn
}  // namespace fbbev

using namespace fbbev;

#ifdef TC_TRACE
int fbbev::ffn_trace_copy(long long* out, int* counts) {
  return tc_trace_copy(out, counts);
}
#endif

FBBEV_API int fbbev_ffn_supported(int32_t embed, int32_t hidden) {
  return embed > 0 && embed <= ffn::kMaxE && embed % 4 == 0 && hidden > 0 &&
                 hidden % ffn::kHC == 0 &&
                 hidden + pad16(embed) + 2 * kKB <= kTmemCols &&
                 hidden <= ffn::kMaxHidden
             ? 1
             : 0;
}

FBBEV_API int fbbev_ffn_fwd(const float* x, int64_t ldx, const float* w1_packed,
                            const float* b1, const float* w2_packed,
                            const float* b2, const float* residual, int64_t ldr,
                            const float* ln_weight, const float* ln_bias,
                            int64_t m, int32_t embed, int32_t hidden,
                            float ln_eps, float* y, int64_t ldy,
                            fbbev_stream_t stream) {
  if (!x || !w1_packed || !w2_packed || !y || m < 0)
    return FBBEV_ERR_INVALID_ARGUMENT;
  if ((ln_weight == nullptr) != (ln_bias == nullptr))
    return FBBEV_ERR_INVALID_ARGUMENT;
  if (!fbbev_ffn_supported(embed, hidden) || m > (int64_t)1 << 30)
    return FBBEV_ERR_UNSUPPORTED;
  if (ldx < embed || ldy < embed || (residual && ldr < embed) || ldx % 4 ||
      ldy % 4 || (residual && ldr % 4))
    return FBBEV_ERR_INVALID_ARGUMENT;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) |
       reinterpret_cast<uintptr_t>(w1_packed) |
       reinterpret_cast<uintptr_t>(w2_packed) |
       reinterpret_cast<uintptr_t>(residual)) & 15)
    return FBBEV_ERR_INVALID_ARGUMENT;
  if (m == 0) return FBBEV_OK;
  ffn::Params p;
  p.x = x; p.w1p = w1_packed; p.b1 = b1; p.w2p = w2_packed; p.b2 = b2;
  p.residual = residual; p.gamma = ln_weight; p.beta = ln_bias; p.y = y;
  p.M = (int)m; p.E = embed; p.hidden = hidden; p.npad = pad16(embed);
  p.n_kb1 = (embed + kKB - 1) / kKB;
  p.n_kb2 = hidden / kKB;
  p.n_hc = hidden / ffn::kHC;
  p.ldx = ldx; p.ldr = ldr; p.ldy = ldy; p.eps = ln_eps;
  const size_t w1_stage = 2 * (size_t)ffn::kHC * kKB * 4;
  const size_t w2_stage = 2 * (size_t)p.npad * kKB * 4;
  const size_t wstage = w1_stage > w2_stage ? w1_stage : w2_stage;
  const size_t fixed =
      2 * (size_t)ffn::kABlock + ffn::kSlabBytes + ffn::kCtrlBytes;
  int S = (int)((kSmemLimit - fixed) / wstage);
  S = S > 4 ? 4 : S;
  if (S < 2) return FBBEV_ERR_UNSUPPORTED;
  p.wstages = S;
  const size_t smem = fixed + (size_t)S * wstage;
  const int n_sm = sm_count();
  // whole tiles per CTA: every tile costs one pass over the weights (410 KB
  // from L2) whatever its row count, so 105 CTAs x 3 full tiles beat 148 CTAs
  // x (2 full + 1 sliver) for 40000 rows: same makespan, 30 % less L2 traffic
  const int n_tiles = (int)ceil_div64(m, kTileM);
  const int tiles_per_cta = (int)ceil_div64(n_tiles, n_sm);
  p.rows_per_cta = tiles_per_cta * kTileM;
  const int grid = (int)ceil_div64(m, p.rows_per_cta);
  if (const int e = raise_smem_limit<ffn::ffn_tf32_kernel>(smem)) return e;
  count_launch();
  ffn::ffn_tf32_kernel<<<grid, ffn::kThreads, smem, as_stream(stream)>>>(p);
  return launch_status();
}
