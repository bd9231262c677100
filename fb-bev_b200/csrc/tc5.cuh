// tc5.cuh -- the tcgen05 side shared by linear_tf32.cu and ffn_tf32.cu:
// tcgen05.mma / commit / ld / st wrappers, shared-memory matrix descriptors
// (K-major, no swizzle), and the pipeline stages both kernels are built from
// (3xTF32 operand split, X loader, k-block MMA issue, LayerNorm epilogue).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bulk.cuh"
#include "common.cuh"

namespace fbbev {

// ------------------------------ tile geometry --------------------------------
constexpr int kKB = 40;                            // floats of K per K-block
constexpr int kChunks = kKB / 4;                   // 16-byte chunks of a row
constexpr int kTileM = 128;                        // rows of a tile (MMA M)
constexpr int kAPart = kTileM * kKB * 4;           // bytes of A_hi (== A_lo)
constexpr int kAChunkStride = (kTileM / 8) * 128;  // bytes between K chunks
constexpr int kTmemCols = 512;
constexpr int kSmemLimit = 232448 - 1024;
constexpr int pad16(int n) { return (n + 15) / 16 * 16; }

// ------------------------------- trace builds --------------------------------
#ifdef TC_TRACE
// -DTC_TRACE: timeline of CTA 0.  Every tracing thread (one per role) appends
// (tag, clock64) to its role's region of a global buffer with plain stores and
// a private counter; fbbev_debug_tc_trace copies it out (tools/tc_trace.py).
constexpr int kTraceRoles = 5, kTraceCap = 200;
static __device__ long long g_tc_trace[kTraceRoles * 2 * kTraceCap];
static __device__ int g_tc_trace_cnt[kTraceRoles];
#define TRACE_DECL int trn_ = 0;
#define TRACE(role, tag)                                                     \
  do {                                                                       \
    if (blockIdx.x == 0 && trn_ < kTraceCap) {                               \
      g_tc_trace[(role) * 2 * kTraceCap + 2 * trn_] = (tag);                 \
      g_tc_trace[(role) * 2 * kTraceCap + 2 * trn_ + 1] = clock64();         \
      g_tc_trace_cnt[role] = ++trn_;                                         \
    }                                                                        \
  } while (0)
// this translation unit's buffer -> host; returns the capacity per role
static inline int tc_trace_copy(long long* out, int* counts) {
  cudaMemcpyFromSymbol(counts, g_tc_trace_cnt, sizeof(int) * kTraceRoles);
  cudaMemcpyFromSymbol(out, g_tc_trace, sizeof(long long) * kTraceRoles * 2 * kTraceCap);
  return kTraceCap;
}
int ffn_trace_copy(long long* out, int* counts);  // ffn_tf32.cu
#else
#define TRACE_DECL
#define TRACE(role, tag) do {} while (0)
#endif

// ------------------------------- PTX wrappers --------------------------------
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 "
      "[%0];" ::"r"(bar)
      : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, tf32 operands, fp32 accumulate
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t da, uint64_t db,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand from tensor memory (lane == row, one 32-bit column per K element),
// B from shared memory:  D[tmem] (+)= A[tmem] . B[smem]^T
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem,
                                            uint64_t db, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// K-major operand without swizzle: 8-row x 16-byte core matrices; `lbo` bytes
// between the two K chunks of one MMA, `sbo` bytes between 8-row groups
// (cute::UMMA::SmemDescriptor, version 1, LayoutType::SWIZZLE_NONE).
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo,
                                              uint32_t sbo) {
  return (uint64_t)((addr >> 4) & 0x3FFFu) |
         ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]),
        "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]),
        "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]),
        "=r"(r[6]), "=r"(r[7])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(
          taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])),
      "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
      "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])),
      "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])),
      "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])),
      "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
      "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// One lane of a CONVERGED warp (elect.sync).  Code that issues tcgen05.mma /
// tcgen05.commit / bulk copies should run as `if (elect_one()) { ... }` inside
// warp-uniform control flow: under a divergent `if (lane == 0)` the compiler
// cannot prove that one thread executes the uniform-datapath instruction and
// wraps EVERY UTCHMMA in an ELECT / BRA.U.ANY serialisation loop (~7 extra
// instructions per MMA on a single-thread critical path).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------- TMEM -------------------------------------
// whole warp: all 512 columns; the base address is written to `slot`
__device__ __forceinline__ void tmem_alloc(uint32_t slot) {
  asm volatile(
      "tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot),
      "r"(kTmemCols)
      : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::
                   : "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base),
               "r"(kTmemCols)
               : "memory");
}

// --------------------------------- 3xTF32 ------------------------------------
// x = hi + lo: hi the upper 19 bits (a tf32 value), lo the exact fp32 remainder
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  lo = x - hi;
}
__device__ __forceinline__ void tf32_split(const float4& x, float4& hi, float4& lo) {
  tf32_split(x.x, hi.x, lo.x);
  tf32_split(x.y, hi.y, lo.y);
  tf32_split(x.z, hi.z, lo.z);
  tf32_split(x.w, hi.w, lo.w);
}

// Byte offset of 16-byte chunk `ch` of `row` in the canonical K-major image
// (8 x 16-byte core matrices, no swizzle) of a `rows`-row operand.
__device__ __forceinline__ uint32_t kmajor_off(int row, int ch,
                                               int rows = kTileM) {
  return (uint32_t)(ch * (rows / 8) + (row >> 3)) * 128u + (row & 7) * 16u;
}

// ------------------------------- X loader ------------------------------------
// Loader thread (lw = loader warp 0..3, lane) of K-block `kb` of the 128-row
// tile at `row0`: rows row0 + 32 lw + (lane & 15) + 16 h (h = i / 5), columns
// kb * 40 + 4 (lane >> 4) + 8 (i % 5); zero outside [.., row_end) x [0, K) and
// when !valid.  With x_add the input is x + x_add (one fp32 add, as torch).
__device__ __forceinline__ void gather_kblock(float4 (&v)[10], const float* x,
                                              int64_t ldx, const float* x_add,
                                              int64_t ldxa, int K, int row0,
                                              int row_end, int kb, bool valid,
                                              int lw, int lane) {
  const int r_lo = lane & 15, c_lo = lane >> 4;
  const int g0 = row0 + lw * 32 + r_lo;
  const int col0 = kb * kKB + 4 * c_lo;
  const float* b0 = x + (size_t)g0 * ldx + col0;
  const float* b1 = b0 + (size_t)16 * ldx;
  const bool ok0 = valid && g0 < row_end;
  const bool ok1 = valid && g0 + 16 < row_end;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int cp = i % 5;
    const bool ok = (i < 5 ? ok0 : ok1) && col0 + 8 * cp < K;
    v[i] = ok ? __ldg(reinterpret_cast<const float4*>((i < 5 ? b0 : b1) + 8 * cp))
              : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (x_add) {
    const float* a0 = x_add + (size_t)g0 * ldxa + col0;
    const float* a1 = a0 + (size_t)16 * ldxa;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      const int cp = i % 5;
      const bool ok = (i < 5 ? ok0 : ok1) && col0 + 8 * cp < K;
      if (ok) {
        const float4 a =
            __ldg(reinterpret_cast<const float4*>((i < 5 ? a0 : a1) + 8 * cp));
        v[i].x = __fadd_rn(v[i].x, a.x);
        v[i].y = __fadd_rn(v[i].y, a.y);
        v[i].z = __fadd_rn(v[i].z, a.z);
        v[i].w = __fadd_rn(v[i].w, a.w);
      }
    }
  }
}
// The gathered K-block, split hi / lo, into its place in the A image at `a`
// (A_hi, then A_lo kAPart bytes later).
__device__ __forceinline__ void store_kblock(unsigned char* a, const float4 (&v)[10],
                                             int lw, int lane) {
  const int r_lo = lane & 15, c_lo = lane >> 4;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int idx = lw * 10 + i;
    const int row = (idx / 5) * 16 + r_lo;
    const int ch = (idx % 5) * 2 + c_lo;
    float4 hi, lo;
    tf32_split(v[i], hi, lo);
    unsigned char* p = a + kmajor_off(row, ch);
    *reinterpret_cast<float4*>(p) = hi;
    *reinterpret_cast<float4*>(p + kAPart) = lo;
  }
}

// ------------------------------- MMA issue -----------------------------------
// instruction descriptor: kind::tf32, fp32 accumulate, A and B K-major,
// M = 128, N = n
__device__ __forceinline__ uint32_t idesc_tf32_m128(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) |
         (8u << 24);
}
// One K-block as 3xTF32 (x_hi.w_hi + x_lo.w_hi + x_hi.w_lo per k-step) into
// the accumulator at d_tmem.  B is the K-major image of one K-block (hi at
// w_hi, lo at w_lo, `lbo_b` bytes between its K chunks: 16 x its rows).  The
// first k-step of K-block 0 overwrites the accumulator.  Issue from ONE
// elected lane (see elect_one()).
//   SS: A hi / lo from the shared-memory image at a_hi (lo kAPart later)
__device__ __forceinline__ void mma_kblock_ss(uint32_t d_tmem, uint32_t a_hi,
                                              uint32_t w_hi, uint32_t w_lo,
                                              uint32_t lbo_b, uint32_t idesc,
                                              int kb) {
  const uint32_t a_lo = a_hi + kAPart;
#pragma unroll
  for (int k = 0; k < kChunks / 2; ++k) {
    const uint32_t ao = 2u * k * kAChunkStride, bo = 2u * k * lbo_b;
    const uint64_t dah = smem_desc(a_hi + ao, kAChunkStride, 128);
    const uint64_t dal = smem_desc(a_lo + ao, kAChunkStride, 128);
    const uint64_t dbh = smem_desc(w_hi + bo, lbo_b, 128);
    const uint64_t dbl = smem_desc(w_lo + bo, lbo_b, 128);
    mma_tf32(d_tmem, dah, dbh, idesc, (kb | k) != 0);
    mma_tf32(d_tmem, dal, dbh, idesc, 1u);
    mma_tf32(d_tmem, dah, dbl, idesc, 1u);
  }
}
//   TS: A hi / lo from tensor-memory columns a_hi / a_lo
__device__ __forceinline__ void mma_kblock_ts(uint32_t d_tmem, uint32_t a_hi,
                                              uint32_t a_lo, uint32_t w_hi,
                                              uint32_t w_lo, uint32_t lbo_b,
                                              uint32_t idesc, int kb) {
#pragma unroll
  for (int k = 0; k < kChunks / 2; ++k) {
    const uint32_t bo = 2u * k * lbo_b;
    const uint64_t dbh = smem_desc(w_hi + bo, lbo_b, 128);
    const uint64_t dbl = smem_desc(w_lo + bo, lbo_b, 128);
    mma_tf32_ts(d_tmem, a_hi + 8u * k, dbh, idesc, (kb | k) != 0);
    mma_tf32_ts(d_tmem, a_lo + 8u * k, dbh, idesc, 1u);
    mma_tf32_ts(d_tmem, a_hi + 8u * k, dbl, idesc, 1u);
  }
}

// --------------------------- LayerNorm epilogue ------------------------------
// One 128-thread group drains a 128 x N accumulator: thread gt owns row gt of
// the tile and keeps it in its row of a shared-memory slab (pitch floats)
// between the passes.

// Residual rows [row0, row0 + 128) -> slab with cp.async (4 threads per row,
// 64 contiguous bytes per row and round: coalesced), committed as one group
// that lands while the tensor pipe is still on the tile.  Rows past row_end
// and columns past n are zero-filled (reading a valid address: row_begin).
__device__ __forceinline__ void prefetch_rows(float* slab, int pitch,
                                              const float* src, int64_t ld,
                                              int row0, int row_end, int row_begin,
                                              int n, int nc16, int gt) {
  const int crow = gt >> 2, cq = gt & 3;
#pragma unroll 1
  for (int c = 0; c < nc16; ++c) {
    const int col = 16 * c + 4 * cq;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = crow + 32 * i;
      const bool ok = row0 + r < row_end && col < n;
      const float* s =
          src + (size_t)(ok ? row0 + r : row_begin) * ld + (ok ? col : 0);
      cp_async16_zfill(smem_u32(slab + (size_t)r * pitch + col), s, ok ? 16 : 0);
    }
  }
  cp_async_commit();
}

// Pass 1: accumulator columns [0, N) at taddr + bias (+ ReLU) (+ the residual
// already in my_row) -> my_row; sum and sum of squares about a shift K = the
// row's first element (a one-pass variance that does not cancel: |mean - K| is
// a few sigma at most).  Arrives on `acc_empty` after the last tcgen05.ld.
struct RowStats {
  float sum, sq, shift;
};
__device__ __forceinline__ RowStats ln_pass1(uint32_t taddr, int nc16, int N,
                                             const float* bias, bool relu,
                                             bool residual, float* my_row,
                                             uint32_t acc_empty) {
  float sum = 0.f, sq = 0.f, shiftK = 0.f;
#pragma unroll 1
  for (int c = 0; c < nc16; ++c) {
    float v[16];
    tmem_ld16(taddr + 16u * c, v);
    tmem_ld_wait();
    if (c == nc16 - 1) {
      tc_fence_before();
      mbar_arrive(acc_empty);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = 16 * c + 4 * j;
      if (col < N) {
        const float4 bb = *reinterpret_cast<const float4*>(bias + col);
        float4 t = make_float4(v[4 * j] + bb.x, v[4 * j + 1] + bb.y,
                               v[4 * j + 2] + bb.z, v[4 * j + 3] + bb.w);
        if (relu) {
          t.x = fmaxf(t.x, 0.f); t.y = fmaxf(t.y, 0.f);
          t.z = fmaxf(t.z, 0.f); t.w = fmaxf(t.w, 0.f);
        }
        float4* cell = reinterpret_cast<float4*>(my_row + col);
        if (residual) {
          const float4 r = *cell;
          t.x += r.x; t.y += r.y; t.z += r.z; t.w += r.w;
        }
        *cell = t;
        if (col == 0) shiftK = t.x;
        const float a = t.x - shiftK, b = t.y - shiftK, cc = t.z - shiftK,
                    d = t.w - shiftK;
        sum += (a + b) + (cc + d);
        sq += (a * a + b * b) + (cc * cc + d * d);
      }
    }
  }
  return {sum, sq, shiftK};
}

// Pass 2: normalise my_row in place.
__device__ __forceinline__ void ln_normalise(float* my_row, int N, const RowStats& s,
                                             float eps, const float* gamma,
                                             const float* beta) {
  const float dm = s.sum / (float)N;  // mean - K
  const float mean = s.shift + dm;
  const float var = fmaxf(s.sq / (float)N - dm * dm, 0.f);
  const float rstd = rsqrtf(var + eps);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll 4
  for (int j = 0; j < (N >> 2); ++j) {
    float4* cell = reinterpret_cast<float4*>(my_row + 4 * j);
    const float4 t = *cell, g = g4[j], b = b4[j];
    *cell = make_float4(fmaf((t.x - mean) * rstd, g.x, b.x),
                        fmaf((t.y - mean) * rstd, g.y, b.y),
                        fmaf((t.z - mean) * rstd, g.z, b.z),
                        fmaf((t.w - mean) * rstd, g.w, b.w));
  }
}

// The finished row leaves as ONE bulk (TMA) store issued by its own thread:
// N * 4 contiguous bytes in the slab and in y.  No barrier and no LDS / STG
// loop: the thread's own STS are ordered before its bulk copy by the proxy
// fence.  Every thread commits a bulk group (empty for rows past row_end).
__device__ __forceinline__ void store_row(float* y, int64_t ldy, int row,
                                          int row_end, const float* my_row, int N) {
  if (row < row_end) {
    fence_proxy_async();
    bulk_s2g(y + (size_t)row * ldy, smem_u32(my_row), (uint32_t)N * 4u);
  }
  bulk_commit();
}

// ------------------------------- host side -----------------------------------
// Raises the dynamic shared-memory limit of `Kernel` when a launch needs more
// than any launch before it.
template <auto Kernel>
static inline int raise_smem_limit(size_t bytes) {
  static size_t allowed = 0;
  if (bytes > allowed) {
    const cudaError_t e = cudaFuncSetAttribute(
        Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
    allowed = bytes;
  }
  return FBBEV_OK;
}

}  // namespace fbbev
