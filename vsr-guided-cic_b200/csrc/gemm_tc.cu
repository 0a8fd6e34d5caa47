// tcgen05 / TMEM / TMA GEMM for the per-step dense contractions (LSTM gates, sentinel / attention
// projections, vocabulary projection):   C[M][N] = sum_seg A_seg[M][K_seg] * W[N][K]^T (+ epilogue).
//
// Precision: "f16x3" error-compensated split.  Every fp32 operand x is carried as two fp16 arrays
//   x_hi = fp16(x),  x_lo = fp16(x - x_hi)          (11-bit significands: hi + lo carries ~22 bits)
// and each product is issued as three tensor-core MMAs into the SAME fp32 TMEM accumulator:
//   A_hi*W_hi + A_hi*W_lo + A_lo*W_hi        (dropped: A_lo*W_lo ~ 2^-22 relative)
// which restores ~fp32 accuracy (SURVEY.md §7: token-identical to the reference where a single
// bf16 / tf32 pass is not) at one third of the 16-bit tensor rate and the same operand bytes as
// fp32.  fp16 rather than bf16 because its 3 extra mantissa bits per half buy 2^-6 in the split;
// the path's operands (|x| << 65504: gates in [-1,1], Xavier weights, pooled CNN features) fit its
// range, lo parts of small values degrade gracefully through fp16 subnormals (abs error <= 2^-25).
//
// Structure (one 128 x BN output tile per CTA, 320 threads):
//   warp 0   : TMA producer   cp.async.bulk.tensor.2d -> swizzled smem tiles, mbarrier expect_tx; the weight halves of
//              the first ring pass are fetched before the programmatic-dependent-launch wait
//   warp 1   : TMEM allocator + single-thread tcgen05.mma issuer (kind::f16, M=128, N=BN, K=16)
//   warps 2-9: epilogue (two warps per TMEM lane quarter): bias -> smem behind the main loop; then one lane quarter at
//              a time TMEM -> swizzled smem tile -> all eight warps with lanes along a row (coalesced operands and
//              outputs): plain / g_t / fused LSTM cells; the vocabulary head keeps the row-per-thread form
// smem ring: kStages x {A_hi, A_lo (128 x KB fp16), W_hi, W_lo (BN x KB fp16)}, full/empty mbarriers; the accumulator
// hand-off to the epilogue is a tcgen05.commit on a third mbarrier.  k_gemm_tcp is the persistent variant
// (double-buffered TMEM accumulator), k_gemm_tc2 the CTA-pair experiment.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include <cuda_fp16.h>

#include <algorithm>

#include "common.cuh"

namespace vsr {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;                 // fp16 elements per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 16;
// warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..9 = epilogue.  TMEM lane quarter q is readable by the warps
// with (warp & 3) == q, so every quarter has two epilogue warps (hsel = 0 / 1).
constexpr int TC_EPI_WARPS = 8;
constexpr int TC_EPI_THREADS = 32 * TC_EPI_WARPS;
constexpr int TC_THREADS = 64 + TC_EPI_THREADS;

// KB = fp16 elements per k-block: 64 (one 128-byte swizzle row) or 32 (64-byte swizzle).  The smaller
// block halves the stage size, i.e. doubles the ring depth that fits in 227 KB of shared memory — these
// GEMMs are bound by operand-delivery latency (measured: 2 -> 3 stages = +17..26 % on the K = 3072 shapes).
template <int BN, int KB> struct TcCfg {
  static constexpr int kStageB = 2 * BM * KB * 2 + 2 * BN * KB * 2;
  static constexpr int kStages = (220 * 1024) / kStageB > 8 ? 8 : (220 * 1024) / kStageB;
  static constexpr int kTmemCols = (BN <= 128) ? 128 : 256;   // power of two >= BN
  static constexpr int kABytes = BM * KB * 2;            // 16 / 8 KB
  static constexpr int kWBytes = BN * KB * 2;
  static constexpr int kStageBytes = 2 * kABytes + 2 * kWBytes;
  static constexpr int kRingBytes = kStages * kStageBytes;
  // epilogue tile: one TMEM lane quarter (32 rows x BN fp32) staged through shared memory (tile_epilogue)
  static constexpr bool kTileEpi = (BN == 128 || BN == 192);
  // (the vocabulary epilogue's 4 KB exchange buffer lives in the same place; the two are never used together)
  static constexpr int kEpiBytes = kTileEpi ? 32 * BN * 4 : 4096;
  static constexpr int kSmemBytes = kRingBytes + 1024 + kEpiBytes;   // + alignment slack
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// K-major operand tile with 64-byte swizzle (rows of 64 B, 8-row groups 512 B apart)
__device__ __forceinline__ uint64_t make_sw64_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;                      // stride byte offset: 8 rows x 64 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;                               // layout type: SWIZZLE_64B
  return d;
}
template <int KB> __device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr);

// K-major, 128-byte-swizzled operand tile (rows of 128 B, 8-row groups 1024 B apart): UMMA smem descriptor
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);          // start address  [0,14)
  d |= (uint64_t)1 << 16;                               // leading byte offset (unused for swizzled K-major) = 1
  d |= (uint64_t)(1024 >> 4) << 32;                     // stride byte offset [32,46): 8 rows x 128 B
  d |= (uint64_t)1 << 46;                               // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                               // layout type: SWIZZLE_128B
  return d;
}

template <> __device__ __forceinline__ uint64_t make_kmajor_desc<64>(uint32_t a) { return make_sw128_desc(a); }
template <> __device__ __forceinline__ uint64_t make_kmajor_desc<32>(uint32_t a) { return make_sw64_desc(a); }

// K-major operand tile with 32-byte swizzle (rows of 32 B, 8-row groups 256 B apart)
__device__ __forceinline__ uint64_t make_sw32_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(256 >> 4) << 32;                      // stride byte offset: 8 rows x 32 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;                               // layout type: SWIZZLE_32B
  return d;
}
// 8-bit (e4m3) operand tiles of a KB-element k-block: rows of KB bytes
template <int KB> __device__ __forceinline__ uint64_t make_kmajor_desc8(uint32_t smem_addr);
template <> __device__ __forceinline__ uint64_t make_kmajor_desc8<64>(uint32_t a) { return make_sw64_desc(a); }
template <> __device__ __forceinline__ uint64_t make_kmajor_desc8<32>(uint32_t a) { return make_sw32_desc(a); }

// instruction descriptor, kind::f16: D=f32 (bit 4), A=B=f16 (format 0), both K-major, M=128, N=BN
template <int BN> __device__ __forceinline__ constexpr uint32_t make_idesc() {
  return (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// kind::f8f6f4 with e4m3 operands (format code 0 in the same descriptor fields): M=128, N=BN, K=32, twice the f16 rate
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}



enum { EPI_PLAIN = 0, EPI_LSTM1 = 1, EPI_LSTM2 = 2, EPI_VOCAB = 3 };

// One GEMM problem.  Up to two independent problems (same tile shape) share a launch.
struct TcProblem {
  CUtensorMap a_hi[3], a_lo[3], w_hi, w_lo;     // fp16 hi; lo = fp16 residual (f16x3) or e4m3 residual (f16+f8x2)
  CUtensorMap a_h8[3], w_h8;                   // f16+f8x2 only: e4m3 copies of hi
  int f8;                                      // 1 = f16+f8x2 mode
  int nseg;
  int kblocks[3];
  int n_tiles, m_tiles, M;
  const uint8_t* row_skip;
  // plain epilogue: C = acc + bias[n] + rowadd[(row/row_div)*rowadd_mul][n] + cadd[row][n]
  const float* bias;
  const float* rowadd; int ld_rowadd, row_div, rowadd_mul;
  const float* cadd; int ld_cadd;
  const float* gather; int ld_gather; const int32_t* gather_idx;   // + gather[gather_idx[row]][n]
  float* c; int ldc;
  // fused LSTM-cell epilogues (gate-interleaved output columns, see cell_col() in common.cuh)
  int mode;
  const float* c_old; float* c_new; float* h_new; TwinOut h_tw;
  float* s_new; TwinOut s_tw; float* gq;
  int ld_state;
  // fused g_t = sig(gq + acc) * tanh(c1') on the tiles with n0 < gt_cols (plain epilogue elsewhere)
  int gt_cols; const float* gt_gq; const float* gt_c1n; float* g_t; TwinOut g_tw;
  // EPI_VOCAB: per (row, N tile) softmax / top-k partial records instead of (or besides, when c != null) the logits
  float* vpart; int n_valid;
  int zero_acc;     // k_gemm_tc only: no main loop, the accumulator is taken as zero
  const float* acc_scale;   // device scalar 1/s undoing the power-of-two scale of the weight's fp16 pair, or null
  float act_inv;            // 1 / (constant scale of the activation twins): folded into the same epilogue multiply
};
struct TcParams {
  TcProblem pr[2];
  int nprob;
  int pdl_flags;
};

// ---------------------------------------------------------------- epilogues
// The accumulator leaves TMEM one ROW per thread.  An epilogue that touches global memory in that layout issues 32
// scattered 16-byte requests per warp instruction — one L1 wavefront each — and measured (clock64 + ablation) the
// fused LSTM epilogue of GEMM-A at 15 us of a 47 us kernel, two thirds of it LSU wavefronts (loads 7.7k cycles,
// stores 9.1k, math 9k).  tile_epilogue therefore stages one TMEM lane quarter at a time (32 rows x BN fp32,
// swizzled) in shared memory and lets all eight epilogue warps work on it with lanes running ALONG a row:
// every global load / store of a warp is then 128 contiguous bytes per row.
__device__ __forceinline__ void epi_bar(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(TC_EPI_THREADS) : "memory"); }

#ifdef VSR_DBG_CLK
// k_gemm_pair's clock64 record of one tile of one CTA (tc_dbg_clk_report): absolute clocks of the CTA's SM, except the
// durations in DBG_MFULL and the per-quarter [dump, epi_bar(3), process, epi_bar(4)] block of epilogue warp 2 at DBG_Q
enum {
  DBG_M0, DBG_M1, DBG_M2, DBG_MFULL,            // MMA issuer (leader): tmem_empty wait from M0 to M1, k-loop M1..M2, sum of full waits
  DBG_E0, DBG_E1, DBG_E2, DBG_E3, DBG_E4,       // epilogue: start, bias + epi_bar(1) done, tmem_full done, accumulator released, end
  DBG_Q, DBG_F = DBG_Q + 16
};
constexpr int DBG_CTAS = 160, DBG_TILES = 48;
__device__ long long g_dbg_clk[DBG_CTAS * DBG_TILES * DBG_F];
__device__ __forceinline__ long long* dbg_rec(int ti) {
  return (blockIdx.x < DBG_CTAS && ti < DBG_TILES) ? g_dbg_clk + ((size_t)blockIdx.x * DBG_TILES + ti) * DBG_F : nullptr;
}
#endif
__device__ __forceinline__ void add4(float4& a, const float4 b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }

// float offset of 16-byte piece c4 of tile row r (XOR swizzle inside aligned groups of 8 pieces: conflict-free both for
// the row-per-thread dump and for the row-major read-back)
template <int BN>
__device__ __forceinline__ int tile_slot(int r, int c4) { return r * BN + ((c4 ^ (r & 7)) << 2); }

// fp32 + optional tensor-core twins of four consecutive values
__device__ __forceinline__ void store4(float* f32, const TwinOut& tw, size_t off, const float4 v) {
  if (f32 != nullptr) *reinterpret_cast<float4*>(f32 + off) = v;
  store_twin4(tw, off, v);
}

// TMEM -> tile: the two warps of quarter q write their 32 rows, each one half of the columns
template <int BN>
__device__ __forceinline__ void tile_dump(uint32_t tlane, float* tile, int hsel, int lane, bool zero_acc, float sc) {
  constexpr int NCH = BN / 16;
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch) {
    if ((ch < NCH / 2) != (hsel == 0)) continue;
    uint32_t r[16];
    if (zero_acc) {
#pragma unroll
      for (int j = 0; j < 16; ++j) r[j] = 0u;
    } else {
      tmem_ld16(tlane + (uint32_t)(ch * 16), r);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      *reinterpret_cast<float4*>(tile + tile_slot<BN>(lane, ch * 4 + j)) =
          make_float4(__uint_as_float(r[4 * j]) * sc, __uint_as_float(r[4 * j + 1]) * sc, __uint_as_float(r[4 * j + 2]) * sc,
                      __uint_as_float(r[4 * j + 3]) * sc);
  }
}

// plain tiles: C = acc + bias + rowadd + cadd + gather, or g_t = sig(gq + acc) * tanh(c1') on the columns < gt_cols
template <int BN>
__device__ __forceinline__ void tile_plain(const TcProblem& p, const float* tile, const float* s_bias, int rowq, int n0, int te) {
  constexpr int P4 = BN / 4, ITEMS = 32 * P4 / TC_EPI_THREADS;     // 16-byte pieces per row, pieces per thread
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  // Tiles with nothing but the bias to add (GEMM-B, the h1' projection outside the g_t columns): the general loop below
  // spends ~6 k cycles per lane quarter in per-piece tests and parameter reloads, more than the 32 KB of stores it
  // issues.  Same sums in the same order (the zero addends included: x + 0 turns -0 into +0), so the results are
  // bit-identical.
  if (n0 >= p.gt_cols && p.rowadd == nullptr && p.cadd == nullptr && p.gather == nullptr) {
    float* const c = p.c;
    const int ldc = p.ldc, live = p.M - rowq;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      const int idx = te + k * TC_EPI_THREADS;
      const int r = idx / P4, c4 = idx - r * P4;
      if (r >= live) break;                // rows grow with k
      float4 o = *reinterpret_cast<const float4*>(tile + tile_slot<BN>(r, c4));
      add4(o, *reinterpret_cast<const float4*>(s_bias + 4 * c4));
      add4(o, zero); add4(o, zero); add4(o, zero);
      *reinterpret_cast<float4*>(c + (size_t)(rowq + r) * ldc + n0 + 4 * c4) = o;
    }
    return;
  }
  float4 acc[ITEMS], x0[ITEMS], x1[ITEMS], x2[ITEMS];
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {        // all loads first: one round trip for the thread's pieces
    const int idx = te + k * TC_EPI_THREADS;
    const int r = idx / P4, c4 = idx - r * P4;
    const int row = rowq + r, n = n0 + 4 * c4;
    acc[k] = *reinterpret_cast<const float4*>(tile + tile_slot<BN>(r, c4));
    x0[k] = zero; x1[k] = zero; x2[k] = zero;
    if (row < p.M) {
      if (n < p.gt_cols) {
        x0[k] = *reinterpret_cast<const float4*>(p.gt_gq + (size_t)row * p.ld_state + n);
        x1[k] = *reinterpret_cast<const float4*>(p.gt_c1n + (size_t)row * p.ld_state + n);
      } else {
        if (p.rowadd != nullptr)
          x0[k] = __ldg(reinterpret_cast<const float4*>(p.rowadd + (size_t)((row / p.row_div) * p.rowadd_mul) * p.ld_rowadd + n));
        if (p.cadd != nullptr) x1[k] = *reinterpret_cast<const float4*>(p.cadd + (size_t)row * p.ld_cadd + n);
        if (p.gather != nullptr) x2[k] = __ldg(reinterpret_cast<const float4*>(p.gather + (size_t)p.gather_idx[row] * p.ld_gather + n));
      }
    }
  }
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    const int idx = te + k * TC_EPI_THREADS;
    const int r = idx / P4, c4 = idx - r * P4;
    const int row = rowq + r, n = n0 + 4 * c4;
    if (row >= p.M) continue;
    if (n < p.gt_cols) {
      // g_t = sig(gq + W1_hg.h1') * tanh(c1')      (controllable_captioning.py:181-182)
      const float4 o = make_float4(fast_sigmoid(x0[k].x + acc[k].x) * fast_tanh(x1[k].x), fast_sigmoid(x0[k].y + acc[k].y) * fast_tanh(x1[k].y),
                                   fast_sigmoid(x0[k].z + acc[k].z) * fast_tanh(x1[k].z), fast_sigmoid(x0[k].w + acc[k].w) * fast_tanh(x1[k].w));
      store4(p.g_t, p.g_tw, (size_t)row * p.ld_state + n, o);
    } else {
      float4 o = acc[k];
      add4(o, *reinterpret_cast<const float4*>(s_bias + 4 * c4));
      add4(o, x0[k]); add4(o, x1[k]); add4(o, x2[k]);
      *reinterpret_cast<float4*>(p.c + (size_t)row * p.ldc + n) = o;
    }
  }
}

// Fused LSTM cell.  The tile's BN = NG*32 columns hold NG gates x 32 units as [gate][32 units] (cell_col()).
// LSTM1: NG = 6 (i,f,g,o | sentinel gate s | shift gate gq), LSTM2: NG = 4.  One item = 4 units of one row:
// pre = acc + bias + rowadd + cadd + gather, then the cell math of nn.LSTMCell.  256 items = one per epilogue thread.
// CH = BN / (NG * 32) 32-unit chunks per tile (2 for the 256-wide LSTM2 tiles of the CTA-pair kernel): h = chunk.
template <int BN, int NG>
__device__ __forceinline__ void tile_cell(const TcProblem& p, const float* tile, const float* s_bias, int rowq, int n0_tile, int n_tile_,
                                          int te, int h = 0) {
  static_assert(BN % (NG * 32) == 0, "whole 32-unit chunks per tile");
  constexpr int CH = BN / (NG * 32);
  const int r = te >> 3, uq = te & 7;
  const int row = rowq + r;
  if (row >= p.M) return;
  const int n_tile = n_tile_ * CH + h;          // 32-unit chunk index
  const int n0 = n0_tile + h * NG * 32;         // first output column of the chunk
  tile += 0; s_bias += h * NG * 32;
  const int cpiece = h * NG * 8;                // first 16-byte piece of the chunk inside the tile row
  const int unit = n_tile * 32 + uq * 4;
  const size_t so = (size_t)row * p.ld_state + unit;
  float4 pre[NG], x0[NG], x1[NG], x2[NG];
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#ifdef VSR_DBG_CLK
  const long long k0 = clock64();
#endif
  const float4 cold = *reinterpret_cast<const float4*>(p.c_old + so);
  const float* radd = p.rowadd != nullptr ? p.rowadd + (size_t)((row / p.row_div) * p.rowadd_mul) * p.ld_rowadd + n0 + uq * 4 : nullptr;
  const float* cadd = p.cadd != nullptr ? p.cadd + (size_t)row * p.ld_cadd + n0 + uq * 4 : nullptr;
  const float* gath = p.gather != nullptr ? p.gather + (size_t)p.gather_idx[row] * p.ld_gather + n0 + uq * 4 : nullptr;
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    pre[g] = *reinterpret_cast<const float4*>(tile + tile_slot<BN>(r, cpiece + g * 8 + uq));
    x0[g] = radd != nullptr ? __ldg(reinterpret_cast<const float4*>(radd + g * 32)) : zero;
    x1[g] = cadd != nullptr ? *reinterpret_cast<const float4*>(cadd + g * 32) : zero;
    x2[g] = gath != nullptr ? __ldg(reinterpret_cast<const float4*>(gath + g * 32)) : zero;
  }
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    add4(pre[g], *reinterpret_cast<const float4*>(s_bias + g * 32 + uq * 4));
    add4(pre[g], x0[g]); add4(pre[g], x1[g]); add4(pre[g], x2[g]);
  }
#ifdef VSR_DBG_CLK
  const long long k1 = clock64();
#endif
  const float pi[4] = {pre[0].x, pre[0].y, pre[0].z, pre[0].w}, pf[4] = {pre[1].x, pre[1].y, pre[1].z, pre[1].w};
  const float pg[4] = {pre[2].x, pre[2].y, pre[2].z, pre[2].w}, po[4] = {pre[3].x, pre[3].y, pre[3].z, pre[3].w};
  const float co[4] = {cold.x, cold.y, cold.z, cold.w};
  float cn[4], hn[4], tc[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float ig = fast_sigmoid(pi[u]), fg = fast_sigmoid(pf[u]), gg = fast_tanh(pg[u]), og = fast_sigmoid(po[u]);
    cn[u] = fg * co[u] + ig * gg;
    tc[u] = fast_tanh(cn[u]);
    hn[u] = og * tc[u];
  }
#ifdef VSR_DBG_CLK
  const long long k2 = clock64();
#endif
  *reinterpret_cast<float4*>(p.c_new + so) = make_float4(cn[0], cn[1], cn[2], cn[3]);
  store4(p.h_new, p.h_tw, so, make_float4(hn[0], hn[1], hn[2], hn[3]));
  if constexpr (NG == 6) {
    const float ps[4] = {pre[4].x, pre[4].y, pre[4].z, pre[4].w};
    store4(p.s_new, p.s_tw, so, make_float4(fast_sigmoid(ps[0]) * tc[0], fast_sigmoid(ps[1]) * tc[1],
                                                     fast_sigmoid(ps[2]) * tc[2], fast_sigmoid(ps[3]) * tc[3]));
    *reinterpret_cast<float4*>(p.gq + so) = pre[5];
  }
#ifdef VSR_DBG_CLK
  if ((te == 0 || te == 200) && blockIdx.x == 5 && p.M > 200 && (rowq & 127) == 0)
    printf("cell NG=%d te=%d: loads+adds %lld math %lld stores %lld\n", NG, te, k1 - k0, k2 - k1, clock64() - k2);
#endif
}

// all eight epilogue warps: quarter by quarter, dump -> barrier -> cooperative pass -> barrier
template <int BN>
__device__ __forceinline__ void tile_epilogue(const TcProblem& p, uint32_t tmem_base, int m0, int n0, int n_tile, int warp, int lane,
                                              const float* s_bias, float* tile, long long* clk = nullptr) {
  const int q = warp & 3, hsel = (warp - 2) >> 2, te = (warp - 2) * 32 + lane;
  const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
  const float sc = (p.acc_scale != nullptr ? __ldg(p.acc_scale) : 1.f) * p.act_inv;
#pragma unroll 1
  for (int qq = 0; qq < 4; ++qq) {
    if (m0 + qq * 32 >= p.M) break;                 // no live row in this or any later quarter (uniform)
#ifdef VSR_DBG_CLK
    const long long c0 = clock64();
#endif
    if (q == qq) tile_dump<BN>(tlane, tile, hsel, lane, p.zero_acc != 0, sc);
#ifdef VSR_DBG_CLK
    const long long c1 = clock64();
#endif
    epi_bar(3);
#ifdef VSR_DBG_CLK
    const long long c2 = clock64();
#endif
    const int rowq = m0 + qq * 32;
    if (p.mode == EPI_PLAIN) tile_plain<BN>(p, tile, s_bias, rowq, n0, te);
    if constexpr (BN == 192) { if (p.mode == EPI_LSTM1) tile_cell<BN, 6>(p, tile, s_bias, rowq, n0, n_tile, te); }
    if constexpr (BN == 128) { if (p.mode == EPI_LSTM2) tile_cell<BN, 4>(p, tile, s_bias, rowq, n0, n_tile, te); }
    if constexpr (BN == 256) {
      if (p.mode == EPI_LSTM2) { tile_cell<BN, 4>(p, tile, s_bias, rowq, n0, n_tile, te, 0); tile_cell<BN, 4>(p, tile, s_bias, rowq, n0, n_tile, te, 1); }
    }
#ifdef VSR_DBG_CLK
    const long long c3 = clock64();
#endif
    epi_bar(4);
#ifdef VSR_DBG_CLK
    if (clk != nullptr && warp == 2 && lane == 0) {    // warp 2 dumps quarter 2; in the others its bar(3) wait is the dump
      long long* q4 = clk + DBG_Q + 4 * qq;
      q4[0] = c1 - c0; q4[1] = c2 - c1; q4[2] = c3 - c2; q4[3] = clock64() - c3;
    }
#endif
  }
}

// Vocabulary-head epilogue: besides storing the logits (acc + bias) the thread that owns a row reduces every 16-column
// chunk of its BN columns to a record {max, sum exp(x - max)}.  k_vocab_merge (vocab_head.cuh: merge_row) finishes
// log-softmax and top-k from the chunk records and re-reads only the few chunks that can hold a top-k element, so the
// 20 MB logits tensor is written but never scanned.  Records are per CHUNK, not per tile: the row's log-sum-exp (and
// with it every returned log-prob) does not depend on the N tile of the launch, i.e. on the batch size or on which
// kernel variant ran (bit-exact caption independence, stacked decodes).
template <int BN>
__device__ __forceinline__ void vocab_epilogue(const TcProblem& p, uint32_t tlane, int row, bool live, int n0,
                                               const float* s_bias, int hsel) {
  constexpr int NCH = BN / 16, H0 = (NCH + 1) / 2;      // chunks [0, H0) -> first warp of the quarter, [H0, NCH) -> second
  float* crow = p.c + (size_t)row * p.ldc;
  float2* rec = reinterpret_cast<float2*>(p.vpart) + (size_t)row * (p.ldc / 16) + n0 / 16;
  const float sc = (p.acc_scale != nullptr ? __ldg(p.acc_scale) : 1.f) * p.act_inv;
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch) {
    if ((ch < H0) != (hsel == 0)) continue;
    uint32_t r[16];
    tmem_ld16(tlane + (uint32_t)(ch * 16), r);
    const int n = n0 + ch * 16;
    if (live) {
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const float4 b = *reinterpret_cast<const float4*>(s_bias + ch * 16 + j);
        v[j] = __uint_as_float(r[j]) * sc + b.x; v[j + 1] = __uint_as_float(r[j + 1]) * sc + b.y;
        v[j + 2] = __uint_as_float(r[j + 2]) * sc + b.z; v[j + 3] = __uint_as_float(r[j + 3]) * sc + b.w;
        *reinterpret_cast<float4*>(crow + n + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      }
      if (n + 16 > p.n_valid) {
#pragma unroll
        for (int j = 0; j < 16; ++j) if (n + j >= p.n_valid) v[j] = -INFINITY;
      }
      float cm = fmaxf(fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])), fmaxf(fmaxf(v[4], v[5]), fmaxf(v[6], v[7])));
      cm = fmaxf(cm, fmaxf(fmaxf(fmaxf(v[8], v[9]), fmaxf(v[10], v[11])), fmaxf(fmaxf(v[12], v[13]), fmaxf(v[14], v[15]))));
      float cs = 0.f;
      if (cm > -INFINITY) {
        float e0 = 0.f, e1 = 0.f, e2 = 0.f, e3 = 0.f;     // exp(-inf) = 0 on masked columns
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          e0 += __expf(v[j] - cm); e1 += __expf(v[j + 1] - cm); e2 += __expf(v[j + 2] - cm); e3 += __expf(v[j + 3] - cm);
        }
        cs = (e0 + e1) + (e2 + e3);
      }
      rec[ch] = make_float2(cm, cs);
    }
  }
}

// Before the accumulator is complete (i.e. behind the main loop), by all epilogue warps: the tile's bias -> shared
// memory, and for the fused cell epilogues an L2 prefetch of the per-row operands the four quarter passes will read.
// The per-word rows of GEMM-A come out of a 246 MB table (one random 768-byte segment per row and tile): a cold
// read costs ~2 us per pass (HBM + TLB miss) when it is first touched inside the pass.
template <int BN>
__device__ __forceinline__ void epi_bias(const TcProblem& p, int m0, int n0, int n_tile, int warp, int lane, float* s_bias,
                                         bool reuse) {
  if (reuse) epi_bar(1);                             // previous tile's readers are done
  const int te = (warp - 2) * 32 + lane;
  for (int i = te; i < BN; i += TC_EPI_THREADS) s_bias[i] = p.bias != nullptr ? __ldg(p.bias + n0 + i) : 0.f;
  if (p.mode == EPI_LSTM1 || p.mode == EPI_LSTM2) {
    const int r = te >> 3, g = te & 7;               // thread (row, gate): one 128-byte line per quarter pass
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) {
      const int row = m0 + qq * 32 + r;
      if (row >= p.M) break;
      const float* line = nullptr;
      if (g < BN / 32) {
        if (p.gather != nullptr) line = p.gather + (size_t)p.gather_idx[row] * p.ld_gather + n0 + g * 32;
      } else if (g == 6) {
        line = p.c_old + (size_t)row * p.ld_state + n_tile * 32;
      } else if (p.rowadd != nullptr) {
        line = p.rowadd + (size_t)((row / p.row_div) * p.rowadd_mul) * p.ld_rowadd + n0;     // first of the caption row's lines
      }
      if (line != nullptr) asm volatile("prefetch.global.L2 [%0];" ::"l"(line));
    }
  }
  epi_bar(1);
}

// row-per-thread plain epilogue (tiles without a staging buffer, and the CTA-pair experiment); `nsplit` warps share a
// TMEM lane quarter and take the column chunks [hsel * NCH / nsplit, ...)
template <int BN>
__device__ __forceinline__ void rowwise_plain(const TcProblem& p, uint32_t tmem_base, int m0, int n0, int warp, int lane,
                                              int hsel, int nsplit) {
  const int q = warp & 3;
  const int row = m0 + q * 32 + lane;
  const bool live = row < p.M;
  const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
  const float* radd = (p.rowadd != nullptr && live)
                          ? p.rowadd + (size_t)((row / p.row_div) * p.rowadd_mul) * p.ld_rowadd : nullptr;
  const float* cadd = (p.cadd != nullptr && live) ? p.cadd + (size_t)row * p.ld_cadd : nullptr;
  const float* gath = (p.gather != nullptr && live) ? p.gather + (size_t)p.gather_idx[row] * p.ld_gather : nullptr;
  float* crow = p.c + (size_t)row * p.ldc;
  constexpr int NCH = BN / 16;
  const float sc = (p.acc_scale != nullptr ? __ldg(p.acc_scale) : 1.f) * p.act_inv;
  const int c_lo = hsel * NCH / nsplit, c_hi = (hsel + 1) * NCH / nsplit;
#pragma unroll 1
  for (int ch = c_lo; ch < c_hi; ++ch) {       // 16 accumulator columns per TMEM load: any BN % 16 == 0
    uint32_t r[16];
    tmem_ld16(tlane + (uint32_t)(ch * 16), r);
    const int n = n0 + ch * 16;
    if (!live) continue;
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
      float4 o = make_float4(__uint_as_float(r[j]) * sc, __uint_as_float(r[j + 1]) * sc, __uint_as_float(r[j + 2]) * sc,
                             __uint_as_float(r[j + 3]) * sc);
      if (p.bias != nullptr) add4(o, __ldg(reinterpret_cast<const float4*>(p.bias + n + j)));
      if (radd != nullptr) add4(o, __ldg(reinterpret_cast<const float4*>(radd + n + j)));
      if (cadd != nullptr) add4(o, *reinterpret_cast<const float4*>(cadd + n + j));
      if (gath != nullptr) add4(o, __ldg(reinterpret_cast<const float4*>(gath + n + j)));
      *reinterpret_cast<float4*>(crow + n + j) = o;
    }
  }
}

// epilogue of the single-CTA kernels (eight epilogue warps)
template <int BN, int KB>
__device__ __forceinline__ void tc_epilogue(const TcProblem& p, uint32_t tmem_base, int m0, int n0, int n_tile,
                                            int warp, int lane, const float* s_bias, float* tile) {
  using Cfg = TcCfg<BN, KB>;
  const int q = warp & 3, hsel = (warp - 2) >> 2;
  if (p.mode == EPI_VOCAB) {
    const int row = m0 + q * 32 + lane;
    vocab_epilogue<BN>(p, tmem_base + ((uint32_t)(q * 32) << 16), row, row < p.M, n0, s_bias, hsel);
  } else if constexpr (Cfg::kTileEpi) {
    tile_epilogue<BN>(p, tmem_base, m0, n0, n_tile, warp, lane, s_bias, tile);
  } else {
    rowwise_plain<BN>(p, tmem_base, m0, n0, warp, lane, hsel, 2);     // host: plain mode only on these tiles
  }
}

// ---------------------------------------------------------------- one ring stage: operand loads and MMA issue
// Stage layout (same bytes in both modes): A hi16 | A second half | W hi16 | W second half, where the second half is
// the fp16 residual tile (f16x3) or the two e4m3 tiles hi8 | lo8 (f16+f8x2).
template <int BN, int KB>
__device__ __forceinline__ void load_w_stage(const TcProblem& p, uint64_t* bar, uint8_t* base, int kb, int n0) {
  using Cfg = TcCfg<BN, KB>;
  uint8_t* w = base + 2 * Cfg::kABytes;
  tma_load_2d(&p.w_hi, bar, w, kb * KB, n0);
  if (p.f8) {
    tma_load_2d(&p.w_h8, bar, w + Cfg::kWBytes, kb * KB, n0);
    tma_load_2d(&p.w_lo, bar, w + Cfg::kWBytes + Cfg::kWBytes / 2, kb * KB, n0);
  } else {
    tma_load_2d(&p.w_lo, bar, w + Cfg::kWBytes, kb * KB, n0);
  }
}
template <int BN, int KB>
__device__ __forceinline__ void load_a_stage(const TcProblem& p, uint64_t* bar, uint8_t* base, int seg, int kk, int m0) {
  using Cfg = TcCfg<BN, KB>;
  tma_load_2d(&p.a_hi[seg], bar, base, kk * KB, m0);
  if (p.f8) {
    tma_load_2d(&p.a_h8[seg], bar, base + Cfg::kABytes, kk * KB, m0);
    tma_load_2d(&p.a_lo[seg], bar, base + Cfg::kABytes + Cfg::kABytes / 2, kk * KB, m0);
  } else {
    tma_load_2d(&p.a_lo[seg], bar, base + Cfg::kABytes, kk * KB, m0);
  }
}
// the MMAs of one k-block into the accumulator at tmem_acc (first = the k-block overwrites instead of accumulating)
template <int BN, int KB>
__device__ __forceinline__ void issue_stage(const TcProblem& p, uint32_t tmem_acc, uint32_t base, bool first) {
  using Cfg = TcCfg<BN, KB>;
  constexpr uint32_t idesc = make_idesc<BN>();
  const uint64_t ah = make_kmajor_desc<KB>(base), wh = make_kmajor_desc<KB>(base + 2 * Cfg::kABytes);
  if (p.f8) {
    // x_hi*w_hi on the fp16 path; x_hi8*w_lo8 + x_lo8*w_hi8 on the fp8 path (K = 32 per instruction, twice the rate)
    const uint64_t a8 = make_kmajor_desc8<KB>(base + Cfg::kABytes), al = make_kmajor_desc8<KB>(base + Cfg::kABytes + Cfg::kABytes / 2);
    const uint64_t w8 = make_kmajor_desc8<KB>(base + 2 * Cfg::kABytes + Cfg::kWBytes);
    const uint64_t wl = make_kmajor_desc8<KB>(base + 2 * Cfg::kABytes + Cfg::kWBytes + Cfg::kWBytes / 2);
#pragma unroll
    for (int k = 0; k < KB / UMMA_K; ++k) {
      const uint64_t off = (uint64_t)((k * UMMA_K * 2) >> 4);     // 32 bytes inside the swizzle row
      umma_f16(tmem_acc, ah + off, wh + off, idesc, (first && k == 0) ? 0u : 1u);
    }
#pragma unroll
    for (int k = 0; k < KB / 32; ++k) {
      const uint64_t off = (uint64_t)((k * 32) >> 4);             // 32 e4m3 = 32 bytes
      umma_f8(tmem_acc, a8 + off, wl + off, idesc, 1u);
      umma_f8(tmem_acc, al + off, w8 + off, idesc, 1u);
    }
  } else {
    const uint64_t al = make_kmajor_desc<KB>(base + Cfg::kABytes), wl = make_kmajor_desc<KB>(base + 2 * Cfg::kABytes + Cfg::kWBytes);
#pragma unroll
    for (int k = 0; k < KB / UMMA_K; ++k) {
      const uint64_t off = (uint64_t)((k * UMMA_K * 2) >> 4);     // advance inside the swizzle row
      umma_f16(tmem_acc, ah + off, wh + off, idesc, (first && k == 0) ? 0u : 1u);
      umma_f16(tmem_acc, ah + off, wl + off, idesc, 1u);
      umma_f16(tmem_acc, al + off, wh + off, idesc, 1u);
    }
  }
}

template <int BN, int KB>
__global__ void __launch_bounds__(TC_THREADS, 1) k_gemm_tc(const __grid_constant__ TcParams params) {
  using Cfg = TcCfg<BN, KB>;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[Cfg::kStages];
  __shared__ __align__(8) uint64_t empty_bar[Cfg::kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float s_bias[BN];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // tile of this CTA: problems back to back; consecutive CTAs walk the M tiles of one W tile (L2 reuse)
  int t = blockIdx.x;
  const int tiles0 = params.pr[0].n_tiles * params.pr[0].m_tiles;
  const int pi = (params.nprob > 1 && t >= tiles0) ? 1 : 0;
  t -= pi * tiles0;
  const TcProblem& p = params.pr[pi];
  const int m_tile = t % p.m_tiles, n_tile = t / p.m_tiles;
  const int m0 = m_tile * BM, n0 = n_tile * BN;

  if (!(params.pdl_flags & 2)) pdl_trigger();
  if (p.row_skip != nullptr) {   // all-padding row tiles produce nothing (block-uniform)
    pdl_wait();                  // the flags come from the previous kernel
    int any = 0;
    if (threadIdx.x < BM && m0 + (int)threadIdx.x < p.M) any = p.row_skip[m0 + threadIdx.x];
    if (!__syncthreads_or(any)) return;
  }

  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);   // SW128 needs 1024-B alignment

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.nseg; ++s) { prefetch_tmap(&p.a_hi[s]); prefetch_tmap(&p.a_lo[s]); if (p.f8) prefetch_tmap(&p.a_h8[s]); }
    prefetch_tmap(&p.w_hi); prefetch_tmap(&p.w_lo); if (p.f8) prefetch_tmap(&p.w_h8);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      mbar_init(&tmem_full_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(Cfg::kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;

  int total_kb = 0;
  for (int s = 0; s < p.nseg; ++s) total_kb += p.kblocks[s];

  if (p.zero_acc) total_kb = 0;          // operands known to be zero: nothing to load or multiply

  if (warp == 0) {
    if (lane == 0) {
      // the WEIGHT halves of the first ring pass do not depend on the previous kernel: fetch them, then wait
      const int pre = !(params.pdl_flags & 1) ? 0 : (total_kb < Cfg::kStages ? total_kb : Cfg::kStages);
      for (int kb = 0; kb < pre; ++kb) {
        mbar_expect_tx(&full_bar[kb], Cfg::kStageBytes);
        load_w_stage<BN, KB>(p, &full_bar[kb], smem + kb * Cfg::kStageBytes, kb, n0);
      }
      pdl_wait();
      int seg = 0, kk = 0;
      for (int kb = 0; kb < total_kb; ++kb) {
        const int st = kb % Cfg::kStages;
        const uint32_t ph = (kb / Cfg::kStages) & 1;
        uint8_t* base = smem + st * Cfg::kStageBytes;
        if (kb >= pre) {
          mbar_wait(&empty_bar[st], ph ^ 1);
          mbar_expect_tx(&full_bar[st], Cfg::kStageBytes);
          load_w_stage<BN, KB>(p, &full_bar[st], base, kb, n0);
        }
        load_a_stage<BN, KB>(p, &full_bar[st], base, seg, kk, m0);
        if (++kk == p.kblocks[seg]) { kk = 0; ++seg; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      for (int kb = 0; kb < total_kb; ++kb) {
        const int st = kb % Cfg::kStages;
        const uint32_t ph = (kb / Cfg::kStages) & 1;
        mbar_wait(&full_bar[st], ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        issue_stage<BN, KB>(p, tmem_base, smem_u32(smem + st * Cfg::kStageBytes), kb == 0);
        umma_commit(&empty_bar[st]);          // frees the smem slot once these MMAs have read it
      }
      umma_commit(&tmem_full_bar);            // accumulator complete -> epilogue
      if (params.pdl_flags & 2) pdl_trigger();
    }
    __syncwarp();
  } else {
    pdl_wait();
#ifdef VSR_DBG_CLK
    const long long tk0 = clock64();
#endif
    epi_bias<BN>(p, m0, n0, n_tile, warp, lane, s_bias, false);
    mbar_wait(&tmem_full_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#ifdef VSR_DBG_CLK
    const long long tk1 = clock64();
#endif
    tc_epilogue<BN, KB>(p, tmem_base, m0, n0, n_tile, warp, lane, s_bias, reinterpret_cast<float*>(smem + Cfg::kRingBytes));
#ifdef VSR_DBG_CLK
    if (lane == 0 && warp == 2 && (blockIdx.x == 5 || blockIdx.x == 100) && p.M > 200)
      printf("gemm BN=%d KB=%d grid=%d cta=%d mode=%d kblocks=%d: main loop %lld cyc, epilogue %lld cyc\n", BN, KB, (int)gridDim.x,
             (int)blockIdx.x, p.mode, total_kb, tk1 - tk0, clock64() - tk1);
#endif
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::kTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------- persistent variant
// One CTA per SM walks the tile list (tile = blockIdx.x + i * gridDim.x).  The smem ring keeps running
// across tiles and the accumulator is double-buffered in TMEM, so the epilogue of tile i (TMEM -> registers
// -> global, incl. the fused LSTM / gate math) overlaps the TMA + MMA main loop of tile i+1, and the
// per-CTA set-up (barrier init, TMEM allocation, descriptor prefetch, pipeline fill) is paid once.
__device__ __forceinline__ bool tile_all_padding(const uint8_t* row_skip, int m0, int M, int lane) {
  if (row_skip == nullptr) return false;
  int any = 0;
  for (int r = lane; r < BM; r += 32) if (m0 + r < M) any |= row_skip[m0 + r];
  return !__any_sync(0xffffffffu, any);
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int BN, int KB>
__global__ void __launch_bounds__(TC_THREADS, 1) k_gemm_tcp(const __grid_constant__ TcParams params) {
  using Cfg = TcCfg<BN, KB>;
  constexpr int kAccCols = (BN <= 128) ? 128 : 256;     // TMEM column stride between the two accumulators
  constexpr int kTmemCols = 2 * kAccCols;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[Cfg::kStages];
  __shared__ __align__(8) uint64_t empty_bar[Cfg::kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float s_bias[BN];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles0 = params.pr[0].n_tiles * params.pr[0].m_tiles;
  const int total_tiles = tiles0 + (params.nprob > 1 ? params.pr[1].n_tiles * params.pr[1].m_tiles : 0);
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);

  if (!(params.pdl_flags & 2)) pdl_trigger();
  bool pdl_waited = false;
  for (int q = 0; q < params.nprob; ++q)
    if (params.pr[q].row_skip != nullptr) pdl_waited = true;     // tile skipping reads the previous kernel's flags
  if (pdl_waited || warp >= 2) pdl_wait();                        // epilogue warps: before any global access
  if (warp == 0 && lane == 0) {
    for (int q = 0; q < params.nprob; ++q) {
      const TcProblem& p = params.pr[q];
      for (int s = 0; s < p.nseg; ++s) { prefetch_tmap(&p.a_hi[s]); prefetch_tmap(&p.a_lo[s]); if (p.f8) prefetch_tmap(&p.a_h8[s]); }
      prefetch_tmap(&p.w_hi); prefetch_tmap(&p.w_lo); if (p.f8) prefetch_tmap(&p.w_h8);
    }
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full_bar[s], 1); mbar_init(&tmem_empty_bar[s], TC_EPI_WARPS); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;

  // every role walks the same tile list and skips the same (all-padding) tiles
  int it = 0;        // running k-block counter -> smem ring stage / phase
  int ti = 0;        // running (non-skipped) tile counter -> accumulator buffer / phase
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    const int pi = (params.nprob > 1 && tile >= tiles0) ? 1 : 0;
    const int t = tile - pi * tiles0;
    const TcProblem& p = params.pr[pi];
    const int m_tile = t % p.m_tiles, n_tile = t / p.m_tiles;
    const int m0 = m_tile * BM, n0 = n_tile * BN;
    if (tile_all_padding(p.row_skip, m0, p.M, lane)) continue;
    int total_kb = 0;
    for (int s = 0; s < p.nseg; ++s) total_kb += p.kblocks[s];
    const int acc = ti & 1;
    const uint32_t aph = (ti >> 1) & 1;
    const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * kAccCols);

    if (warp == 0) {
      if (lane == 0) {
        // first tile of this CTA: weight halves of the first ring pass before the dependency wait (see k_gemm_tc)
        int pre = 0;
        if (!pdl_waited) {
          pre = !(params.pdl_flags & 1) ? 0 : (total_kb < Cfg::kStages ? total_kb : Cfg::kStages);
          for (int kb = 0; kb < pre; ++kb) {
            mbar_expect_tx(&full_bar[kb], Cfg::kStageBytes);
            load_w_stage<BN, KB>(p, &full_bar[kb], smem + kb * Cfg::kStageBytes, kb, n0);
          }
          pdl_wait();
          pdl_waited = true;
        }
        int seg = 0, kk = 0;
        for (int kb = 0; kb < total_kb; ++kb) {
          const int st = (it + kb) % Cfg::kStages;
          const uint32_t ph = ((it + kb) / Cfg::kStages) & 1;
          uint8_t* base = smem + st * Cfg::kStageBytes;
          if (kb >= pre) {
            mbar_wait(&empty_bar[st], ph ^ 1);
            mbar_expect_tx(&full_bar[st], Cfg::kStageBytes);
            load_w_stage<BN, KB>(p, &full_bar[st], base, kb, n0);
          }
          load_a_stage<BN, KB>(p, &full_bar[st], base, seg, kk, m0);
          if (++kk == p.kblocks[seg]) { kk = 0; ++seg; }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      if (lane == 0) {
        mbar_wait(&tmem_empty_bar[acc], aph ^ 1);       // the epilogue has drained this accumulator
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        for (int kb = 0; kb < total_kb; ++kb) {
          const int st = (it + kb) % Cfg::kStages;
          const uint32_t ph = ((it + kb) / Cfg::kStages) & 1;
          mbar_wait(&full_bar[st], ph);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          issue_stage<BN, KB>(p, tmem_acc, smem_u32(smem + st * Cfg::kStageBytes), kb == 0);
          umma_commit(&empty_bar[st]);
        }
        umma_commit(&tmem_full_bar[acc]);
        if ((params.pdl_flags & 2) && tile + (int)gridDim.x >= total_tiles) pdl_trigger();   // last tile of this CTA
      }
      __syncwarp();
    } else {
      epi_bias<BN>(p, m0, n0, n_tile, warp, lane, s_bias, ti != 0);
      mbar_wait(&tmem_full_bar[acc], aph);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      tc_epilogue<BN, KB>(p, tmem_acc, m0, n0, n_tile, warp, lane, s_bias, reinterpret_cast<float*>(smem + Cfg::kRingBytes));
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);   // every epilogue warp -> accumulator free again
    }
    it += total_kb;
    ++ti;
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// x -> (fp16 hi, fp16 lo) with lo = fp16(x - hi)
// ---------------------------------------------------------------- CTA-pair kernel (cta_group::2), persistent
// What bounds the single-CTA kernels once the batch is large (ncu on the stacked 400-caption decode: tensor pipe 40-45 %
// active, L2 -> SM 10-12 TB/s) is operand delivery: a 128 x 128 tile pulls (128 + 128) x KB x 4 bytes through L2 and
// shared memory per k-block, whichever passes are issued.  Here the two CTAs of a cluster (one TPC) compute a 256 x BN
// tile: each stages its own 128 rows of A and HALF of the W tile (BN / 2 rows); the leader issues tcgen05.mma
// .cta_group::2 (M = 256), which reads both CTAs' shared memory, and each CTA ends up with its 128 x BN accumulator in
// its own TMEM.  Bytes per output element halve (BN = 256), which is also what lets the e4m3 residual MMAs run near their
// rate.  Persistent (one cluster per TPC walks the tile list), accumulators double-buffered in TMEM (2 x 256 columns), the
// same shared-memory-tile epilogues as the single-CTA kernels (plain / g_t / LSTM cell 1 at BN = 192 / LSTM cell 2 at 256).
// VOCAB: the row-per-thread vocabulary epilogue needs no shared-memory tile, which buys one more stage (measured: -2 %).
// (32-element k-blocks — the same ring bytes in twice as many, finer stages — were measured SLOWER for the fp16-only
// GEMM-A: 201 vs 179 us on the M=1900, N=6144, K=3072 self-test shape; KB_ stays 64.)
template <int BN, int KB_ = 64, bool VOCAB = false> struct PairCfg {
  static constexpr int KB = KB_;
  static constexpr int kABytes = BM * KB * 2;                 // fp16 tile of this CTA's 128 A rows (the second half of the
  static constexpr int kWBytes = (BN / 2) * KB * 2;           //   stage holds lo16, or hi8 | lo8); this CTA's half of the W tile
  static constexpr int kStageBytes = 2 * kABytes + 2 * kWBytes;
  static constexpr int kEpiBytes = VOCAB ? 0 : 32 * BN * 4;
  static constexpr int kStages = (227 * 1024 - 2048 - 1024 - kEpiBytes) / kStageBytes;      // (2 KB: static shared memory)
  static constexpr int kRingBytes = kStages * kStageBytes;
  static constexpr int kSmemBytes = kRingBytes + 1024 + kEpiBytes;
  static constexpr int kAccCols = 256, kTmemCols = 512;
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive (count 1) on the same mbarrier of CTA `rank` of this cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}
// TMA load whose completion bytes are credited to the LEADER CTA's mbarrier (peer bit of the address cleared)
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_f8_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// commit: arrive on the same mbarrier in BOTH CTAs of the pair once the issued MMAs have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
template <int BN> __device__ __forceinline__ constexpr uint32_t make_idesc_pair() {   // M = 256
  return (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}

template <int BN, int KB_, bool VOCAB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1) k_gemm_pair(const __grid_constant__ TcParams params) {
  using Cfg = PairCfg<BN, KB_, VOCAB>;
  constexpr int KB = Cfg::KB;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[Cfg::kStages];       // waited on in the leader CTA only
  __shared__ __align__(8) uint64_t empty_bar[Cfg::kStages];      // per CTA, signalled by the leader's multicast commits
  __shared__ __align__(8) uint64_t tmem_full_bar[2];             // per CTA, likewise
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];            // leader's: 2 x 8 epilogue warps arrive (peer's remotely)
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float s_bias[BN];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();                       // 0 = leader (issues the MMAs), 1 = peer
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
  const int mp0 = (params.pr[0].m_tiles + 1) >> 1;
  const int tiles0 = params.pr[0].n_tiles * mp0;
  const int total_tiles = tiles0 + (params.nprob > 1 ? params.pr[1].n_tiles * ((params.pr[1].m_tiles + 1) >> 1) : 0);
  // 1 KB-aligned by pointer arithmetic on smem_raw (not through an integer): the epilogue's staging-tile accesses then
  // compile to shared-memory loads / stores instead of generic ones
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

  pdl_trigger();
  pdl_wait();                       // (no early weight prefetch here: multi-wave launches hide the set-up anyway)
  if (warp == 0 && lane == 0) {
    for (int q = 0; q < params.nprob; ++q) {
      const TcProblem& p = params.pr[q];
      for (int s = 0; s < p.nseg; ++s) { prefetch_tmap(&p.a_hi[s]); prefetch_tmap(&p.a_lo[s]); if (p.f8) prefetch_tmap(&p.a_h8[s]); }
      prefetch_tmap(&p.w_hi); prefetch_tmap(&p.w_lo); if (p.f8) prefetch_tmap(&p.w_h8);
    }
  }
  if (warp == 1) {
    if (lane == 0) {
      // full: ONE arrival (the leader's expect_tx, which announces both CTAs' bytes); the peer's loads are accounted for
      // by their complete_tx on the leader's barrier alone (a remote release-arrive per stage measured ~2x slower)
      for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full_bar[s], 1); mbar_init(&tmem_empty_bar[s], 2 * TC_EPI_WARPS); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(Cfg::kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync_all();               // barriers of both CTAs initialised, TMEM allocated in both
  __syncthreads();                  // (the cluster barrier already orders the allocator's write of tmem_base_slot; this one is
                                    //  what compute-sanitizer's racecheck recognises)
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;

  int it = 0;        // running k-block counter -> smem ring stage / phase
  int ti = 0;        // running tile counter -> accumulator buffer / phase
  for (int tile = cluster_id; tile < total_tiles; tile += n_clusters) {
    const int pi = (params.nprob > 1 && tile >= tiles0) ? 1 : 0;
    const int t = tile - pi * tiles0;
    const TcProblem& p = params.pr[pi];
    const int m_pairs = (p.m_tiles + 1) >> 1;
    const int m_pair = t % m_pairs, n_tile = t / m_pairs;
    const int m0 = (m_pair * 2 + (int)rank) * BM, n0 = n_tile * BN;
    int total_kb = 0;
    for (int s = 0; s < p.nseg; ++s) total_kb += p.kblocks[s];
    const int acc = ti & 1;
    const uint32_t aph = (ti >> 1) & 1;
    const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * Cfg::kAccCols);

    if (warp == 0) {
      if (lane == 0) {
        const int wrow = n0 + (int)rank * (BN / 2);     // this CTA's half of the W tile
        int seg = 0, kk = 0;
        for (int kb = 0; kb < total_kb; ++kb) {
          const int st = (it + kb) % Cfg::kStages;
          const uint32_t ph = ((it + kb) / Cfg::kStages) & 1;
          mbar_wait(&empty_bar[st], ph ^ 1);
          uint8_t* base = smem + st * Cfg::kStageBytes;
          uint8_t* wb = base + 2 * Cfg::kABytes;
          if (rank == 0) mbar_expect_tx(&full_bar[st], 2 * Cfg::kStageBytes);   // both CTAs' bytes land on the leader's barrier
          tma_load_2d_pair(&p.a_hi[seg], &full_bar[st], base, kk * KB, m0);
          tma_load_2d_pair(&p.w_hi, &full_bar[st], wb, kb * KB, wrow);
          if (p.f8) {
            tma_load_2d_pair(&p.a_h8[seg], &full_bar[st], base + Cfg::kABytes, kk * KB, m0);
            tma_load_2d_pair(&p.a_lo[seg], &full_bar[st], base + Cfg::kABytes + Cfg::kABytes / 2, kk * KB, m0);
            tma_load_2d_pair(&p.w_h8, &full_bar[st], wb + Cfg::kWBytes, kb * KB, wrow);
            tma_load_2d_pair(&p.w_lo, &full_bar[st], wb + Cfg::kWBytes + Cfg::kWBytes / 2, kb * KB, wrow);
          } else {
            tma_load_2d_pair(&p.a_lo[seg], &full_bar[st], base + Cfg::kABytes, kk * KB, m0);
            tma_load_2d_pair(&p.w_lo, &full_bar[st], wb + Cfg::kWBytes, kb * KB, wrow);
          }
          if (++kk == p.kblocks[seg]) { kk = 0; ++seg; }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      if (lane == 0 && rank == 0) {
        constexpr uint32_t idesc = make_idesc_pair<BN>();
#ifdef VSR_DBG_CLK
        long long* clk = dbg_rec(ti);
        const long long m0c = clock64();
        long long mfull = 0;
#endif
        mbar_wait(&tmem_empty_bar[acc], aph ^ 1);       // both CTAs' epilogues have drained this accumulator
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#ifdef VSR_DBG_CLK
        const long long m1c = clock64();
#endif
        for (int kb = 0; kb < total_kb; ++kb) {
          const int st = (it + kb) % Cfg::kStages;
          const uint32_t ph = ((it + kb) / Cfg::kStages) & 1;
#ifdef VSR_DBG_CLK
          const long long f0 = clock64();
#endif
          mbar_wait(&full_bar[st], ph);
#ifdef VSR_DBG_CLK
          mfull += clock64() - f0;
#endif
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t base = smem_u32(smem + st * Cfg::kStageBytes);
          const uint32_t wbase = base + 2 * Cfg::kABytes;
          const uint64_t ah = make_kmajor_desc<KB>(base), wh = make_kmajor_desc<KB>(wbase);
          if (p.f8) {
            const uint64_t a8 = make_kmajor_desc8<KB>(base + Cfg::kABytes), al = make_kmajor_desc8<KB>(base + Cfg::kABytes + Cfg::kABytes / 2);
            const uint64_t w8 = make_kmajor_desc8<KB>(wbase + Cfg::kWBytes), wl = make_kmajor_desc8<KB>(wbase + Cfg::kWBytes + Cfg::kWBytes / 2);
#pragma unroll
            for (int k = 0; k < KB / UMMA_K; ++k) {
              const uint64_t off = (uint64_t)((k * UMMA_K * 2) >> 4);
              umma_f16_pair(tmem_acc, ah + off, wh + off, idesc, (kb | k) != 0 ? 1u : 0u);
            }
#pragma unroll
            for (int k = 0; k < KB / 32; ++k) {
              const uint64_t off = (uint64_t)((k * 32) >> 4);
              umma_f8_pair(tmem_acc, a8 + off, wl + off, idesc, 1u);
              umma_f8_pair(tmem_acc, al + off, w8 + off, idesc, 1u);
            }
          } else {
            const uint64_t al = make_kmajor_desc<KB>(base + Cfg::kABytes), wl = make_kmajor_desc<KB>(wbase + Cfg::kWBytes);
#pragma unroll
            for (int k = 0; k < KB / UMMA_K; ++k) {
              const uint64_t off = (uint64_t)((k * UMMA_K * 2) >> 4);
              umma_f16_pair(tmem_acc, ah + off, wh + off, idesc, (kb | k) != 0 ? 1u : 0u);
              umma_f16_pair(tmem_acc, ah + off, wl + off, idesc, 1u);
              umma_f16_pair(tmem_acc, al + off, wh + off, idesc, 1u);
            }
          }
          umma_commit_pair(&empty_bar[st]);     // frees this stage in BOTH CTAs
        }
        umma_commit_pair(&tmem_full_bar[acc]);  // accumulators complete in both CTAs -> epilogues
#ifdef VSR_DBG_CLK
        if (clk != nullptr) { clk[DBG_M0] = m0c; clk[DBG_M1] = m1c; clk[DBG_M2] = clock64(); clk[DBG_MFULL] = mfull; }
#endif
      }
      __syncwarp();
    } else {
      // bias of the tile -> shared memory behind the main loop
#ifdef VSR_DBG_CLK
      long long* clk = (warp == 2 && lane == 0) ? dbg_rec(ti) : nullptr;
      const long long e0c = clock64();
#endif
      if (ti != 0) epi_bar(1);                  // previous tile's readers are done
      for (int i = (warp - 2) * 32 + lane; i < BN; i += TC_EPI_THREADS) s_bias[i] = p.bias != nullptr ? __ldg(p.bias + n0 + i) : 0.f;
      epi_bar(1);
#ifdef VSR_DBG_CLK
      const long long e1c = clock64();
#endif
      mbar_wait(&tmem_full_bar[acc], aph);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#ifdef VSR_DBG_CLK
      const long long e2c = clock64();
#else
      long long* clk = nullptr;
#endif
      if constexpr (VOCAB) {
        const int q = warp & 3, row = m0 + q * 32 + lane;
        vocab_epilogue<BN>(p, tmem_acc + ((uint32_t)(q * 32) << 16), row, row < p.M, n0, s_bias, (warp - 2) >> 2);
      } else {
        tile_epilogue<BN>(p, tmem_acc, m0, n0, n_tile, warp, lane, s_bias, reinterpret_cast<float*>(smem + Cfg::kRingBytes), clk);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) {                          // every epilogue warp of both CTAs -> the leader's barrier
        if (rank == 0) mbar_arrive(&tmem_empty_bar[acc]); else mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
      }
#ifdef VSR_DBG_CLK
      if (clk != nullptr) { clk[DBG_E0] = e0c; clk[DBG_E1] = e1c; clk[DBG_E2] = e2c; clk[DBG_E3] = clk[DBG_E4] = clock64(); }
#endif
    }
    it += total_kb;
    ++ti;
  }
  // neither CTA may release TMEM / exit while the pair's MMAs, remote arrivals or the other epilogue are still running
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync_all();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::kTmemCols) : "memory");
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)sym;
  }
  return fn;
}

}  // namespace

// 2-D fp16 tensor map over a row-major [rows][ld] buffer: box = 64 (K) x box_rows, 128-byte swizzle
int make_tmap_f16(void* out_map, const void* base, int rows, int cols, int ld, int box_rows, int kb) {
  EncodeTiledFn enc = get_encode();
  VSR_REQUIRE(enc != nullptr, VSR_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)kb, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = enc((CUtensorMap*)out_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstr,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, kb == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VSR_REQUIRE(r == CUDA_SUCCESS, VSR_ECUDA, "cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%d", (int)r, rows, cols, ld);
  return VSR_OK;
}

// max |x| as the bit pattern of a non-negative float (monotone as unsigned)
__global__ void k_absmax(const float* __restrict__ x, size_t n, unsigned* __restrict__ out) {
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = fabsf(x[i]);
    if (v == v && v < INFINITY) m = fmaxf(m, v);
  }
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}
// scale[0] = 2^e with max|x| * 2^e in (2^12, 2^13]  (1 for an all-zero tensor), scale[1] = 2^-e
// (2^13: the e4m3 copy hi / 32 then stays below the format's maximum of 448)
__global__ void k_pick_scale(float* scale) {
  const float m = __uint_as_float(*reinterpret_cast<unsigned*>(scale));
  int e = 0;
  if (m > 0.f) { int ex; frexpf(m, &ex); e = 13 - ex; }     // m = f * 2^ex, f in [0.5, 1)
  e = e > 100 ? 100 : (e < -100 ? -100 : e);
  scale[0] = ldexpf(1.f, e);
  scale[1] = ldexpf(1.f, -e);
}

// 2-D e4m3 (uint8) tensor map over a row-major [rows][ld] buffer: box = kb (K) x box_rows, rows of kb bytes
int make_tmap_u8(void* out_map, const void* base, int rows, int cols, int ld, int box_rows, int kb) {
  EncodeTiledFn enc = get_encode();
  VSR_REQUIRE(enc != nullptr, VSR_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)ld};
  const cuuint32_t box[2] = {(cuuint32_t)kb, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = enc((CUtensorMap*)out_map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstr,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, kb == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VSR_REQUIRE(r == CUDA_SUCCESS, VSR_ECUDA, "cuTensorMapEncodeTiled (u8) failed (%d) rows=%d cols=%d ld=%d", (int)r, rows, cols, ld);
  return VSR_OK;
}

int make_pair_maps(F16Pair* b, int pair_rows) {
  b->pair_rows = 0;
  if (b->hi == nullptr || pair_rows <= 0) return VSR_OK;
  VSR_TRY(make_tmap_f16(b->pair_hi, b->hi, b->rows, b->ld, b->ld, pair_rows));
  if (b->lo != nullptr) VSR_TRY(make_tmap_f16(b->pair_lo16, b->lo, b->rows, b->ld, b->ld, pair_rows));
  if (b->hi8 != nullptr) {
    VSR_TRY(make_tmap_u8(b->pair_h8, b->hi8, b->rows, b->ld, b->ld, pair_rows));
    VSR_TRY(make_tmap_u8(b->pair_lo, b->lo8, b->rows, b->ld, b->ld, pair_rows));
  }
  b->pair_rows = pair_rows;
  return VSR_OK;
}

namespace {
// x -> whichever twins `o` has; s = *scale (weights) or o.scale (activations)
__global__ void k_split_pair(const float* __restrict__ x, TwinOut o, size_t n4, const float* __restrict__ scale) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  if (scale != nullptr) o.scale = scale[0];
  store_twin4(o, i * 4, *reinterpret_cast<const float4*>(x + i * 4));
}
}  // namespace

int launch_split_pair(const float* x, const F16Pair& p, size_t n, cudaStream_t st, bool weight_scale) {
  if (n == 0 || p.hi == nullptr) return VSR_OK;
  VSR_REQUIRE(n % 4 == 0, VSR_EINVAL, "launch_split_pair: element count %zu not a multiple of 4", n);
  float* scale = weight_scale ? p.scale : nullptr;
  if (scale != nullptr) {
    VSR_CHECK_CUDA(cudaMemsetAsync(scale, 0, 2 * sizeof(float), st));
    k_absmax<<<296, 256, 0, st>>>(x, n, reinterpret_cast<unsigned*>(scale));
    k_pick_scale<<<1, 1, 0, st>>>(scale);
  }
  k_split_pair<<<(unsigned)((n / 4 + 255) / 256), 256, 0, st>>>(x, twin_out(&p), n / 4, scale);
  VSR_CHECK_CUDA(cudaGetLastError());
  return VSR_OK;
}

int tc_gemm_init() {
  // function attributes are per device: track which devices of this process have been set up
  static unsigned long long done_mask = 0ull;
  int dev = 0;
  VSR_CHECK_CUDA(cudaGetDevice(&dev));
  const bool done = dev < 64 && ((done_mask >> dev) & 1ull);
  if (done) return VSR_OK;
#define TC_SET_SMEM(BN_, KB_) VSR_CHECK_CUDA(cudaFuncSetAttribute(k_gemm_tc<BN_, KB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<BN_, KB_>::kSmemBytes))
  TC_SET_SMEM(256, 64); TC_SET_SMEM(192, 64); TC_SET_SMEM(128, 64);
  TC_SET_SMEM(256, 32); TC_SET_SMEM(192, 32); TC_SET_SMEM(128, 32);
  TC_SET_SMEM(144, 64); TC_SET_SMEM(240, 32);
#define TCP_SET_SMEM(BN_, KB_) VSR_CHECK_CUDA(cudaFuncSetAttribute(k_gemm_tcp<BN_, KB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<BN_, KB_>::kSmemBytes))
  TCP_SET_SMEM(128, 64); TCP_SET_SMEM(144, 64); TCP_SET_SMEM(192, 32); TCP_SET_SMEM(192, 64); TCP_SET_SMEM(128, 32);
#undef TCP_SET_SMEM
#undef TC_SET_SMEM
#define PAIR_SET_SMEM(BN_, KB_, V_) VSR_CHECK_CUDA(cudaFuncSetAttribute(k_gemm_pair<BN_, KB_, V_>, cudaFuncAttributeMaxDynamicSharedMemorySize, PairCfg<BN_, KB_, V_>::kSmemBytes))
  PAIR_SET_SMEM(192, 64, false); PAIR_SET_SMEM(192, 64, true); PAIR_SET_SMEM(256, 64, false);
#undef PAIR_SET_SMEM
  if (dev < 64) done_mask |= 1ull << dev;
  return VSR_OK;
}

#ifdef VSR_DBG_CLK
void tc_dbg_clk_report(const char* label) {
  std::vector<long long> r((size_t)DBG_CTAS * DBG_TILES * DBG_F);
  void* sym = nullptr;
  if (cudaDeviceSynchronize() != cudaSuccess || cudaGetSymbolAddress(&sym, g_dbg_clk) != cudaSuccess ||
      cudaMemcpy(r.data(), sym, r.size() * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) {
    printf("clk %s: no records\n", label);
    return;
  }
  cudaMemset(sym, 0, r.size() * sizeof(long long));
  int khz = 1;
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, 0);
  enum { S_MWAIT, S_MLOOP, S_MFULL, S_BIAS, S_EWAIT, S_RELEASE, S_BODY, S_DUMP, S_BAR3, S_PROC, S_BAR4, S_N };
  static const char* names[S_N] = {"mma: wait tmem_empty", "mma: k-loop span", "mma:   of it waiting full_bar", "epi: bias + epi_bar(1)",
                                   "epi: wait tmem_full", "epi: full -> accumulator released", "epi: full -> tile done",
                                   "epi: dump (4 quarters)", "epi: epi_bar(3) (4 quarters)", "epi: process (4 quarters)",
                                   "epi: epi_bar(4) (4 quarters)"};
  std::vector<double> v[S_N];
  double span = 0, mma_busy = 0, epi_busy = 0, overlap = 0;
  int ctas = 0, max_tiles = 0;
  for (int b = 0; b < DBG_CTAS; ++b) {
    const long long* c = r.data() + (size_t)b * DBG_TILES * DBG_F;
    int nt = 0;
    while (nt < DBG_TILES && c[nt * DBG_F + DBG_E4] != 0) ++nt;
    if (nt == 0) continue;
    max_tiles = nt > max_tiles ? nt : max_tiles;
    const bool leader = c[DBG_M2] != 0;
    for (int t = 0; t < nt; ++t) {
      const long long* x = c + t * DBG_F;
      if (leader) { v[S_MWAIT].push_back(x[DBG_M1] - x[DBG_M0]); v[S_MLOOP].push_back(x[DBG_M2] - x[DBG_M1]); v[S_MFULL].push_back(x[DBG_MFULL]); }
      v[S_BIAS].push_back(x[DBG_E1] - x[DBG_E0]); v[S_EWAIT].push_back(x[DBG_E2] - x[DBG_E1]);
      v[S_RELEASE].push_back(x[DBG_E3] - x[DBG_E2]); v[S_BODY].push_back(x[DBG_E4] - x[DBG_E2]);
      for (int ph = 0; ph < 4; ++ph) {
        long long sum = 0;
        for (int q = 0; q < 4; ++q) sum += x[DBG_Q + 4 * q + ph];
        v[S_DUMP + ph].push_back(sum);
      }
    }
    if (!leader) continue;
    // the leader's MMA issuer and epilogue share the SM clock: how much of the epilogue ran under a k-loop
    ++ctas;
    span += c[(nt - 1) * DBG_F + DBG_E4] - c[DBG_M0];
    for (int t = 0; t < nt; ++t) {
      const long long* e = c + t * DBG_F;
      mma_busy += e[DBG_M2] - e[DBG_M1];
      epi_busy += e[DBG_E4] - e[DBG_E2];
      for (int u = 0; u < nt; ++u) {
        const long long* m = c + u * DBG_F;
        const long long lo = m[DBG_M1] > e[DBG_E2] ? m[DBG_M1] : e[DBG_E2], hi = m[DBG_M2] < e[DBG_E4] ? m[DBG_M2] : e[DBG_E4];
        if (hi > lo) overlap += hi - lo;
      }
    }
  }
  const double us = 1e3 / khz;
  printf("clk %s: %d leader CTAs, up to %d tiles per CTA, cycles per tile (us at %d MHz): mean / median / p90\n", label, ctas,
         max_tiles, khz / 1000);
  for (int k = 0; k < S_N; ++k) {
    std::vector<double>& x = v[k];
    if (x.empty()) continue;
    std::sort(x.begin(), x.end());
    double m = 0;
    for (double y : x) m += y;
    m /= x.size();
    printf("  %-36s %8.0f %8.0f %8.0f  (%.2f us)\n", names[k], m, x[x.size() / 2], x[x.size() * 9 / 10], m * us);
  }
  if (ctas > 0)
    printf("  per leader CTA: span %.1f us, k-loops %.1f us, epilogues %.1f us, epilogue under a k-loop %.1f us (%.0f %% of the epilogue)\n",
           span / ctas * us, mma_busy / ctas * us, epi_busy / ctas * us, overlap / ctas * us, 100.0 * overlap / (epi_busy > 0 ? epi_busy : 1));
}
#endif

static int fill_problem(TcProblem* p, const GemmArgs& g, int BN, int kb = 64, bool pair = false) {
  VSR_REQUIRE(g.M > 0 && g.N >= round_up(g.wb->n_valid, BN), VSR_EINVAL, "launch_gemm_tc: N=%d too small for N tile %d", g.N, BN);
  p->nseg = g.nseg;
  p->f8 = g.f8 ? 1 : 0;
  VSR_REQUIRE(g.f8 ? (g.wb->hi8 != nullptr && g.wb->lo8 != nullptr) : g.wb->lo != nullptr, VSR_EINVAL,
              "launch_gemm_tc: the weight has no %s twin", g.f8 ? "e4m3" : "fp16 residual");
  for (int s = 0; s < g.nseg; ++s) {
    const F16Pair* b = g.seg[s].b;
    VSR_REQUIRE(b != nullptr && g.seg[s].k % BK == 0, VSR_EINVAL, "launch_gemm_tc: segment %d not tensor-core ready", s);
    VSR_REQUIRE(g.f8 ? (b->hi8 != nullptr && b->lo8 != nullptr) : b->lo != nullptr, VSR_EINVAL,
                "launch_gemm_tc: segment %d has no %s twin", s, g.f8 ? "e4m3" : "fp16 residual");
    VSR_REQUIRE(b->act_scale == g.seg[0].b->act_scale, VSR_EINVAL, "launch_gemm_tc: segments with different activation scales");
    memcpy(&p->a_hi[s], kb == 32 ? b->map32_hi : b->map_hi, sizeof(CUtensorMap));
    if (g.f8) {
      memcpy(&p->a_h8[s], kb == 32 ? b->map8_32_hi : b->map8_hi, sizeof(CUtensorMap));
      memcpy(&p->a_lo[s], kb == 32 ? b->map8_32_lo : b->map8_lo, sizeof(CUtensorMap));
    } else {
      memcpy(&p->a_lo[s], kb == 32 ? b->map32_lo : b->map_lo, sizeof(CUtensorMap));
    }
    p->kblocks[s] = g.seg[s].k / kb;
  }
  const bool alt = !pair && BN == g.wb->alt_bn && BN != g.wb->box_rows;
  if (pair) {       // CTA-pair kernel: half-tile maps (BN / 2 rows), 64-element k-blocks
    VSR_REQUIRE(g.wb->pair_rows * 2 == BN && kb == 64, VSR_EINVAL, "launch_gemm_tc: weight has no pair maps for N tile %d", BN);
    memcpy(&p->w_hi, g.wb->pair_hi, sizeof(CUtensorMap));
    memcpy(&p->w_lo, g.f8 ? g.wb->pair_lo : g.wb->pair_lo16, sizeof(CUtensorMap));
    if (g.f8) memcpy(&p->w_h8, g.wb->pair_h8, sizeof(CUtensorMap));
  } else {
  memcpy(&p->w_hi, alt ? g.wb->alt_hi : (kb == 32 ? g.wb->map32_hi : g.wb->map_hi), sizeof(CUtensorMap));
  if (g.f8) {
    memcpy(&p->w_h8, alt ? g.wb->alt8_hi : (kb == 32 ? g.wb->map8_32_hi : g.wb->map8_hi), sizeof(CUtensorMap));
    memcpy(&p->w_lo, alt ? g.wb->alt8_lo : (kb == 32 ? g.wb->map8_32_lo : g.wb->map8_lo), sizeof(CUtensorMap));
  } else {
    memcpy(&p->w_lo, alt ? g.wb->alt_lo : (kb == 32 ? g.wb->map32_lo : g.wb->map_lo), sizeof(CUtensorMap));
  }
  }
  p->acc_scale = g.wb->scale != nullptr ? g.wb->scale + 1 : nullptr;
  p->act_inv = 1.f / g.seg[0].b->act_scale;
  p->n_tiles = (g.wb->n_valid + BN - 1) / BN; p->m_tiles = (g.M + BM - 1) / BM; p->M = g.M; p->row_skip = g.row_skip;
  p->bias = g.bias; p->rowadd = g.rowadd; p->ld_rowadd = g.ld_rowadd; p->row_div = g.row_div > 0 ? g.row_div : 1;
  p->rowadd_mul = g.rowadd_mul; p->cadd = g.cadd; p->ld_cadd = g.ld_cadd; p->c = g.c; p->ldc = g.ldc;
  p->gather = g.gather; p->ld_gather = g.ld_gather; p->gather_idx = g.gather_idx;
  const FusedCell& f = g.cell;
  p->mode = f.mode;
  if (f.mode == EPI_VOCAB) {
    VSR_REQUIRE(f.vocab_part != nullptr && g.bias != nullptr && g.c != nullptr && g.ldc % 16 == 0 && g.N % BN == 0, VSR_EINVAL,
                "launch_gemm_tc: vocabulary epilogue needs a bias, an output padded to whole tiles and a record buffer (N tile %d)", BN);
    p->vpart = f.vocab_part; p->n_valid = g.wb->n_valid;
  } else if (f.mode != 0) {
    VSR_REQUIRE((f.mode == EPI_LSTM1 && BN == 192) || (f.mode == EPI_LSTM2 && (BN == 128 || (pair && BN == 256))), VSR_EINVAL,
                "launch_gemm_tc: fused cell mode %d does not fit N tile %d", f.mode, BN);
    p->c_old = f.c_old; p->c_new = f.c_new; p->h_new = f.h_new; p->h_tw = twin_out(f.h_b);
    p->s_new = f.s_new; p->s_tw = twin_out(f.s_b); p->gq = f.gq;
  }
  VSR_REQUIRE(f.gt_cols == 0 || BN == 128 || BN == 192 || (pair && BN == 256 && f.gt_cols % 256 == 0), VSR_EINVAL,
              "launch_gemm_tc: g_t fusion needs a 128- or 192-wide tile");
  p->zero_acc = g.zero_acc ? 1 : 0;
  p->ld_state = f.ld_state;
  p->gt_cols = f.gt_cols; p->gt_gq = f.gt_gq; p->gt_c1n = f.gt_c1n; p->g_t = f.g_t;
  p->g_tw = twin_out(f.g_b);
  return VSR_OK;
}

// Can this launch run on the CTA-pair kernel?  Large row counts only (at a few hundred rows the 256-row pair tiles leave
// most SMs idle: measured slower), pair maps present, tile-compatible epilogues, whole tiles in N.
static bool pair_ok(const GemmArgs& g) {
  if (!g.allow_pair || g.wb == nullptr || g.wb->pair_rows <= 0 || g.M < g.pair_min_rows || g.row_skip != nullptr || g.zero_acc) return false;
  const int BN = 2 * g.wb->pair_rows;
  if (g.N % BN != 0 || (BN != 192 && BN != 256)) return false;
  const int mode = g.cell.mode;
  if (mode == EPI_VOCAB && BN != 192) return false;     // row-per-thread epilogue: 12 chunks per row keep its registers in check
  if (mode == EPI_LSTM1 && BN != 192) return false;
  if (mode == EPI_LSTM2 && BN != 256) return false;
  if (g.cell.gt_cols % BN != 0) return false;
  return true;
}

static int launch_gemm_pair(const GemmArgs& g, const GemmArgs* g2, cudaStream_t st) {
  const int BN = 2 * g.wb->pair_rows;
  const bool vocab = g.cell.mode == EPI_VOCAB;
  const int kb = 64;
  TcParams p;
  memset(&p, 0, sizeof(p));
  VSR_TRY(fill_problem(&p.pr[0], g, BN, kb, true));
  p.nprob = 1;
  int tiles = p.pr[0].n_tiles * ((p.pr[0].m_tiles + 1) / 2);
  if (g2 != nullptr) {
    VSR_TRY(fill_problem(&p.pr[1], *g2, BN, kb, true));
    p.nprob = 2;
    tiles += p.pr[1].n_tiles * ((p.pr[1].m_tiles + 1) / 2);
  }
  static int sms = 0;
  if (sms == 0) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  const int clusters = tiles < sms / 2 ? tiles : sms / 2;
#define PAIR_LAUNCH(BN_, KB_, V_) VSR_CHECK_CUDA(launch_k(k_gemm_pair<BN_, KB_, V_>, dim3(2 * clusters), dim3(TC_THREADS), PairCfg<BN_, KB_, V_>::kSmemBytes, st, g.pdl, p))
  if (BN == 192 && vocab) PAIR_LAUNCH(192, 64, true);
  else if (BN == 192) PAIR_LAUNCH(192, 64, false);
  else PAIR_LAUNCH(256, 64, false);
#undef PAIR_LAUNCH
  VSR_CHECK_CUDA(cudaGetLastError());
  return VSR_OK;
}

// g2 (optional) is an independent problem with the same N tile that shares the launch
int launch_gemm_tc(const GemmArgs& g, const GemmArgs* g2, cudaStream_t st) {
  VSR_TRY(tc_gemm_init());
  if (pair_ok(g) && (g2 == nullptr || (pair_ok(*g2) && g2->wb->pair_rows == g.wb->pair_rows))) return launch_gemm_pair(g, g2, st);
  int BN = g.wb->box_rows;
  VSR_REQUIRE(BN == 128 || BN == 192 || BN == 256, VSR_EINVAL, "launch_gemm_tc: unsupported N tile %d", BN);
  VSR_REQUIRE(g2 == nullptr || g2->wb->box_rows == BN, VSR_EINVAL, "launch_gemm_tc: grouped problems need one tile shape");
  TcParams p;            // ~2.7 KB; passed by value at launch
  memset(&p, 0, sizeof(p));
  int kb = g.wb->kb;          // k-block (64 or 32 fp16) chosen per weight at pack time
  VSR_REQUIRE(g2 == nullptr || g2->wb->kb == kb, VSR_EINVAL, "launch_gemm_tc: grouped problems need one k-block size");
  // Tile choice: operand delivery bounds these GEMMs, so a tile costs ~ (BM + BN) and a launch costs
  // waves(tiles / 148 SMs) * (BM + BN).  Take the alternative N tile when that is cheaper.
  if (g.wb->alt_bn > 0 && !g.no_alt && (g.cell.mode == 0 || g.cell.mode == EPI_VOCAB) && (g2 == nullptr || (g2->wb->alt_bn == g.wb->alt_bn && g2->cell.mode == 0))) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    const int mt = (g.M + BM - 1) / BM;
    auto cost = [&](int bn) {
      int tiles = mt * ((g.wb->n_valid + bn - 1) / bn);
      if (g2 != nullptr) tiles += ((g2->M + BM - 1) / BM) * ((g2->wb->n_valid + bn - 1) / bn);
      return ((tiles + sms - 1) / sms) * (BM + bn);
    };
    if (cost(g.wb->alt_bn) < cost(BN)) { BN = g.wb->alt_bn; kb = g.wb->alt_kb; }
  }
  VSR_TRY(fill_problem(&p.pr[0], g, BN, kb));
  p.nprob = 1;
  p.pdl_flags = g.pdl_flags;
  int tiles = p.pr[0].n_tiles * p.pr[0].m_tiles;
  if (g2 != nullptr) {
    VSR_TRY(fill_problem(&p.pr[1], *g2, BN, kb));
    p.nprob = 2;
    tiles += p.pr[1].n_tiles * p.pr[1].m_tiles;
  }
  static int persist = -1, sms = 148;
  if (persist < 0) {
    const char* e = getenv("VSRDEC_PERSIST");
    persist = (e == nullptr) ? 1 : atoi(e);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  }
  // persistent tiles pay off only when a CTA gets more than one tile (epilogue / main-loop overlap);
  // for single-wave launches the plain kernel measured 5-10 % faster
  // (and measured neutral-to-worse for the grouped two-problem launch, whose tiles are uneven)
  if (persist && tiles > sms && g2 == nullptr && (BN == 128 || BN == 144 || BN == 192)) {
    const int grid = tiles < sms ? tiles : sms;
#define TCP_LAUNCH(BN_, KB_) VSR_CHECK_CUDA(launch_k(k_gemm_tcp<BN_, KB_>, dim3(grid), dim3(TC_THREADS), TcCfg<BN_, KB_>::kSmemBytes, st, g.pdl, p))
    if (BN == 144) TCP_LAUNCH(144, 64);
    else if (BN == 192) { if (kb == 32) TCP_LAUNCH(192, 32); else TCP_LAUNCH(192, 64); }
    else { if (kb == 32) TCP_LAUNCH(128, 32); else TCP_LAUNCH(128, 64); }
#undef TCP_LAUNCH
    VSR_CHECK_CUDA(cudaGetLastError());
    return VSR_OK;
  }
#define TC_LAUNCH(BN_, KB_) VSR_CHECK_CUDA(launch_k(k_gemm_tc<BN_, KB_>, dim3(tiles), dim3(TC_THREADS), TcCfg<BN_, KB_>::kSmemBytes, st, g.pdl, p))
  if (BN == 144) TC_LAUNCH(144, 64);
  else if (BN == 240) TC_LAUNCH(240, 32);
  else if (kb == 32) {
    if (BN == 256) TC_LAUNCH(256, 32); else if (BN == 192) TC_LAUNCH(192, 32); else TC_LAUNCH(128, 32);
  } else {
    if (BN == 256) TC_LAUNCH(256, 64); else if (BN == 192) TC_LAUNCH(192, 64); else TC_LAUNCH(128, 64);
  }
#undef TC_LAUNCH
  VSR_CHECK_CUDA(cudaGetLastError());
  return VSR_OK;
}

}  // namespace vsr
