// Shared declarations of libvsrdec: context, packed-weight layout, launch helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/vsrdec.h"

namespace vsr {

// ---------------------------------------------------------------- errors
void set_error(const char* fmt, ...);
#define VSR_CHECK_CUDA(expr)                                                                 \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      vsr::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,                   \
                     cudaGetErrorString(_e));                                                \
      return VSR_ECUDA;                                                                      \
    }                                                                                        \
  } while (0)
#define VSR_REQUIRE(cond, code, ...)                                                         \
  do {                                                                                       \
    if (!(cond)) {                                                                           \
      vsr::set_error(__VA_ARGS__);                                                           \
      return (code);                                                                         \
    }                                                                                        \
  } while (0)
#define VSR_TRY(expr)                                                                        \
  do {                                                                                       \
    int _r = (expr);                                                                         \
    if (_r != VSR_OK) return _r;                                                             \
  } while (0)

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

#ifdef __CUDACC__
}  // namespace vsr
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
namespace vsr {
// Gate non-linearities on the SFU (ex2.approx + fast reciprocal): absolute error ~1e-7, i.e. fp32 rounding
// level, at ~1/4 of the instructions of expf/tanhf.  tanh via 1 - 2/(e^{2x}+1) saturates cleanly (e^{2x} = inf
// -> 1, = 0 -> -1); its relative error grows for |x| << 1 but the ABSOLUTE error stays ~1e-7, which is what
// the attention scores / LSTM cells need (checked by the parity tests against the fp32 oracle).
__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float fast_tanh(float x) { return 1.f - __fdividef(2.f, __expf(2.f * x) + 1.f); }

// Caller features (det, det_seqs) are fp32, fp16 or bf16 (vsr_prologue_ex).  Four consecutive elements, widened to
// fp32 as they are loaded: exact, so every kernel that reads features does the same fp32 arithmetic in the same order
// whatever the storage type.  fp32 is one 16-byte load, half precision one 8-byte load (a row of F % 8 == 4 half
// elements is only 8-byte aligned).
__device__ __forceinline__ float4 ldg_feat4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ldg_feat4(const __half* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 ldg_feat4(const __nv_bfloat16* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
#endif

// element size in bytes of a feature dtype tag (VSR_DT_F32 / F16 / BF16), 0 for any other tag
static inline int feat_elem_size(int dt) { return dt == VSR_DT_F32 ? 4 : (dt == VSR_DT_F16 || dt == VSR_DT_BF16) ? 2 : 0; }

// K (reduction) dims are padded to KPAD floats (one 128-byte swizzle row of fp32), output-feature
// dims to NPAD rows, activation row counts to MPAD rows; pads are zero so they never contribute.
constexpr int KPAD = 64;    // 64 fp16 = one 128-byte swizzle row of the tensor-core operand tiles
constexpr int NPAD = 256;   // widest UMMA N tile
constexpr int MPAD = 128;   // UMMA M tile

// An fp32 matrix carried as an error-compensated fp16 pair (x = hi + lo + O(2^-22 x)) with the TMA
// tensor maps (64 x box_rows boxes, 128-byte swizzle) the tcgen05 GEMM loads it through.
// Activation twins of the f16+f8x2 GEMM mode are stored scaled by ACT_SCALE_F8 (a power of two, exact): their
// residuals x*s - fp16(x*s) then sit in the normal range of e4m3 for the |x| ~ 1e-2..1 of the decoder's states.
constexpr float ACT_SCALE_F8 = 256.f;

struct F16Pair {
  void* hi = nullptr;   // __half [rows][ld]
  void* lo = nullptr;   // __half residual (f16x3 mode), or null
  // f16+f8x2 mode: e4m3 twins, uint8 [rows][ld].  hi8 = e4m3(hi / 32), lo8 = e4m3((x*s - hi) * 32): with these
  // shifts hi*W_hi (fp16), hi8*W_lo8 and lo8*W_hi8 (fp8) all carry the same power-of-two scale and accumulate into
  // ONE fp32 TMEM accumulator; both e4m3 operands stay inside the format's normal range (|hi| <= 2^13).
  void* hi8 = nullptr;
  void* lo8 = nullptr;
  float act_scale = 1.f;   // activations: the constant the producer multiplied x by (1, or ACT_SCALE_F8 in f16+f8x2 mode)
  int rows = 0, ld = 0, box_rows = 0;
  // (weights only) device [2] = {s, 1/s}: the pair holds x * s with s the power of two that brings max|x| to 2^13..2^14,
  // so lo parts of small weights stay out of the fp16 subnormals; the GEMM epilogue multiplies the accumulator by 1/s
  // (exact).  Null = unscaled (activations: |x| ~ 1).
  float* scale = nullptr;
  int kb = 64;          // (weights only) k-block of the GEMMs that use this weight: 64 (128B swizzle) or 32 (64B)
  alignas(64) unsigned char map_hi[128];
  alignas(64) unsigned char map_lo[128];
  alignas(64) unsigned char map32_hi[128];   // 32-element k-blocks, 64-byte swizzle
  alignas(64) unsigned char map32_lo[128];
  alignas(64) unsigned char map8_hi[128];    // e4m3 twins, 64-element k-blocks (64-byte rows, 64-byte swizzle)
  alignas(64) unsigned char map8_lo[128];
  alignas(64) unsigned char map8_32_hi[128]; // e4m3 twins, 32-element k-blocks (32-byte rows, 32-byte swizzle)
  alignas(64) unsigned char map8_32_lo[128];
  alignas(64) unsigned char alt8_hi[128];    // e4m3 twins, alternative N tile
  alignas(64) unsigned char alt8_lo[128];
  // (weights only) CTA-pair kernel: each CTA of the pair loads pair_rows = BN / 2 rows of a BN-wide W tile (64-element k-blocks)
  int pair_rows = 0;
  alignas(64) unsigned char pair_hi[128];
  alignas(64) unsigned char pair_lo[128];    // e4m3 residual (f16+f8x2)
  alignas(64) unsigned char pair_lo16[128];  // fp16 residual (f16x3)
  alignas(64) unsigned char pair_h8[128];    // e4m3 copy of hi (f16+f8x2)
  // (weights only) alternative N tile, chosen per launch when it needs fewer waves over the 148 SMs
  int n_valid = 0;      // real number of output rows (<= rows)
  int alt_bn = 0, alt_kb = 64;
  alignas(64) unsigned char alt_hi[128];
  alignas(64) unsigned char alt_lo[128];
};

// Where a kernel writes the tensor-core twins of an activation it produces (any pointer may be null).
struct TwinOut {
  void* hi; void* lo; uint8_t* hi8; uint8_t* lo8;
  float scale;
};
inline TwinOut twin_out(const F16Pair* b, bool enabled = true) {
  TwinOut o{nullptr, nullptr, nullptr, nullptr, 1.f};
  if (b != nullptr && enabled) { o.hi = b->hi; o.lo = b->lo; o.hi8 = (uint8_t*)b->hi8; o.lo8 = (uint8_t*)b->lo8; o.scale = b->act_scale; }
  return o;
}
#ifdef __CUDACC__
// twins of four consecutive values at element offset off (multiple of 4)
__device__ __forceinline__ void store_twin4(const TwinOut& o, size_t off, const float4 v) {
  if (o.hi == nullptr) return;
  const float x[4] = {fminf(fmaxf(v.x * o.scale, -65504.f), 65504.f), fminf(fmaxf(v.y * o.scale, -65504.f), 65504.f),
                      fminf(fmaxf(v.z * o.scale, -65504.f), 65504.f), fminf(fmaxf(v.w * o.scale, -65504.f), 65504.f)};
  __align__(8) __half h[4];
  float hf[4], r[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { h[j] = __float2half_rn(x[j]); hf[j] = __half2float(h[j]); r[j] = x[j] - hf[j]; }
  *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(o.hi) + off) = *reinterpret_cast<const uint2*>(h);
  if (o.lo != nullptr) {
    __align__(8) __half l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) l[j] = __float2half_rn(r[j]);
    *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(o.lo) + off) = *reinterpret_cast<const uint2*>(l);
  }
  if (o.hi8 != nullptr) {
    const unsigned h01 = __nv_cvt_float2_to_fp8x2(make_float2(hf[0] * 0.03125f, hf[1] * 0.03125f), __NV_SATFINITE, __NV_E4M3);
    const unsigned h23 = __nv_cvt_float2_to_fp8x2(make_float2(hf[2] * 0.03125f, hf[3] * 0.03125f), __NV_SATFINITE, __NV_E4M3);
    const unsigned l01 = __nv_cvt_float2_to_fp8x2(make_float2(r[0] * 32.f, r[1] * 32.f), __NV_SATFINITE, __NV_E4M3);
    const unsigned l23 = __nv_cvt_float2_to_fp8x2(make_float2(r[2] * 32.f, r[3] * 32.f), __NV_SATFINITE, __NV_E4M3);
    *reinterpret_cast<uint32_t*>(o.hi8 + off) = h01 | (h23 << 16);
    *reinterpret_cast<uint32_t*>(o.lo8 + off) = l01 | (l23 << 16);
  }
}
#endif

// ---------------------------------------------------------------- GEMM (C = sum_seg A_seg * W_seg^T + ...)
struct GemmSeg {
  const float* a;   // [M][lda] activations, K contiguous
  int lda;
  int k;            // padded K of this segment in the weight layout (multiple of KPAD)
  int k_valid;      // readable columns of a (multiple of 4, <= k); the rest reads as zero
  const F16Pair* b = nullptr;   // fp16 hi/lo twin of a (tensor-core path), or null
};
// Column of (gate g, hidden unit u) in a gate-interleaved LSTM pre-activation row with NG gates: 32-unit chunks,
// each laid out as [gate][32 units], so that one 128 x (NG*32) tensor-core tile holds every gate of its 32 units
// (the cell math runs in the GEMM epilogue) and the 32 units of a gate are 128 contiguous bytes (coalesced operands).
__host__ __device__ inline int cell_col(int g, int u, int ng) {
  return (u >> 5) * (ng * 32) + g * 32 + (u & 31);
}

// Optional epilogue fusion of the tensor-core GEMM (ignored by the FFMA twin, whose callers run the
// stand-alone pointwise kernels instead).
// ---------------------------------------------------------------- programmatic dependent launch (PDL)
// The kernels of a decoder step form one dependency chain.  Launched with the programmatic-serialization attribute,
// kernel N+1 may become resident while kernel N drains: it runs its own set-up (barrier init, TMEM allocation,
// descriptor prefetch, WEIGHT tile prefetch) and then blocks in pdl_wait() until kernel N has completed and its
// writes are visible.  Rule for every such kernel: before pdl_wait() touch nothing but launch arguments and data
// that is constant over the whole decode (weights, prologue products); write nothing.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                            Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
#endif

struct FusedCell {
  int mode = 0;                 // 0 = plain, 1 = LSTM cell 1 (+ sentinel gate, 6 gates), 2 = LSTM cell 2 (4 gates)
  const float* c_old = nullptr; float* c_new = nullptr; float* h_new = nullptr;
  const F16Pair *h_b = nullptr, *s_b = nullptr, *g_b = nullptr;     // twins of h_new / s_new / g_t to write (or null)
  float* s_new = nullptr;                                           // mode 1: s_t = sig(s) * tanh(c1')
  float* gq = nullptr;                                              // mode 1: shift-gate pre-activation (input_1 part)
  int ld_state = 0;
  // plain mode only: on output columns [0, gt_cols) write g_t = sig(gq + acc) * tanh(c1') instead of acc
  int gt_cols = 0; const float* gt_gq = nullptr; const float* gt_c1n = nullptr;
  float* g_t = nullptr;
  // mode 3 (vocabulary head): besides the logits, per (row, N tile) records of VOCAB_REC floats
  // {tile max, sum exp(x - max), max of each 16-column chunk}.  *vocab_tiles_out / *vocab_bn_out = tiling of the launch.
  float* vocab_part = nullptr; int* vocab_tiles_out = nullptr; int* vocab_bn_out = nullptr;
};
constexpr int VOCAB_REC = 16;

struct GemmArgs {
  GemmSeg seg[3];
  int nseg;
  const float* w;   // [N][ldw] packed weights, K contiguous, segments back to back
  int ldw;
  const float* bias;    // [N] or null
  const float* rowadd;  // [(row / row_div) * rowadd_mul][ld_rowadd] added per row, or null
  int ld_rowadd, row_div, rowadd_mul;
  const float* cadd;    // [M][ld_cadd] added element-wise, or null
  int ld_cadd;
  float* c;             // [M][ldc]
  int ldc;
  int M, N;             // N multiple of NPAD
  const float* gather = nullptr;      // optional [*][ld_gather]: adds gather[gather_idx[row]][n] (embedding-side
  int ld_gather = 0;                  //   projections precomputed per vocabulary entry)
  const int32_t* gather_idx = nullptr;
  const uint8_t* row_skip;  // optional [M]: a row tile whose flags are all 0 is skipped
  const F16Pair* wb = nullptr;  // fp16 hi/lo twin of w (tensor-core path), or null
  bool allow_pair = false;      // may run on the CTA-pair kernel when the launch is large enough (step GEMMs A, B, D+C, E)
  int pair_min_rows = 1024;     //   ... i.e. has at least this many rows
  bool no_alt = false;          // keep the weight's default N tile (whose epilogue is the coalesced shared-memory tile one)
  bool f8 = false;              // f16+f8x2 mode: residual products on the fp8 tensor path (operand pairs need hi8 / lo8)
  bool pdl = false;             // launch with programmatic dependent launch (decoder-step GEMMs only)
  bool relu = false;            // FFMA twin only: max(0, .) on the output (feed-forward layers of the S-level SSP sorter)
  bool zero_acc = false;        // every A operand is known to be zero (h = 0 at t = 0): skip the main loop, acc := 0
  int pdl_flags = 0;            // bit 0: weight tiles before the dependency wait; bit 1: trigger after the main loop
  FusedCell cell;               // epilogue fusion (tensor-core path only)
};
struct Ctx;
// tcgen05 when every operand has an fp16 twin, else FFMA; g2 = optional independent problem sharing the launch
int launch_gemm(Ctx* c, const GemmArgs& g, cudaStream_t st, const GemmArgs* g2 = nullptr);
int launch_gemm_simt(const GemmArgs& g, cudaStream_t st);
int launch_gemm_tc(const GemmArgs& g, const GemmArgs* g2, cudaStream_t st);
bool gemm_uses_tc(const Ctx* c, const GemmArgs& g);
int make_tmap_f16(void* out_map, const void* base, int rows, int cols, int ld, int box_rows, int kb = 64);
int make_tmap_u8(void* out_map, const void* base, int rows, int cols, int ld, int box_rows, int kb = 64);
int make_pair_maps(F16Pair* b, int pair_rows);   // tensor maps of a weight for the CTA-pair kernel (after hi/lo/hi8/lo8 are set)
// x -> pair (fp16 hi + fp16 lo and/or e4m3 hi8/lo8, whichever arrays the pair has); scale = device {s, 1/s} computed
// here from max|x| (weights), or null: x is multiplied by p.act_scale (activations)
int launch_split_pair(const float* x, const F16Pair& p, size_t n, cudaStream_t st, bool weight_scale = false);
#ifdef VSR_DBG_CLK
// debug builds only: prints the per-tile clock64 phases recorded by the last k_gemm_pair launch, then clears them
void tc_dbg_clk_report(const char* label);
#endif

// ---------------------------------------------------------------- context
struct Phase {
  const char* name;
  std::vector<cudaEvent_t> ev;  // start/stop pairs recorded during the last decode
  int launches = 0;
};

enum PhaseId {
  PH_PROLOGUE = 0, PH_GEMM_A, PH_LSTM1, PH_GEMM_B, PH_GT, PH_GEMM_C, PH_ATTEND, PH_GEMM_D, PH_LSTM2,
  PH_GEMM_E, PH_SOFTMAX_TOPK, PH_BEAM, PH_REORDER, PH_FINAL, PH_COUNT
};

struct Ctx {
  VsrDims d;
  int device;
  // model dims and padded dims
  int V, E, H, F, A;
  int Hp, Ep, Fp, Ap;          // K-padded
  int NA, NB1, NB2, NC, ND, NE;  // padded output widths of the stacked GEMMs
  int NB1v, NB2v;                // their un-padded widths
  int KA;                      // [h2 (Hp, if h2_first) | h1 (Hp)]  (the xt part is a per-word table, see X)
  int KD;                      // [att (Fp) | h1' (Hp) | h2 (Hp)]  (h2 last: dropped at t = 0 where it is zero)
  // column offsets of the stacked output blocks (KPAD-aligned so float4 epilogues stay aligned)
  int oB1_sa;                  // sent:  sentinel at 0 (F) | sa at oB1_sa (A)
  int oB2_ha, oB2_p2;          // hb:    hg at 0 (H) | ha at oB2_ha (A) ; oB2_p2 = end of the valid columns
  // packed weights
  float *WA, *WU, *bU;         // [NA][KA], [NA][Fp], [NA]   rows: i,f,g,o (4H) | s (H) | g (H)
  float *WB1, *bB1;            // [NB1][Hp]: s_fc (F) | att_sa (A)
  float *WB2;                  // [NB2][Hp]: W1_hg (H) | att_ha (A)
  float *WC;                   // [NC][Hp]: att_ga
  float *WD, *bD;              // [ND][KD]: lstm2.W_ih[:, H:H+F] | lstm2.W_hh | lstm2.W_ih[:, :H] ; b_ih2 + b_hh2
  float *WU2;                  // [ND][Fp]: lstm2.W_ih[:, H+F:H+2F] (img_second_lstm) or null
  float *WE, *bE;              // [NE][Hp]: out_fc
  float *Wva;                  // [Ap128][Fp]: att_va
  float *v_a, *v_s, *v_g;      // [Ap]
  float *embed;                // [V][Ep]
  float *WAx;                  // [NA][Ep]  xt columns of the stacked lstm1 / s-gate / g-gate input weights
  float *X;                    // [V][NA]   X[v] = WAx . embed[v]: the xt contribution per vocabulary entry
  int NVA;                     // padded rows of Wva
  // fp16 hi/lo twins for the tcgen05 GEMMs
  bool use_tc = true;
  int pair_min_rows = 640;       // B, D + C, E take the CTA-pair kernel from this many rows (VSRDEC_PAIR_MIN_ROWS; measured:
                                 //   slower at 500 rows, 6 % faster at 1000)
  bool use_pair = true;          // CTA-pair (cta_group::2) kernel for the large-batch step GEMMs (VSRDEC_PAIR=0 disables)
  bool gemm_f8 = true;           // step GEMMs in f16+f8x2 mode (VSRDEC_GEMM=f16x3 keeps all three passes in fp16)
  bool use_alt_tiles = true;     // per-launch choice between the default and the alternative N tile (VSRDEC_ALT_TILES=0)
  int gemm_kb = 64;              // k-block of the tensor-core GEMMs (VSRDEC_KB=32: 64-byte swizzle, deeper ring)
  F16Pair WA_b, WB1_b, WB2_b, WC_b, WD_b, WE_b;
  F16Pair WU_b, WU2_b, Wva_b;   // prologue weights
  F16Pair ds_b, img_b;          // prologue activations: slot rows [b*L*R][Fp], image descriptors [n_img][Fp]
  F16Pair h1_b, h2_b, s_t_b, h1n_b, g_t_b, att_b, h2n_b;
  // batched teacher-forced forward: h2' of every (caption, step) [b*T][Hp] twins, their logits and gate rows
  F16Pair h2all_b; float* logits_all = nullptr; float* gate_all = nullptr; int cap_fwd_rows = 0;
  // verb table (device CSR)
  int64_t* vt_keys = nullptr; int32_t* vt_off = nullptr; int32_t* vt_idx = nullptr; int vt_n = 0;
  // prologue products (per batch)
  bool have_prologue = false;
  int b = 0, D = 0, L = 0, R = 0, n_img = 0;
  // caller features, element type feat_dtype (VSR_DT_F32 / F16 / BF16) for det and det_seqs alike
  const void* det_seqs = nullptr;        // materialised slot tiles (b,L,R,F), or null in index form
  const int32_t* slot_index = nullptr;   // index form: (b,L,R) detection row / -2 mean row / -1 padding
  const void* det = nullptr; int64_t det_stride = 0;   // index form: detections (n_img, D, F); stride in elements
  int feat_dtype = VSR_DT_F32;
  float* Pmean = nullptr;                // index form: att_va projection of the image mean rows [n_img][NVA]
  const void* verbs = nullptr; int verbs_dtype = 0;
  float* img = nullptr;        // [n_img_alloc][Fp]
  float* U = nullptr;          // [n_img_alloc][NA]
  float* U2 = nullptr;         // [n_img_alloc][ND]
  float* P = nullptr;          // [b*L*R (alloc)][NVA] att_va projections
  uint8_t* seq_valid = nullptr;  // [b*L*R]
  unsigned long long* slot_mask = nullptr;  // [b*L] bit r set = region r of the slot is a real (non-padding) row
  // tensor-core path, materialised slots: only the valid rows are split to fp16 and projected; the valid rows of
  // slot s occupy P rows slot_base[s] .. slot_base[s] + popcount(slot_mask[s]) - 1 (null = P row == slot row)
  int32_t* slot_base = nullptr;             // [b*L]
  uint8_t* comp_valid = nullptr;            // [rows of P] 1 for the rows in use (tile skipping of the projection GEMM)
  bool p_compact = false;
  uint8_t* det_valid = nullptr;  // [n_img*D]
  size_t cap_img = 0, cap_P = 0, cap_detv = 0, cap_slots = 0;
  // per-row workspace (rows = captions * beam), capacity cap_rows (multiple of MPAD)
  int cap_rows = 0;
  float *h1, *c1, *h2, *c2;          // current state [rows][Hp]
  float *h1n, *c1n, *h2n, *c2n;      // state produced by the step
  int32_t *word_idx;                 // [rows] input token of the step (bos / previous pick / teacher token)
  int32_t *ptr, *ptrn;               // slot pointer per row
  float *pre1;                       // [rows][NA]
  float *s_t, *g_t;                  // [rows][Hp]
  float *gq;                         // [rows][Hp] shift-gate pre-activation, input_1 part (W1_ig . input_1 + biases)
  float *sent;                       // [rows][NB1] sentinel (F) | sa (A)
  float *hb;                         // [rows][NB2] hg (H) | ha (A) | pre2_h1 (4H)
  float *ga;                         // [rows][NC]
  float *att;                        // [rows][Fp]
  float *pre2;                       // [rows][ND]
  float *logits;                     // [rows][NE]
  float *gate_lp;                    // [rows][2]
  float *shift;                      // [rows] raw shift-gate logit
  float *row_max, *row_lsum;         // [rows]
  int32_t *forced;                   // [rows] forced vocab idx or -1
  int32_t *cand;                     // [rows][VSR_MAX_BEAM]
  float *vpart;                      // [rows][NE / 16][2] per-chunk softmax records {max, sum exp} of the vocabulary GEMM
  // beam workspace
  int cap_caps = 0, cap_T = 0;
  float *seq_lp, *seq_lp_n;          // [caps][beam]
  float *m0, *m1, *m0n, *m1n;        // sticky EOS masks [caps][beam]
  int32_t *sel_beam, *sel_word, *sel_gate;  // [caps][beam] selections of the current step
  int32_t *sel_beam_n, *sel_word_n, *sel_gate_n;
  int cap_sel = 0;                   // capacity of the six sel_* buffers in rows (ensure_sel)
  int32_t *hist_parent, *hist_word, *hist_gate;  // [T][caps][beam]
  float *hist_score, *hist_lpw, *hist_lpg;       // [T][caps][beam]
  int hist_T = 0, hist_b = 0, hist_k = 0;
  int64_t* word_in = nullptr;        // [rows] scratch (teacher forcing / step)
  // attention capture (vsr_set_attention_capture): per step t, rows t * attn_step_rows .. of [R+1] weights and the
  // slot each row read; attn_path = the back-tracked rows of the returned beams [b][out_size][T]
  bool attn_capture = false;
  float* attn_alpha = nullptr; int32_t* attn_slot = nullptr; int32_t* attn_path = nullptr;
  size_t cap_attn_alpha = 0, cap_attn_slot = 0, cap_attn_path = 0;   // capacities in elements
  // what the last decode left for vsr_get_attention: captured (attn_ready), shape, and whether rows follow attn_path
  bool attn_ready = false, attn_beam = false;
  int attn_T = 0, attn_R = 0, attn_n_out = 0;
  int64_t attn_step_rows = 0;
  // bookkeeping
  int64_t launches = 0;
  bool profiling = false;
  Phase phases[PH_COUNT];
  std::vector<cudaEvent_t> step_ev;  // profiling: one event before every step of the last beam search + one after it
  std::vector<void*> owned;          // every cudaMalloc'd pointer (freed in destroy)
  // CUDA-graph cache of whole beam searches (api.cu).  A decode is ~140 launches with no host decision in
  // between; replaying it as one graph removes the per-launch cost (and its sensitivity to PCIe traffic).
  // Key = every value baked into the kernels' arguments; `epoch` changes whenever a device buffer is (re)allocated.
  struct GraphKey {
    uint64_t epoch;
    int64_t kind;                    // 0 = steps of a beam search, 1 = prologue, 2 = teacher-forced forward
    const void* captions;
    const void *det, *det_seqs, *slot_index, *verbs;
    int64_t det_stride, eos0, eos1;
    int32_t b, D, L, R, n_img, verbs_dtype, k, use_verbs, gt, T, attn, feat_dtype;
  };
  struct GraphEntry { GraphKey key; cudaGraphExec_t exec; int64_t launches; uint64_t last_use; };
  std::vector<GraphEntry> graphs;
  std::vector<GraphKey> graph_seen;  // keys decoded once eagerly; the second sighting captures
  uint64_t epoch = 0, graph_clock = 0;
  cudaStream_t cap_stream = nullptr;
  bool attend_attr_set = false;
  bool sample_attr_set = false;     // k_sample_pick may take up to 192 KB of dynamic shared memory
  bool state_h32 = true;             // the last step wrote fp32 h1'/h2' (always on the FFMA twin)
  bool use_graphs = true;            // VSRDEC_GRAPH=0 disables
  bool zero_state_opt = true;        // VSRDEC_ZERO_STATE=0: run the h-dependent GEMM parts at t = 0 although h = 0
  bool use_pdl = true;               // VSRDEC_PDL=0: plain stream serialization between the step kernels
  // VSRDEC_PDL_MODE bits: 1 = GEMM launches, 2 = small kernels, 4 = weight prefetch before the wait, 8 = GEMMs
  // trigger after their main loop.  Measured inside the decode graph (ms per decode): off 4.07, 1: 4.02, 1|4: 4.00,
  // 1|2|4: 4.18 (early-resident CTAs of the many-CTA kernels pile up on the SMs that drain first), 1|2|8: 4.08.
  int pdl_mode = 5;
};

int dev_alloc(Ctx* c, void** p, size_t bytes, bool zero = true);

struct PhaseScope {  // records start/stop events around a phase when profiling is on
  Ctx* c; int id; cudaStream_t st;
  PhaseScope(Ctx* c_, int id_, cudaStream_t st_);
  ~PhaseScope();
};

// ---------------------------------------------------------------- kernels (defined in *.cu)
int pack_weights(Ctx* c, const float* const* w, cudaStream_t st);
int run_prologue(Ctx* c, const void* det, int64_t det_stride, cudaStream_t st);
int run_prologue_indexed(Ctx* c, const void* det, int64_t det_stride, cudaStream_t st);
int ensure_rows(Ctx* c, int rows);
int ensure_beam_ws(Ctx* c, int caps, int T);
int ensure_sel(Ctx* c, int rows);

struct StepIO {
  int rows;          // rows processed this step
  int cur_beam;      // rows per caption
  bool use_verbs, gt;
  float* out_logp;   // optional full log-prob rows
  int64_t out_stride;
  float* gate_out;   // optional (rows,2) post-forcing gate log-probs
  int64_t gate_stride;
  int topk;          // number of word candidates to extract per row (0 = none)
  bool zero_state;   // h1 = h2 = 0 on entry (first step after init_state): their GEMM contributions are skipped
  bool skip_vocab;   // stop after LSTM cell 2 (batched teacher-forced forward: out_fc + log-softmax run once after the loop)
  bool need_h32;     // the caller reads the fp32 h1'/h2' (vsr_step); the tensor-core path itself only needs the fp16 twins
  float* attn_alpha;    // optional [rows][R+1] attention weights of the step (capture), with ...
  int32_t* attn_slot;   // ... [rows] the slot each row read; both null when capture is off
};
int run_step(Ctx* c, const StepIO& io, cudaStream_t st);

int launch_state_init(Ctx* c, int rows, cudaStream_t st);
int launch_words(Ctx* c, const int64_t* words, int rows, cudaStream_t st);
int launch_beam_step(Ctx* c, int t, int b, int cur, int k, int64_t eos0, int64_t eos1,
                     const int32_t* f_beam, const int32_t* f_word, const int32_t* f_gate, bool advance,
                     cudaStream_t st);
int launch_backtrack(Ctx* c, int b, int k, int T, int out_size, int64_t* out_words,
                     int64_t* out_gates, float* lp_words, float* lp_gates, int32_t* path_row, cudaStream_t st);
int launch_attn_gather(Ctx* c, const int32_t* path_row, int n_out, int T, float* alpha, int32_t* slot, cudaStream_t st);
int launch_commit_identity(Ctx* c, int rows, const int64_t* next_words, int64_t word_stride,
                           int next_slot, cudaStream_t st);
int launch_greedy_pick(Ctx* c, int rows, int t, int T, int64_t* out_words, int64_t* out_gates,
                       cudaStream_t st);
// draws of the sampling decode: rows = captions * p.n, row = caption * p.n + draw
int launch_sample_pick(Ctx* c, int rows, int t, int T, const VsrSampleParams& p, int64_t* out_words,
                       int64_t* out_gates, float* lp_words, float* lp_gates, cudaStream_t st);
int launch_gate_head(Ctx* c, int rows, float* gate_out, int64_t gate_stride, cudaStream_t st);
int launch_rows_to_all(Ctx* c, const F16Pair& src, const F16Pair& dst, int rows, int T, int t, cudaStream_t st);
int run_vocab_rows(Ctx* c, const F16Pair& a_b, float* logits, int M, float* out_logp, cudaStream_t st, bool softmax_only);

}  // namespace vsr
