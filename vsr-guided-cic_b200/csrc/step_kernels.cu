// Per-step kernels of the role-shift decoder: LSTM-cell / gate pointwise math, the slot
// attention + shift-gate kernel, and the fused log-softmax + verb forcing + per-row top-k.
// Reference math: models/controllable_captioning.py:117-190 (step) and :192-297 (step_v);
// algebra and buffer names follow SURVEY.md Appendix A.
#include <float.h>
#include <math.h>

#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>
#include <type_traits>
#include "common.cuh"
#include "vocab_head.cuh"

namespace vsr {

namespace {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// store the tensor-core twins of one value (the FFMA-twin path never has any: o.hi == null there)
using PairOut = TwinOut;
__device__ __forceinline__ void store_pair(const PairOut& o, size_t i, float v) {
  if (o.hi == nullptr) return;
  v = fminf(fmaxf(v * o.scale, -65504.f), 65504.f);   // fp16 range (saturate, never inf)
  const __half h = __float2half_rn(v);
  reinterpret_cast<__half*>(o.hi)[i] = h;
  const float r = v - __half2float(h);
  if (o.lo != nullptr) reinterpret_cast<__half*>(o.lo)[i] = __float2half_rn(r);
  if (o.hi8 != nullptr) {
    o.hi8[i] = (uint8_t)__nv_cvt_float_to_fp8(__half2float(h) * 0.03125f, __NV_SATFINITE, __NV_E4M3);
    o.lo8[i] = (uint8_t)__nv_cvt_float_to_fp8(r * 32.f, __NV_SATFINITE, __NV_E4M3);
  }
}


// ---------------------------------------------------------------- LSTM cell 1 + sentinel gate
// (FFMA-twin path; the tensor-core path runs this math in the GEMM-A epilogue.)
// pre1 columns are gate-interleaved: gate g of unit u at cell_col(g, u, 6); gates i,f,g,o,s,gq.
// c1' = sig(f) c1 + sig(i) tanh(g); h1' = sig(o) tanh(c1'); s_t = sig(s) tanh(c1')   (:151-154)
__global__ void k_lstm1(const float* __restrict__ pre1, int ld_pre, const float* __restrict__ c1,
                        float* __restrict__ h1n, float* __restrict__ c1n, float* __restrict__ s_t,
                        float* __restrict__ gq, PairOut h1n_b, PairOut s_t_b, int ld, int H, int rows) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (u >= H || n >= rows) return;
  const float* p = pre1 + (size_t)n * ld_pre;
  const float ig = sigmoidf_(p[cell_col(0, u, 6)]), fg = sigmoidf_(p[cell_col(1, u, 6)]),
              gg = tanhf(p[cell_col(2, u, 6)]), og = sigmoidf_(p[cell_col(3, u, 6)]),
              sg = sigmoidf_(p[cell_col(4, u, 6)]);
  gq[(size_t)n * ld + u] = p[cell_col(5, u, 6)];
  const float c = fg * c1[(size_t)n * ld + u] + ig * gg;
  const float tc = tanhf(c);
  c1n[(size_t)n * ld + u] = c;
  const float hv = og * tc, sv = sg * tc;
  h1n[(size_t)n * ld + u] = hv;
  s_t[(size_t)n * ld + u] = sv;
  store_pair(h1n_b, (size_t)n * ld + u, hv);
  store_pair(s_t_b, (size_t)n * ld + u, sv);
}

// g_t = sig(gq + hg) * tanh(c1')   (:181-182; hg = W1_hg . h1' comes from the h1' GEMM)
__global__ void k_gt(const float* __restrict__ gq_in, const float* __restrict__ hb, int ld_hb,
                     const float* __restrict__ c1n, float* __restrict__ g_t, PairOut g_t_b, int ld, int H,
                     int rows) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (u >= H || n >= rows) return;
  const float gq = gq_in[(size_t)n * ld + u] + hb[(size_t)n * ld_hb + u];
  const float gv = sigmoidf_(gq) * tanhf(c1n[(size_t)n * ld + u]);
  g_t[(size_t)n * ld + u] = gv;
  store_pair(g_t_b, (size_t)n * ld + u, gv);
}

// LSTM cell 2 (FFMA-twin path): pre2 columns gate-interleaved, cell_col(g, u, 4)   (:177 / :258)
__global__ void k_lstm2(const float* __restrict__ pre2, int ld_pre, const float* __restrict__ c2,
                        float* __restrict__ h2n, float* __restrict__ c2n, PairOut h2n_b, int ld, int H,
                        int rows) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (u >= H || n >= rows) return;
  const float* p = pre2 + (size_t)n * ld_pre;
  const float ig = sigmoidf_(p[cell_col(0, u, 4)]), fg = sigmoidf_(p[cell_col(1, u, 4)]),
              gg = tanhf(p[cell_col(2, u, 4)]), og = sigmoidf_(p[cell_col(3, u, 4)]);
  const float c = fg * c2[(size_t)n * ld + u] + ig * gg;
  c2n[(size_t)n * ld + u] = c;
  const float hv = og * tanhf(c);
  h2n[(size_t)n * ld + u] = hv;
  store_pair(h2n_b, (size_t)n * ld + u, hv);
}

// ---------------------------------------------------------------- slot attention + shift gate
// One CTA per row.  Reads only the VALID region rows of the row's current slot tile
// det_seqs[caption, ptr] (128-bit coalesced loads) plus their hoisted att_va projections P.
//   e_r   = att_a . tanh(P_r + ha)            (padding rows: P_r = 0)          :161-162
//   e_s   = att_s . tanh(sa + ha)                                              :163-164
//   alpha = softmax([e_s, e_0..e_{R-1}]) * mask ; alpha /= sum(alpha)          :167-169
//   att   = alpha_s * sentinel + sum_r alpha_r * region_r                      :171
//   gate  = log_softmax([att_g . tanh(ga + ha), sum_{valid r} e_r])            :184-188
constexpr int ATT_THREADS = 256;
constexpr int ATT_MAX_R = 64;

struct AttendArgs {
  // caller features det_seqs / det: element type feat_dtype (VSR_DT_F32 / F16 / BF16), the Elem of k_attend<Elem>
  const void* det_seqs;    // (b, L, R, F) materialised slot tiles, or null in index form
  const float* P;          // materialised: [b*L*R][ldP]; index form: [n_img*D][ldP] (per detection row)
  // index form (vsr_prologue_indexed): region = det[img][idx] (idx >= 0) or the image mean row (idx == -2, fp32
  // whatever Elem is: the mean is computed in fp32 by k_pool)
  const int32_t* slot_index; const void* det; int64_t det_stride; int D;
  const float* img; int ld_img; const float* Pmean; int img_mul;
  const unsigned long long* slot_mask;  // [b*L] validity bits of each slot tile
  const int32_t* slot_base;             // [b*L] first P row of the slot when only valid rows were projected, or null
  const int32_t* ptr;      // [rows]
  const float* sent; int ld_sent; int o_sa;   // sentinel (F) at 0 | sa (A) at o_sa
  const float* hb; int ld_hb; int o_ha;       // hg (H) at 0 | ha (A) at o_ha | ...
  const float *v_a, *v_s;
  float* att; int ld_att;
  PairOut att_b;
  float* shift;            // [rows] sum of the valid region scores = the "shift" gate logit (:187)
  // attention capture (null = off): the row's R+1 weights after the masked renormalisation, column 0 = sentinel,
  // column r+1 = region r of the slot it reads ([rows][R+1]), and that slot ([rows])
  float* alpha_out; int32_t* slot_out;
  int rows, cur_beam, L, R, F, A, H, ldP;
  int feat_dtype;
};

template <typename Elem>
__global__ void __launch_bounds__(ATT_THREADS) k_attend(const AttendArgs a) {
  constexpr bool f32 = std::is_same<Elem, float>::value;
  extern __shared__ __align__(16) float sm[];
  float* ha = sm;                       // [A]
  float* Ps = ha + a.A;                 // [R][A] att_va projections of the slot's valid regions (cp.async)
  float* e = Ps + (size_t)a.R * a.A;    // [R+1] scores, later alpha; index 0 = sentinel
  __shared__ float red[ATT_THREADS / 32];
  __shared__ float s_pad;
  __shared__ int s_rows[ATT_MAX_R];     // compacted valid region rows and their weights
  __shared__ float s_w[ATT_MAX_R];
  __shared__ int s_nv;
  __shared__ const void* s_feat[ATT_MAX_R];    // feature row of every region of the slot
  // half-precision features: 1 = the row is fp32 (the index form's image mean row), 0 = a row of Elem
  __shared__ uint8_t s_row_f32[f32 ? 1 : ATT_MAX_R];

  const int n = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int nwarp = ATT_THREADS / 32;
#ifdef VSR_DBG_CLK
  long long tk[8]; int nt = 0;
#define TICK() do { if (lane == 0) tk[nt++] = clock64(); } while (0)
#else
#define TICK() do {} while (0)
#endif
  TICK();
  pdl_trigger();
  pdl_wait();          // every input of this kernel comes from the step's earlier kernels
  const int cap = n / a.cur_beam;
  const float* sent = a.sent + (size_t)n * a.ld_sent;   // sentinel feature row
  const float* sa = sent + a.o_sa;
  // loads that depend only on the row index go first so that they overlap the ptr -> mask chain
  float4 sent_v[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int f = tid * 4 + u * ATT_THREADS * 4;
    sent_v[u] = f < a.F ? *reinterpret_cast<const float4*>(sent + f) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float ha_v[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int i = tid + u * ATT_THREADS;
    ha_v[u] = i < a.A ? a.hb[(size_t)n * a.ld_hb + a.o_ha + i] : 0.f;
  }
  // all L slot masks of the caption are fetched alongside the slot pointer; the right one is picked by shuffle
  unsigned long long vmask;
  int slot;
  int pbase = -1;                       // compact form: P row of the slot's first valid region
  if (a.L <= 32) {
    const unsigned long long ml = lane < a.L ? a.slot_mask[(size_t)cap * a.L + lane] : 0ull;
    const int bl = (a.slot_base != nullptr && lane < a.L) ? a.slot_base[(size_t)cap * a.L + lane] : -1;
    slot = a.ptr[n];
    vmask = __shfl_sync(0xffffffffu, ml, slot);
    pbase = __shfl_sync(0xffffffffu, bl, slot);
  } else {
    slot = a.ptr[n];
    vmask = a.slot_mask[(size_t)cap * a.L + slot];
    if (a.slot_base != nullptr) pbase = a.slot_base[(size_t)cap * a.L + slot];
  }
  const size_t tile_row0 = ((size_t)cap * a.L + slot) * a.R;
  const int imgi = cap * a.img_mul;

  // stage the valid regions' projections with cp.async (16-byte chunks, no registers held) and pull the
  // valid feature rows towards L2 while the scores are computed; one warp per region row, no divisions
  for (int r = warp; r < a.R; r += nwarp) {
    if (!((vmask >> r) & 1ull)) continue;
    const float* prow;
    const void* frow;
    bool row_f32 = f32;
    if (a.slot_index == nullptr) {
      prow = a.P + (pbase >= 0 ? (size_t)(pbase + __popcll(vmask & ((1ull << r) - 1ull))) : tile_row0 + r) * a.ldP;
      frow = static_cast<const Elem*>(a.det_seqs) + (tile_row0 + r) * a.F;
    } else {
      const int idx = a.slot_index[tile_row0 + r];
      if (idx >= 0) {
        prow = a.P + ((size_t)imgi * a.D + idx) * a.ldP;
        frow = static_cast<const Elem*>(a.det) + (size_t)imgi * a.det_stride + (size_t)idx * a.F;
      } else {
        prow = a.Pmean + (size_t)imgi * a.ldP;
        frow = a.img + (size_t)imgi * a.ld_img;
        row_f32 = true;
      }
    }
    if (lane == 0) {
      s_feat[r] = frow;
      if constexpr (!f32) s_row_f32[r] = row_f32 ? 1 : 0;
    }
    float* pdst = Ps + (size_t)r * a.A;
    for (int ch = lane * 4; ch < a.A; ch += 128) {
      const unsigned dst = (unsigned)__cvta_generic_to_shared(pdst + ch);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(prow + ch) : "memory");
    }
    // one 128-byte line per lane: the row is F * sizeof(element) bytes
    if constexpr (f32) {
      for (int f = lane * 32; f < a.F; f += 32 * 32)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(static_cast<const float*>(frow) + f));
    } else {
      const int bytes = a.F * (row_f32 ? (int)sizeof(float) : (int)sizeof(Elem));
      for (int o = lane * 128; o < bytes; o += 32 * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(static_cast<const char*>(frow) + o));
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int i = tid + u * ATT_THREADS;
    if (i < a.A) ha[i] = ha_v[u];
  }
  for (int i = tid + 2 * ATT_THREADS; i < a.A; i += ATT_THREADS) ha[i] = a.hb[(size_t)n * a.ld_hb + a.o_ha + i];
  // sum of the sentinel row (its mask is computed like any region row, :159)
  float ssum = ((sent_v[0].x + sent_v[0].y) + (sent_v[0].z + sent_v[0].w)) + ((sent_v[1].x + sent_v[1].y) + (sent_v[1].z + sent_v[1].w));
  for (int f = tid * 4 + 2 * ATT_THREADS * 4; f < a.F; f += ATT_THREADS * 4) {
    const float4 v = *reinterpret_cast<const float4*>(sent + f);
    ssum += (v.x + v.y) + (v.z + v.w);
  }
  ssum = warp_sum(ssum);
  if (lane == 0) red[warp] = ssum;
  TICK();
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  TICK();

  // scores: job 0 = sentinel, 1 = padding-row score, 2.. = valid regions; one warp per job
  for (int job = warp; job < a.R + 2; job += nwarp) {
    const float* add = nullptr;
    const float* vec = a.v_a;
    if (job == 0) { add = sa; vec = a.v_s; }
    else if (job >= 2) {
      const int r = job - 2;
      if (!((vmask >> r) & 1ull)) continue;
      add = Ps + (size_t)r * a.A;
    }
    float acc = 0.f;
    for (int i0 = 0; i0 < a.A; i0 += 512) {     // 4 x float4 per lane in flight, then the tanh math
      float4 pv[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = i0 + q * 128 + lane * 4;
        pv[q] = (add != nullptr && i < a.A) ? *reinterpret_cast<const float4*>(add + i)
                                             : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = i0 + q * 128 + lane * 4;
        if (i < a.A) {
          const float4 hv = *reinterpret_cast<const float4*>(ha + i);
          const float4 vv = __ldg(reinterpret_cast<const float4*>(vec + i));
          acc += vv.x * fast_tanh(pv[q].x + hv.x) + vv.y * fast_tanh(pv[q].y + hv.y) +
                 vv.z * fast_tanh(pv[q].z + hv.z) + vv.w * fast_tanh(pv[q].w + hv.w);
        }
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      if (job == 0) e[0] = acc;
      else if (job == 1) s_pad = acc;       // score shared by all padding rows
      else e[job - 1] = acc;
    }
  }
  TICK();
  __syncthreads();

  if (warp == 0) {
    float sent_sum = 0.f;
    for (int w = 0; w < nwarp; ++w) sent_sum += red[w];
    if (a.R + 1 <= 32) {
      // masked softmax over [sentinel, regions] with one lane per entry (:167-169)
      const bool in = lane <= a.R;
      const bool valid = in && (lane == 0 ? (sent_sum != 0.f) : (((vmask >> (lane - 1)) & 1ull) != 0));
      const bool region = in && lane >= 1 && valid;
      float ev = -INFINITY;
      if (in) ev = (lane == 0 || valid) ? e[lane] : s_pad;
      const float m = warp_max(ev);
      float w = in ? expf(ev - m) : 0.f;
      const float S = warp_sum(w);
      w = valid ? w / S : 0.f;
      const float T = warp_sum(w);
      w = w / T;
      const float shift = warp_sum(region ? ev : 0.f);
      if (a.alpha_out != nullptr && in) a.alpha_out[(size_t)n * (a.R + 1) + lane] = w;
      const unsigned msk = __ballot_sync(0xffffffffu, region);
      if (region) { const int pos = __popc(msk & ((1u << lane) - 1u)); s_rows[pos] = lane - 1; s_w[pos] = w; }
      if (lane == 0) {
        e[0] = w; s_nv = __popc(msk); a.shift[n] = shift;
        if (a.slot_out != nullptr) a.slot_out[n] = slot;
      }
    } else if (lane == 0) {
      const float e_pad = s_pad;
      float m = e[0];
      float shift = 0.f;
      for (int r = 0; r < a.R; ++r) {
        if (!((vmask >> r) & 1ull)) e[r + 1] = e_pad; else shift += e[r + 1];
        m = fmaxf(m, e[r + 1]);
      }
      float S = 0.f;
      for (int r = 0; r <= a.R; ++r) { e[r] = expf(e[r] - m); S += e[r]; }
      float T = 0.f;
      for (int r = 0; r <= a.R; ++r) {
        const bool valid = (r == 0) ? (sent_sum != 0.f) : (((vmask >> (r - 1)) & 1ull) != 0);
        e[r] = valid ? e[r] / S : 0.f;
        T += e[r];
      }
      int nv = 0;
      for (int r = 0; r <= a.R; ++r) {
        e[r] = e[r] / T;
        if (r > 0 && ((vmask >> (r - 1)) & 1ull)) { s_rows[nv] = r - 1; s_w[nv] = e[r]; ++nv; }
      }
      s_nv = nv;
      a.shift[n] = shift;    // the gate head is finished in k_softmax_topk (needs the att_ga projection)
      if (a.alpha_out != nullptr) {
        for (int r = 0; r <= a.R; ++r) a.alpha_out[(size_t)n * (a.R + 1) + r] = e[r];
        a.slot_out[n] = slot;
      }
    }
  }
  __syncthreads();

  TICK();
  // weighted sum over sentinel + valid regions: each thread owns two float4 columns, 4 rows x 2 columns
  // (8 independent 128-bit loads) in flight
  float* out = a.att != nullptr ? a.att + (size_t)n * a.ld_att : nullptr;
  const float a_s = e[0];
  const int nv = s_nv;
  for (int f0 = tid * 4; f0 < a.F; f0 += ATT_THREADS * 8) {
    const int f1 = f0 + ATT_THREADS * 4;
    const bool two = f1 < a.F;
    const float4 s0 = *reinterpret_cast<const float4*>(sent + f0);
    const float4 s1 = two ? *reinterpret_cast<const float4*>(sent + f1) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 acc0 = make_float4(a_s * s0.x, a_s * s0.y, a_s * s0.z, a_s * s0.w);
    float4 acc1 = make_float4(a_s * s1.x, a_s * s1.y, a_s * s1.z, a_s * s1.w);
    for (int i = 0; i < nv; i += 4) {
      float4 v0[4], v1[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int row = s_rows[min(i + u, nv - 1)];
        if (f32 || s_row_f32[row]) {
          const float* rp = static_cast<const float*>(s_feat[row]);
          v0[u] = __ldg(reinterpret_cast<const float4*>(rp + f0));
          v1[u] = two ? __ldg(reinterpret_cast<const float4*>(rp + f1)) : make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
          const Elem* rp = static_cast<const Elem*>(s_feat[row]);
          v0[u] = ldg_feat4(rp + f0);
          v1[u] = two ? ldg_feat4(rp + f1) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float w = (i + u < nv) ? s_w[i + u] : 0.f;
        acc0.x += w * v0[u].x; acc0.y += w * v0[u].y; acc0.z += w * v0[u].z; acc0.w += w * v0[u].w;
        acc1.x += w * v1[u].x; acc1.y += w * v1[u].y; acc1.z += w * v1[u].z; acc1.w += w * v1[u].w;
      }
    }
    if (out != nullptr) *reinterpret_cast<float4*>(out + f0) = acc0;
    store_twin4(a.att_b, (size_t)n * a.ld_att + f0, acc0);
    if (two) {
      if (out != nullptr) *reinterpret_cast<float4*>(out + f1) = acc1;
      store_twin4(a.att_b, (size_t)n * a.ld_att + f1, acc1);
    }
  }
  TICK();
#ifdef VSR_DBG_CLK
  if (lane == 0 && (n == 7 || n == 301) && (warp == 0 || warp == 5))
    printf("attend n=%d warp=%d nv=%d: setup %lld  wait+bar %lld  scores %lld  bar+softmax+bar %lld  wsum %lld\n", n, warp, nv,
           tk[1] - tk[0], tk[2] - tk[1], tk[3] - tk[2], tk[4] - tk[3], tk[5] - tk[4]);
#endif
}

// ---------------------------------------------------------------- log-softmax + gate head + verb forcing + top-k
// One CTA per row; the row's logits are read ONCE into registers.  Also finishes the
// shift-gate head (stay logit = att_g . tanh(ga + ha), controllable_captioning.py:184-188) so the
// att_ga projection is off the attention kernel's critical path, and applies verb forcing (:271-295).

// One pass over the row (each thread: its float4s in register batches): online (max, sum exp) per thread,
// merged block-wide, plus the thread's two best elements.  Every warp then picks the top-k of its 64
// candidates with redux.sync rounds (no shuffles trees, no barriers), and after the single block barrier
// warp 0 merges the 8 x k survivors the same way.  That is exact unless one thread owns three of the
// top-k, which the final pick reveals (a thread's SECOND candidate chosen); such rows (~1e-4 of them)
// take the slow exact path: k rounds of block arg-best with the owner rescanning its elements.
// Serial single-warp sections are kept to a few hundred cycles: they dominated earlier versions.
constexpr int SM_THREADS = 256;

__global__ void __launch_bounds__(SM_THREADS) k_softmax_topk(const SoftmaxArgs a) {
  constexpr int THREADS = SM_THREADS;
  constexpr int NW = THREADS / 32;
  __shared__ float red_m[NW], red_s[NW], red_g[NW];
  __shared__ float wl_v[NW][VSR_MAX_BEAM];      // per-warp top-k lists
  __shared__ int wl_i[NW][VSR_MAX_BEAM];
  __shared__ int wl_second[NW][VSR_MAX_BEAM];
  __shared__ float red_v[2][NW];
  __shared__ int red_i[2][NW];
  __shared__ int s_forced, s_slow;
  __shared__ int s_pick[VSR_MAX_BEAM];
  const int n = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_trigger();
  pdl_wait();
  const float* x = a.logits + (size_t)n * a.ld;
  const int V = a.V;
  const int n4 = (V + 3) >> 2;
  const int topk = a.topk;

  // thread 0 starts its dependent loads early (slot pointer -> verb id, shift logit)
  int64_t verb = -1; float shift_logit = 0.f;
  const bool gate_head = a.ha != nullptr;      // null: log-softmax of the vocabulary rows only (batched forward)
  if (tid == 0 && gate_head) {
    shift_logit = a.shift[n];
    if (a.use_verbs && a.verbs != nullptr)
      verb = load_verb(a.verbs, a.verbs_dtype, (size_t)(n / a.cur_beam) * a.L + a.ptr[n]);
  }

  // stay-gate logit att_g . tanh(ga + ha): every thread takes a slice (loads issued before the row scan)
  float stay_part = 0.f;
  if (gate_head) {
    const float* ha = a.ha + (size_t)n * a.ld_ha;
    const float* ga = a.ga + (size_t)n * a.ld_ga;
    for (int i = tid; i < a.A; i += THREADS) stay_part += a.v_g[i] * fast_tanh(ga[i] + ha[i]);
  }
  float v1 = -INFINITY, v2 = -INFINITY; int i1 = 0x7fffffff, i2 = 0x7fffffff;   // this thread's two best
  float m = -INFINITY, ssum = 0.f;
  constexpr int PRE = 5;
  for (int j0 = tid; j0 < n4; j0 += THREADS * PRE) {
    float4 q[PRE];
#pragma unroll
    for (int u = 0; u < PRE; ++u) {
      const int j = j0 + u * THREADS;
      q[u] = j < n4 ? *reinterpret_cast<const float4*>(x + j * 4) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
    float bm = -INFINITY;
#pragma unroll
    for (int u = 0; u < PRE; ++u) {
      const int v0 = (j0 + u * THREADS) * 4;
      if (v0 + 3 >= V) {                        // only the row's last float4 (or an out-of-range one) needs masking
        if (v0 + 1 >= V) q[u].y = -INFINITY;
        if (v0 + 2 >= V) q[u].z = -INFINITY;
        q[u].w = -INFINITY;
        if (v0 >= V) q[u].x = -INFINITY;
      }
      const float e4[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float val = e4[e];
        bm = fmaxf(bm, val);
        if (val > v2) {                         // strict: equal values keep the earlier (smaller) index
          if (val > v1) { v2 = v1; i2 = i1; v1 = val; i1 = v0 + e; } else { v2 = val; i2 = v0 + e; }
        }
      }
    }
    if (bm > m) { ssum *= __expf(m - bm); m = bm; }
    if (m > -INFINITY) {
#pragma unroll
      for (int u = 0; u < PRE; ++u)
        ssum += (__expf(q[u].x - m) + __expf(q[u].y - m)) + (__expf(q[u].z - m) + __expf(q[u].w - m));   // exp(-inf) = 0
    }
  }
  {
    const float wm = warp_max(m);
    const float ws = warp_sum(m > -INFINITY ? ssum * expf(m - wm) : 0.f);
    const float wg = warp_sum(stay_part);
    if (lane == 0) { red_m[warp] = wm; red_s[warp] = ws; red_g[warp] = wg; }
  }
  // warp-level top-k of the warp's 64 candidates
  {
    int head = 0;
    for (int j = 0; j < topk; ++j) {
      const float hv = head == 0 ? v1 : (head == 1 ? v2 : -INFINITY);
      const int hi = head == 0 ? i1 : (head == 1 ? i2 : 0x7fffffff);
      unsigned kb; int ib;
      warp_argbest_redux(hv, hi, kb, ib);
      const bool mine = hi == ib && ib != 0x7fffffff;
      if (mine) { wl_v[warp][j] = hv; wl_i[warp][j] = hi; wl_second[warp][j] = head; ++head; }
      if (ib == 0x7fffffff && lane == 0) { wl_v[warp][j] = -INFINITY; wl_i[warp][j] = 0x7fffffff; wl_second[warp][j] = 0; }
    }
  }
  if (tid == 0) s_slow = 0;
  __syncthreads();

  float mx = red_m[0];
#pragma unroll
  for (int w = 1; w < NW; ++w) mx = fmaxf(mx, red_m[w]);
  float se = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) se += red_s[w] * expf(red_m[w] - mx);
  const float lsum = logf(se);

  if (warp == 0) {
    // merge the NW per-warp lists (NW * topk <= 64 entries: two per lane)
    float cvv[2] = {-INFINITY, -INFINITY}; int cii[2] = {0x7fffffff, 0x7fffffff}; int csec[2] = {0, 0};
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int e = lane + 32 * q;
      if (e < NW * topk) { cvv[q] = wl_v[e / topk][e % topk]; cii[q] = wl_i[e / topk][e % topk]; csec[q] = wl_second[e / topk][e % topk]; }
    }
    int slow = 0;
    for (int j = 0; j < topk; ++j) {
      const bool first = before(cvv[0], cii[0], cvv[1], cii[1]);
      const float hv = first ? cvv[0] : cvv[1];
      const int hi = first ? cii[0] : cii[1];
      unsigned kb; int ib;
      warp_argbest_redux(hv, hi, kb, ib);
      if (hi == ib && ib != 0x7fffffff) {
        slow |= first ? csec[0] : csec[1];
        if (first) { cvv[0] = -INFINITY; cii[0] = 0x7fffffff; } else { cvv[1] = -INFINITY; cii[1] = 0x7fffffff; }
      }
      if (lane == 0) s_pick[j] = ib;
    }
    slow = __any_sync(0xffffffffu, slow != 0);
    if (lane == 0) s_slow = slow;
  }

  if (tid == 0) {
    // verb forcing (:271-295): which vocabulary index does the current slot force, if any
    int forced = -1;
    if (verb != -1) {
      if (a.gt) {
        forced = (int)verb;
      } else {
        forced = 0;   // key missing or empty list -> vocabulary index 0 (:291-292)
        int lo = 0, hi = a.vt_n - 1, pos = -1;
        while (lo <= hi) {
          const int mid = (lo + hi) >> 1;
          const int64_t k = a.vt_keys[mid];
          if (k == verb) { pos = mid; break; }
          if (k < verb) lo = mid + 1; else hi = mid - 1;
        }
        if (pos >= 0 && a.vt_off[pos + 1] > a.vt_off[pos]) {
          float best = -1e6f; int best_i = -1;    // strict '>' : first maximum wins (:284-289)
          for (int qq = a.vt_off[pos]; qq < a.vt_off[pos + 1]; ++qq) {
            const int idx = a.vt_idx[qq];
            const float lp = (x[idx] - mx) - lsum;
            if (lp > best) { best = lp; best_i = idx; }
          }
          forced = best_i < 0 ? V - 1 : best_i;   // python index -1 == last vocabulary entry
        }
      }
      forced = min(max(forced, 0), V - 1);
    }
    s_forced = forced;
    if (gate_head) {
    a.row_max[n] = mx;
    a.row_lsum[n] = lsum;
    a.forced[n] = forced;
    // gate head: log_softmax([stay, shift]) (:187-188), or [-1e3, 0] on a verb slot (:295)
    float g0, g1;
    if (forced >= 0) { g0 = -1e3f; g1 = 0.f; }
    else {
      float stay = 0.f;
#pragma unroll
      for (int w = 0; w < NW; ++w) stay += red_g[w];
      const float gm = fmaxf(stay, shift_logit);
      const float ls = logf(expf(stay - gm) + expf(shift_logit - gm));
      g0 = (stay - gm) - ls; g1 = (shift_logit - gm) - ls;
    }
    a.gate_lp[(size_t)n * 2] = g0; a.gate_lp[(size_t)n * 2 + 1] = g1;
    if (a.gate_out != nullptr) {
      a.gate_out[(size_t)n * a.gate_stride + 0] = g0;
      a.gate_out[(size_t)n * a.gate_stride + 1] = g1;
    }
    }
  }
  if (a.out_logp == nullptr && topk <= 0) return;
  __syncthreads();
  const int forced = s_forced;

  if (a.out_logp != nullptr) {
    float* o = a.out_logp + (size_t)n * a.out_stride;
    for (int v = tid; v < V; v += THREADS)
      o[v] = forced >= 0 ? (v == forced ? 0.f : -1e6f) : (x[v] - mx) - lsum;
  }
  if (topk <= 0) return;

  int32_t* cd = a.cand + (size_t)n * VSR_MAX_BEAM;
  if (forced >= 0) {
    // forced word first, then the lowest other indices (all tied at -1e6)
    if (tid == 0) {
      cd[0] = forced;
      int v = 0;
      for (int j = 1; j < topk; ++j) { if (v == forced) ++v; cd[j] = min(v, V - 1); ++v; }
    }
    return;
  }
  if (!s_slow) {
    if (tid < topk) cd[tid] = s_pick[tid];
    return;
  }
  // ---- slow exact path (block-uniform): k rounds of block arg-best, owners rescan from global memory
  float cv = v1; int ci = i1;
  for (int j = 0; j < topk; ++j) {
    float bv = cv; int bi = ci;
    warp_argbest(bv, bi);
    if (lane == 0) { red_v[j & 1][warp] = bv; red_i[j & 1][warp] = bi; }
    __syncthreads();
    bv = red_v[j & 1][0]; bi = red_i[j & 1][0];
#pragma unroll
    for (int w = 1; w < NW; ++w)
      if (before(red_v[j & 1][w], red_i[j & 1][w], bv, bi)) { bv = red_v[j & 1][w]; bi = red_i[j & 1][w]; }
    if (tid == 0) cd[j] = bi;
    if (ci == bi) {   // owner: next best strictly after (bv, bi) among its own elements
      cv = -INFINITY; ci = 0x7fffffff;
      for (int jj = tid; jj < n4; jj += THREADS) {
        const float4 qq = *reinterpret_cast<const float4*>(x + jj * 4);
        const int v0 = jj * 4;
        const float e4[4] = {qq.x, qq.y, qq.z, qq.w};
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (v0 + u < V && before(bv, bi, e4[u], v0 + u) && before(e4[u], v0 + u, cv, ci)) { cv = e4[u]; ci = v0 + u; }
      }
    }
  }
}

constexpr int VM_WARPS = 4;
// k_vocab_merge: vocab_head.cuh (merge_row) — one warp per row finishes the vocabulary head from the GEMM's records
__global__ void __launch_bounds__(VM_WARPS * 32) k_vocab_merge(const SoftmaxArgs a, const float* __restrict__ vpart, int n_chunks) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * VM_WARPS + (threadIdx.x >> 5);
  pdl_trigger();
  pdl_wait();
  if (n >= a.rows) return;
  RowHead h;
  merge_row(a, vpart, n_chunks, n, lane, h);
  if (lane == 0) {
    a.row_max[n] = h.mx; a.row_lsum[n] = h.lsum; a.forced[n] = h.forced;
    a.gate_lp[(size_t)n * 2] = h.g0; a.gate_lp[(size_t)n * 2 + 1] = h.g1;
    if (a.gate_out != nullptr) {
      a.gate_out[(size_t)n * a.gate_stride + 0] = h.g0;
      a.gate_out[(size_t)n * a.gate_stride + 1] = h.g1;
    }
  }
  if (lane < a.topk) a.cand[(size_t)n * VSR_MAX_BEAM + lane] = h.pick;
}

// ---------------------------------------------------------------- batched teacher-forced forward helpers
// Gate head alone (no verb forcing), one warp per row: gate = log_softmax([att_g . tanh(ga + ha), shift])   (:184-188)
__global__ void __launch_bounds__(128) k_gate_head(const float* __restrict__ ha, int ld_ha, const float* __restrict__ ga, int ld_ga,
                                                   const float* __restrict__ v_g, int A, const float* __restrict__ shift,
                                                   float* __restrict__ gate_out, int64_t gate_stride, int rows) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (n >= rows) return;
  const float4* h4 = reinterpret_cast<const float4*>(ha + (size_t)n * ld_ha);
  const float4* g4 = reinterpret_cast<const float4*>(ga + (size_t)n * ld_ga);
  const float4* v4 = reinterpret_cast<const float4*>(v_g);
  float stay = 0.f;
  for (int i = lane; i < A / 4; i += 32) {
    const float4 h = h4[i], g = g4[i], w = __ldg(v4 + i);
    stay += (w.x * fast_tanh(g.x + h.x) + w.y * fast_tanh(g.y + h.y)) + (w.z * fast_tanh(g.z + h.z) + w.w * fast_tanh(g.w + h.w));
  }
  stay = warp_sum(stay);
  if (lane == 0) {
    const float sh = shift[n];
    const float gm = fmaxf(stay, sh);
    const float ls = logf(expf(stay - gm) + expf(sh - gm));
    gate_out[(size_t)n * gate_stride] = (stay - gm) - ls;
    gate_out[(size_t)n * gate_stride + 1] = (sh - gm) - ls;
  }
}

// dst row (i * T + t) <- src row i, for up to three raw twin arrays (16-byte vectors)
struct RowScatter { int n; const uint4* src[3]; uint4* dst[3]; int vec[3]; };
__global__ void __launch_bounds__(128) k_rows_to_all(const RowScatter r, int T, int t) {
  const int i = blockIdx.x;
  for (int q = 0; q < r.n; ++q) {
    const uint4* s = r.src[q] + (size_t)i * r.vec[q];
    uint4* d = r.dst[q] + ((size_t)i * T + t) * r.vec[q];
    for (int e = threadIdx.x; e < r.vec[q]; e += blockDim.x) d[e] = s[e];
  }
}

}  // namespace

int launch_gate_head(Ctx* c, int rows, float* gate_out, int64_t gate_stride, cudaStream_t st) {
  k_gate_head<<<(rows + 3) / 4, 128, 0, st>>>(c->hb + c->oB2_ha, c->NB2, c->ga, c->NC, c->v_g, c->A, c->shift, gate_out, gate_stride, rows);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

// twins of h2' (rows i) -> rows i * T + t of the all-steps operand of the batched vocabulary GEMM
int launch_rows_to_all(Ctx* c, const F16Pair& src, const F16Pair& dst, int rows, int T, int t, cudaStream_t st) {
  RowScatter r{};
  auto add = [&](const void* s, void* d, int bytes) {
    if (s == nullptr || d == nullptr) return;
    r.src[r.n] = (const uint4*)s; r.dst[r.n] = (uint4*)d; r.vec[r.n] = c->Hp * bytes / 16; ++r.n;
  };
  add(src.hi, dst.hi, 2); add(src.lo, dst.lo, 2); add(src.hi8, dst.hi8, 1); add(src.lo8, dst.lo8, 1);
  k_rows_to_all<<<rows, 128, 0, st>>>(r, T, t);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

// logits[M][NE] = out_fc . h2'[M] + b for M rows of an all-steps operand, then out[M][V] = log_softmax (full rows)
int run_vocab_rows(Ctx* c, const F16Pair& a_b, float* logits, int M, float* out_logp, cudaStream_t st, bool softmax_only) {
  if (!softmax_only) {
    PhaseScope ps(c, PH_GEMM_E, st);
    GemmArgs g{};
    g.nseg = 1; g.seg[0] = {nullptr, c->Hp, c->Hp, c->Hp, &a_b};
    g.w = c->WE; g.ldw = c->Hp; g.bias = c->bE; g.wb = &c->WE_b;
    g.c = logits; g.ldc = c->NE; g.M = M; g.N = c->NE;
    g.f8 = c->gemm_f8; g.allow_pair = true; g.no_alt = true;
    VSR_TRY(launch_gemm(c, g, st)); c->launches++;
    return VSR_OK;
  }
  PhaseScope ps(c, PH_SOFTMAX_TOPK, st);
  SoftmaxArgs a{};
  a.logits = logits; a.ld = c->NE; a.rows = M; a.V = c->V; a.cur_beam = 1; a.L = c->L; a.topk = 0;
  a.out_logp = out_logp; a.out_stride = c->V;
  k_softmax_topk<<<M, SM_THREADS, 0, st>>>(a);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

// ---------------------------------------------------------------- one decoder step (host side)
static PairOut pair_out(const Ctx* c, const F16Pair& b) { return twin_out(&b, c->use_tc); }

int run_step(Ctx* c, const StepIO& io, cudaStream_t st) {
  const int rows = io.rows, H = c->H;
  VSR_REQUIRE(rows > 0 && rows <= c->cap_rows, VSR_ESTATE, "run_step: rows=%d cap=%d", rows, c->cap_rows);
  VSR_REQUIRE(c->R <= ATT_MAX_R, VSR_EINVAL, "max_detections per slot R=%d > %d", c->R, ATT_MAX_R);
  const bool h2f = c->d.h2_first_lstm != 0;
  const dim3 pw_grid((H + 127) / 128, rows);
  bool fused = false;   // tensor-core path: cell / gate pointwise math runs inside the GEMM epilogues

  {  // A: pre1 = [h2 | h1_old] . WA^T + U[img] + X[word]
    PhaseScope ps(c, PH_GEMM_A, st);
    GemmArgs g{};
    int s = 0;
    if (h2f) g.seg[s++] = {c->h2, c->Hp, c->Hp, c->Hp, &c->h2_b};
    g.seg[s++] = {c->h1, c->Hp, c->Hp, c->Hp, &c->h1_b};
    g.nseg = s;
    g.w = c->WA; g.ldw = c->KA; g.wb = &c->WA_b;
    g.gather = c->X; g.ld_gather = c->NA; g.gather_idx = c->word_idx;
    g.rowadd = c->U; g.ld_rowadd = c->NA; g.row_div = io.cur_beam; g.rowadd_mul = (c->n_img == 1 ? 0 : 1);
    g.c = c->pre1; g.ldc = c->NA; g.M = rows; g.N = c->NA;
    g.zero_acc = io.zero_state;           // [h2 | h1] = 0 at t = 0: pre1 = U[caption] + X[bos], no main loop
    g.pdl = c->use_pdl && (c->pdl_mode & 1); g.pdl_flags = ((c->pdl_mode & 4) ? 1 : 0) | ((c->pdl_mode & 8) ? 2 : 0);
    g.allow_pair = true;
    // GEMM-A runs on the CTA-pair kernel at EVERY row count (its 32 N tiles fill the machine from 2 row tiles on, and
    // below that the pair splits the weight stream over two SMs: faster than the single-CTA kernel at 100, 500 and 5000
    // rows alike), with the residual passes in fp8.  One kernel and one operand mode at every batch size keeps a
    // caption's result independent of what else is in the batch.  (On the single-CTA kernel its 192-wide tile only fits
    // 32-element k-blocks, whose 32-byte e4m3 rows load poorly: that path keeps three fp16 passes, VSRDEC_PAIR=0.)
    g.f8 = c->gemm_f8 && c->use_pair; g.pair_min_rows = 1;
    fused = gemm_uses_tc(c, g);
    c->state_h32 = !fused || io.need_h32;
    if (fused) {   // LSTM cell 1 + sentinel gate in the epilogue: pre1 is never written
      // fp32 copies of h1', s_t (and g_t, att, h2' below) feed only the FFMA twin and vsr_step's outputs: the
      // tensor-core GEMMs read the fp16 hi/lo twins, so those stores (and their reorder copies) are skipped
      g.cell.mode = 1; g.cell.c_old = c->c1; g.cell.c_new = c->c1n; g.cell.h_new = io.need_h32 ? c->h1n : nullptr;
      g.cell.h_b = &c->h1n_b;
      g.cell.s_new = nullptr; g.cell.s_b = &c->s_t_b;
      g.cell.gq = c->gq; g.cell.ld_state = c->Hp;
    }
    VSR_TRY(launch_gemm(c, g, st)); c->launches++;
  }
  if (!fused) {
    PhaseScope ps(c, PH_LSTM1, st);
    k_lstm1<<<pw_grid, 128, 0, st>>>(c->pre1, c->NA, c->c1, c->h1n, c->c1n, c->s_t, c->gq, pair_out(c, c->h1n_b),
                                     pair_out(c, c->s_t_b), c->Hp, H, rows);
    VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  }
  {  // B: [sentinel | sa] = WB1 . s_t + b ;  [hg | ha] = WB2 . h1'
    PhaseScope ps(c, PH_GEMM_B, st);
    GemmArgs g{};
    g.nseg = 1; g.seg[0] = {c->s_t, c->Hp, c->Hp, c->Hp, &c->s_t_b};
    g.w = c->WB1; g.ldw = c->Hp; g.bias = c->bB1; g.wb = &c->WB1_b;
    g.c = c->sent; g.ldc = c->NB1; g.M = rows; g.N = c->NB1;
    GemmArgs g2{};
    g2.nseg = 1; g2.seg[0] = {c->h1n, c->Hp, c->Hp, c->Hp, &c->h1n_b};
    g2.w = c->WB2; g2.ldw = c->Hp; g2.wb = &c->WB2_b; g2.f8 = c->gemm_f8; g2.allow_pair = true; g2.pair_min_rows = c->pair_min_rows;
    g2.c = c->hb; g2.ldc = c->NB2; g2.M = rows; g2.N = c->NB2;
    if (fused) {   // g_t = sig(gq + W1_hg.h1') * tanh(c1') on the hg column block of the h1' projection
      g2.cell.gt_cols = c->oB2_ha; g2.cell.gt_gq = c->gq; g2.cell.gt_c1n = c->c1n; g2.cell.g_t = nullptr;
      g2.cell.g_b = &c->g_t_b; g2.cell.ld_state = c->Hp;
    }
    g.pdl = c->use_pdl && (c->pdl_mode & 1); g.pdl_flags = ((c->pdl_mode & 4) ? 1 : 0) | ((c->pdl_mode & 8) ? 2 : 0);
    g.f8 = c->gemm_f8; g.allow_pair = true; g.pair_min_rows = c->pair_min_rows;
    VSR_TRY(launch_gemm(c, g, st, &g2)); c->launches += fused ? 1 : 2;   // one grouped launch on tensor cores
  }
  if (!fused) {
    PhaseScope ps(c, PH_GT, st);
    k_gt<<<pw_grid, 128, 0, st>>>(c->gq, c->hb, c->NB2, c->c1n, c->g_t, pair_out(c, c->g_t_b), c->Hp, H, rows);
    VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  }
  {
    PhaseScope ps(c, PH_ATTEND, st);
    AttendArgs a{};
    a.det_seqs = c->det_seqs; a.feat_dtype = c->feat_dtype; a.P = c->P; a.slot_mask = c->slot_mask; a.ptr = c->ptr;
    a.slot_base = c->p_compact ? c->slot_base : nullptr;
    a.slot_index = c->slot_index; a.det = c->det; a.det_stride = c->det_stride; a.D = c->D;
    a.img = c->img; a.ld_img = c->Fp; a.Pmean = c->Pmean; a.img_mul = (c->n_img == 1 ? 0 : 1);
    a.sent = c->sent; a.ld_sent = c->NB1; a.o_sa = c->oB1_sa;
    a.hb = c->hb; a.ld_hb = c->NB2; a.o_ha = c->oB2_ha;
    a.v_a = c->v_a; a.v_s = c->v_s;
    a.att = fused ? nullptr : c->att; a.ld_att = c->Fp; a.att_b = pair_out(c, c->att_b); a.shift = c->shift;
    a.rows = rows; a.cur_beam = io.cur_beam; a.L = c->L; a.R = c->R; a.F = c->F; a.A = c->A; a.H = H;
    a.ldP = c->NVA;
    a.alpha_out = io.attn_alpha; a.slot_out = io.attn_slot;
    const size_t smem = sizeof(float) * ((size_t)c->A + (size_t)c->R * c->A + c->R + 1);
    void (*const kern[3])(const AttendArgs) = {k_attend<float>, k_attend<__half>, k_attend<__nv_bfloat16>};
    if (!c->attend_attr_set) {     // per device, hence per handle
      for (auto k : kern) VSR_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      c->attend_attr_set = true;
    }
    VSR_REQUIRE(smem <= 200 * 1024, VSR_EINVAL, "attention tile (R=%d x A=%d) does not fit shared memory", c->R, c->A);
    const int ki = c->feat_dtype == VSR_DT_F16 ? 1 : c->feat_dtype == VSR_DT_BF16 ? 2 : 0;
    VSR_CHECK_CUDA(launch_k(kern[ki], dim3(rows), dim3(ATT_THREADS), smem, st, c->use_pdl && (c->pdl_mode & 2), a));
    VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  }
  {  // D: pre2 = WD . [att | h2_old | h1'] + b (+ U2[img]);  C: ga = att_ga . g_t rides in the same launch
     // (the stay-gate logit that needs ga is finished in k_softmax_topk, off the attention's critical path)
    PhaseScope ps(c, PH_GEMM_D, st);
    GemmArgs gc{};
    gc.nseg = 1; gc.seg[0] = {c->g_t, c->Hp, c->Hp, c->Hp, &c->g_t_b};
    gc.w = c->WC; gc.ldw = c->Hp; gc.wb = &c->WC_b; gc.f8 = c->gemm_f8; gc.allow_pair = true; gc.pair_min_rows = c->pair_min_rows;
    gc.c = c->ga; gc.ldc = c->NC; gc.M = rows; gc.N = c->NC;
    GemmArgs g{};
    g.nseg = io.zero_state ? 2 : 3;       // h2 = 0 at t = 0: its K segment (last in WD) is not read
    g.seg[0] = {c->att, c->Fp, c->Fp, c->Fp, &c->att_b};
    g.seg[1] = {c->h1n, c->Hp, c->Hp, c->Hp, &c->h1n_b};
    g.seg[2] = {c->h2, c->Hp, c->Hp, c->Hp, &c->h2_b};
    g.w = c->WD; g.ldw = c->KD; g.bias = c->bD; g.wb = &c->WD_b;
    if (c->d.img_second_lstm) {
      g.rowadd = c->U2; g.ld_rowadd = c->ND; g.row_div = io.cur_beam; g.rowadd_mul = (c->n_img == 1 ? 0 : 1);
    }
    g.c = c->pre2; g.ldc = c->ND; g.M = rows; g.N = c->ND;
    if (fused) {   // LSTM cell 2 in the epilogue
      g.cell.mode = 2; g.cell.c_old = c->c2; g.cell.c_new = c->c2n; g.cell.h_new = io.need_h32 ? c->h2n : nullptr;
      g.cell.h_b = &c->h2n_b; g.cell.ld_state = c->Hp;
    }
    g.pdl = c->use_pdl && (c->pdl_mode & 1); g.pdl_flags = ((c->pdl_mode & 4) ? 1 : 0) | ((c->pdl_mode & 8) ? 2 : 0);
    g.f8 = c->gemm_f8; g.allow_pair = true; g.pair_min_rows = c->pair_min_rows;
    VSR_TRY(launch_gemm(c, g, st, &gc)); c->launches += fused ? 1 : 2;
  }
  if (!fused) {
    PhaseScope ps(c, PH_LSTM2, st);
    k_lstm2<<<pw_grid, 128, 0, st>>>(c->pre2, c->ND, c->c2, c->h2n, c->c2n, pair_out(c, c->h2n_b), c->Hp, H, rows);
    VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  }
  if (io.skip_vocab) return VSR_OK;     // batched forward: the vocabulary projection of all steps runs after the loop
  // Fused vocabulary head (tensor-core path, nobody needs full log-prob rows): the GEMM epilogue also reduces
  // every tile to a softmax record and k_vocab_merge finishes the row without scanning the logits.
  static const bool fuse_enabled = [] { const char* e = getenv("VSRDEC_FUSE_VOCAB"); return e == nullptr || atoi(e) != 0; }();
  const bool fuse_vocab = fuse_enabled && fused && io.out_logp == nullptr && io.topk > 0;
  {  // E: logits = out_fc . h2' + b
    PhaseScope ps(c, PH_GEMM_E, st);
    GemmArgs g{};
    g.nseg = 1; g.seg[0] = {c->h2n, c->Hp, c->Hp, c->Hp, &c->h2n_b};
    g.w = c->WE; g.ldw = c->Hp; g.bias = c->bE; g.wb = &c->WE_b;
    g.c = c->logits; g.ldc = c->NE; g.M = rows; g.N = c->NE;
    g.pdl = c->use_pdl && (c->pdl_mode & 1); g.pdl_flags = ((c->pdl_mode & 4) ? 1 : 0) | ((c->pdl_mode & 8) ? 2 : 0);
    g.f8 = c->gemm_f8; g.allow_pair = true; g.pair_min_rows = c->pair_min_rows;
    if (fuse_vocab) {
      g.cell.mode = 3; g.cell.vocab_part = c->vpart;
    }
    VSR_TRY(launch_gemm(c, g, st)); c->launches++;
  }
  {
    PhaseScope ps(c, PH_SOFTMAX_TOPK, st);
    SoftmaxArgs a = make_softmax_args(c, rows, io.cur_beam, io.topk, io.use_verbs, io.gt);
    a.out_logp = io.out_logp; a.out_stride = io.out_stride;
    a.gate_out = io.gate_out; a.gate_stride = io.gate_stride;
    if (fuse_vocab) {
      VSR_CHECK_CUDA(launch_k(k_vocab_merge, dim3((rows + VM_WARPS - 1) / VM_WARPS), dim3(VM_WARPS * 32), 0, st, c->use_pdl && (c->pdl_mode & 2),
                              a, (const float*)c->vpart, c->NE / 16));
    } else {
      VSR_CHECK_CUDA(launch_k(k_softmax_topk, dim3(rows), dim3(SM_THREADS), 0, st, c->use_pdl && (c->pdl_mode & 2), a));
    }
    VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  }
  return VSR_OK;
}

}  // namespace vsr
