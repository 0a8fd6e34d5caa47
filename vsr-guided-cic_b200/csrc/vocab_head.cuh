// Device code shared by the kernels that finish the vocabulary head of a decoder step: log-softmax statistics, exact
// top-k word candidates, the shift-gate head and verb forcing for ONE row by ONE warp (merge_row), from the per-tile
// records the vocabulary GEMM's epilogue leaves (gemm_tc.cu: vocab_epilogue).
// Reference math: models/controllable_captioning.py:178 (out_fc + log_softmax), :184-188 (gate head), :271-295 (verb forcing).
#pragma once
#include <math.h>

#include "common.cuh"

namespace vsr {
namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ int64_t load_verb(const void* verbs, int dtype, size_t i) {
  if (dtype == VSR_DT_F64) return (int64_t) reinterpret_cast<const double*>(verbs)[i];
  if (dtype == VSR_DT_F32) return (int64_t) reinterpret_cast<const float*>(verbs)[i];
  return reinterpret_cast<const int64_t*>(verbs)[i];
}

// (value desc, index asc) total order: is (v1,i1) before (v2,i2)?
__device__ __forceinline__ bool before(float v1, int i1, float v2, int i2) {
  return v1 > v2 || (v1 == v2 && i1 < i2);
}
__device__ __forceinline__ void warp_argbest(float& bv, int& bi) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (before(ov, oi, bv, bi)) { bv = ov; bi = oi; }
  }
}
__device__ __forceinline__ unsigned orderable(float v) {     // monotone float -> unsigned
  const unsigned u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// warp arg-best in (value desc, index asc) order with two redux.sync; every lane gets the winner
__device__ __forceinline__ void warp_argbest_redux(float v, int i, unsigned& kbest, int& ibest) {
  const unsigned key = orderable(v);
  kbest = __reduce_max_sync(0xffffffffu, key);
  ibest = (int)__reduce_min_sync(0xffffffffu, key == kbest ? (unsigned)i : 0xffffffffu);
}

// n-gram blocking (vsr_set_no_repeat_ngram).  h = a row's emitted words y_0 .. y_{t-1}; with block size N the word
// y_{i+N-1} is banned at step t for every start 0 <= i <= t - N with y_i .. y_{i+N-2} == y_{t-N+1} .. y_{t-1}.  f(w) is
// called once per matching start (a word may come up more than once); the caller's threads split the starts as
// first, first + stride, ...  Every consumer of the ban (merge_row, k_softmax_topk, k_sample_pick) goes through here.
template <typename F>
__device__ __forceinline__ void for_each_banned(const int32_t* h, int t, int N, int first, int stride, F&& f) {
  for (int i = first; i <= t - N; i += stride) {
    bool match = true;
    for (int q = 0; q < N - 1 && match; ++q) match = h[i + q] == h[t - N + 1 + q];
    if (match) f((int)h[i + N - 1]);
  }
}
// shared-memory bitmap of the banned words of a row for one CTA (bit w of word w >> 5), vocabularies up to 49152
constexpr int BAN_WORDS = 49152 / 32;
__device__ __forceinline__ void build_ban_bitmap(unsigned* bits, const int32_t* h, int t, int N, int V) {
  for (int i = threadIdx.x; i < (V + 31) >> 5; i += blockDim.x) bits[i] = 0u;
  __syncthreads();
  for_each_banned(h, t, N, threadIdx.x, blockDim.x, [&](int w) { atomicOr(&bits[w >> 5], 1u << (w & 31)); });
  __syncthreads();
}

struct SoftmaxArgs {
  const float* logits; int ld;   // [rows][ld]
  int rows, V, cur_beam, L, topk;
  // n-gram blocking: whist [rows][whist_ld] = the rows' words of steps 0 .. hist_t - 1, block size ngram; null = off
  const int32_t* whist; int whist_ld, hist_t, ngram;
  const int32_t* ptr;
  const void* verbs; int verbs_dtype; int use_verbs, gt;
  const int64_t* vt_keys; const int32_t* vt_off; const int32_t* vt_idx; int vt_n;
  // gate head inputs
  const float* ha; int ld_ha;     // [rows] att_ha . h1'   (A wide)
  const float* ga; int ld_ga;     // [rows] att_ga . g_t
  const float* v_g; int A;
  const float* shift;             // [rows] sum of the valid region scores (from the attention kernel)
  float* row_max; float* row_lsum; int32_t* forced; int32_t* cand;  // cand [rows][VSR_MAX_BEAM]
  float* gate_lp;                 // [rows][2] post-forcing gate log-probs
  float* out_logp; int64_t out_stride;   // optional full rows
  float* gate_out; int64_t gate_stride;  // optional copy of the gate rows
};

// host: the arguments of the head kernels for one step
inline SoftmaxArgs make_softmax_args(const Ctx* c, int rows, int cur_beam, int topk, bool use_verbs, bool gt) {
  SoftmaxArgs a{};
  a.logits = c->logits; a.ld = c->NE; a.rows = rows; a.V = c->V; a.cur_beam = cur_beam; a.L = c->L;
  a.topk = topk; a.ptr = c->ptr;
  a.verbs = c->verbs; a.verbs_dtype = c->verbs_dtype; a.use_verbs = use_verbs; a.gt = gt;
  a.vt_keys = c->vt_keys; a.vt_off = c->vt_off; a.vt_idx = c->vt_idx; a.vt_n = c->vt_n;
  a.ha = c->hb + c->oB2_ha; a.ld_ha = c->NB2; a.ga = c->ga; a.ld_ga = c->NC; a.v_g = c->v_g; a.A = c->A;
  a.shift = c->shift;
  a.row_max = c->row_max; a.row_lsum = c->row_lsum; a.forced = c->forced; a.cand = c->cand;
  a.gate_lp = c->gate_lp;
  return a;
}

// which vocabulary index does verb id `verb` force (:271-295)?  x = the row's logits, (mx, lsum) its softmax statistics
__device__ __forceinline__ int forced_word(const SoftmaxArgs& a, int64_t verb, const float* x, float mx, float lsum) {
  if (verb == -1) return -1;
  const int V = a.V;
  int forced;
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
  return min(max(forced, 0), V - 1);
}

// What one warp knows about its row when merge_row returns (every lane holds the scalars; lane j < topk holds the
// j-th best word candidate in `pick`, with its raw logit in `pick_logit` unless the row is verb-forced).
struct RowHead {
  float mx, lsum;       // row max and log(sum exp(x - max)) of the logits
  int forced;           // forced vocabulary index or -1
  float g0, g1;         // post-forcing gate log-probs (stay, shift)
  int pick;             // lane j: j-th candidate (forced row: forced word first, then the lowest other indices)
  float pick_logit;     // lane j: logit of pick (unforced rows)
};

// The vocabulary GEMM's epilogue leaves one record {max, sum exp(x - max)} per (row, 16-column chunk).  One WARP per
// row: row max / log-sum-exp from the records (lanes stride the chunks, so the summation order depends on nothing but
// the vocabulary size); then the topk chunks by (max desc, position asc), whose topk * 16 logits are re-read, and the
// topk elements among them.
// Exact: if an element e of chunk C were in the row's top-k without C being among the topk chunks in that order, each
// of the topk chunks ahead of C would hold an element ordered before e (larger, or equal with a smaller index).
// Composite keys orderable(value) : ~position make "ordered before" a plain unsigned 64-bit '>'.  The chunk maxima stay
// in registers across the topk rounds when the row has at most 32 * VM_CPL chunks (V <= 12288), else they are re-read.
// N-gram blocking (a.whist): the log-sum-exp still comes from the unchanged records.  Then every chunk that holds a
// banned word gets the max of its words that are not banned, from its 16 re-read logits, written over the record's max
// (-inf when all of them are banned: the chunk drops out), and both rounds run as above with banned words skipped.  The
// argument above carries over unchanged with "element" read as "word that is not banned": each chunk's key is then
// the max of exactly those words.
constexpr int VM_CPL = 24;

// bits e of the banned words C * 16 + e of chunk C
__device__ __forceinline__ unsigned chunk_ban_mask(const int32_t* h, int t, int N, int C) {
  unsigned m = 0u;
  for_each_banned(h, t, N, 0, 1, [&](int w) { if ((w >> 4) == C) m |= 1u << (w & 15); });
  return m;
}

__device__ __forceinline__ void merge_row(const SoftmaxArgs& a, float* vpart, int n_chunks, int n, int lane,
                                          RowHead& out) {
  const int V = a.V, topk = a.topk;
  float2* rec = reinterpret_cast<float2*>(vpart) + (size_t)n * n_chunks;
  const float* x = a.logits + (size_t)n * a.ld;
  const int used = (V + 15) >> 4;               // chunks that hold vocabulary entries

  int64_t verb = -1; float shift_logit = 0.f;
  if (lane == 0) {
    shift_logit = a.shift[n];
    if (a.use_verbs && a.verbs != nullptr)
      verb = load_verb(a.verbs, a.verbs_dtype, (size_t)(n / a.cur_beam) * a.L + a.ptr[n]);
  }
  const bool in_regs = used <= 32 * VM_CPL;
  float cmx[VM_CPL];
  float m = -INFINITY, ssum = 0.f;
  if (in_regs) {
    float2 ms[VM_CPL];
#pragma unroll
    for (int q = 0; q < VM_CPL; ++q) {
      const int t = lane + 32 * q;
      ms[q] = t < used ? rec[t] : make_float2(-INFINITY, 0.f);
    }
#pragma unroll
    for (int q = 0; q < VM_CPL; ++q) {
      cmx[q] = ms[q].x;
      if (ms[q].x > m) { ssum *= __expf(m - ms[q].x); m = ms[q].x; }
      if (ms[q].x > -INFINITY) ssum += ms[q].y * __expf(ms[q].x - m);
    }
  } else {
    for (int t = lane; t < used; t += 32) {
      const float2 r2 = rec[t];
      if (r2.x > m) { ssum *= __expf(m - r2.x); m = r2.x; }
      if (r2.x > -INFINITY) ssum += r2.y * __expf(r2.x - m);
    }
  }
  // stay-gate logit att_g . tanh(ga + ha)
  float stay = 0.f;
  {
    const float4* ha = reinterpret_cast<const float4*>(a.ha + (size_t)n * a.ld_ha);
    const float4* ga = reinterpret_cast<const float4*>(a.ga + (size_t)n * a.ld_ga);
    const float4* vg = reinterpret_cast<const float4*>(a.v_g);
    for (int i = lane; i < a.A / 4; i += 32) {
      const float4 h = ha[i], g = ga[i], w = __ldg(vg + i);
      stay += (w.x * fast_tanh(g.x + h.x) + w.y * fast_tanh(g.y + h.y)) + (w.z * fast_tanh(g.z + h.z) + w.w * fast_tanh(g.w + h.w));
    }
  }
  const float mx = warp_max(m);
  const float se = warp_sum(m > -INFINITY ? ssum * expf(m - mx) : 0.f);
  const float lsum = logf(se);
  stay = warp_sum(stay);

  const bool ban = a.whist != nullptr && a.hist_t >= a.ngram;   // warp-uniform
  const int32_t* hrow = ban ? a.whist + (size_t)n * a.whist_ld : nullptr;
  if (ban) {
    __syncwarp();                                 // every lane has read its records
    for_each_banned(hrow, a.hist_t, a.ngram, lane, 32, [&](int w) {
      const int C = w >> 4;
      const unsigned m = chunk_ban_mask(hrow, a.hist_t, a.ngram, C);
      float cm = -INFINITY;
      for (int e = 0; e < 16; ++e)
        if (!((m >> e) & 1u) && C * 16 + e < V) cm = fmaxf(cm, x[C * 16 + e]);
      rec[C].x = cm;                              // (lanes that hit the same chunk write the same value)
    });
    __syncwarp();
    if (in_regs) {
#pragma unroll
      for (int q = 0; q < VM_CPL; ++q) {
        const int t = lane + 32 * q;
        if (t < used) cmx[q] = rec[t].x;
      }
    }
  }

  //   1. the topk CHUNKS by chunk max (round j: every lane's best key strictly below the previous winner, then a warp
  //      arg-best; lane j keeps winner j)
  unsigned long long prev = ~0ull;
  int my_chunk = -1;
  for (int j = 0; j < topk; ++j) {
    unsigned long long best = 0ull;
    if (in_regs) {
#pragma unroll
      for (int q = 0; q < VM_CPL; ++q) {
        const int t = lane + 32 * q;
        const unsigned long long key = ((unsigned long long)orderable(cmx[q]) << 32) | (unsigned)(~(unsigned)t);
        if (cmx[q] > -INFINITY && key < prev && key > best) best = key;
      }
    } else {
      for (int t = lane; t < used; t += 32) {
        const float cm = rec[t].x;
        const unsigned long long key = ((unsigned long long)orderable(cm) << 32) | (unsigned)(~(unsigned)t);
        if (cm > -INFINITY && key < prev && key > best) best = key;
      }
    }
    const unsigned hi = __reduce_max_sync(0xffffffffu, (unsigned)(best >> 32));
    const unsigned lo = __reduce_max_sync(0xffffffffu, (unsigned)(best >> 32) == hi ? (unsigned)best : 0u);
    prev = ((unsigned long long)hi << 32) | lo;
    if (hi == 0u && lo == 0u) break;          // fewer chunks than topk (uniform)
    if (lane == j) my_chunk = (int)(~lo);
  }
  //   2. the topk ELEMENTS among those chunks' logits: lane owns elements e = lane + 32 * q of the topk * 16
  constexpr int EQ = VSR_MAX_BEAM * 16 / 32;
  float cv[EQ]; int ci[EQ];
  const unsigned my_mask = (ban && my_chunk >= 0) ? chunk_ban_mask(hrow, a.hist_t, a.ngram, my_chunk) : 0u;
#pragma unroll
  for (int q = 0; q < EQ; ++q) {
    const int e = lane + 32 * q;
    const int chunk = __shfl_sync(0xffffffffu, my_chunk, (e >> 4) & 31);
    const unsigned cmask = ban ? __shfl_sync(0xffffffffu, my_mask, (e >> 4) & 31) : 0u;
    cv[q] = -INFINITY; ci[q] = 0x7fffffff;
    if (e < topk * 16 && chunk >= 0 && !((cmask >> (e & 15)) & 1u)) {
      const int col = chunk * 16 + (e & 15);
      if (col < V) { cv[q] = x[col]; ci[q] = col; }
    }
  }
  int my_pick = 0x7fffffff; float my_logit = -INFINITY;
  for (int j = 0; j < topk; ++j) {
    float bv = -INFINITY; int bi = 0x7fffffff;
#pragma unroll
    for (int q = 0; q < EQ; ++q) if (before(cv[q], ci[q], bv, bi)) { bv = cv[q]; bi = ci[q]; }
    unsigned kb; int ib;
    warp_argbest_redux(bv, bi, kb, ib);
    const float wv = __shfl_sync(0xffffffffu, bv, __ffs(__ballot_sync(0xffffffffu, bi == ib)) - 1);
#pragma unroll
    for (int q = 0; q < EQ; ++q) if (ci[q] == ib) { cv[q] = -INFINITY; ci[q] = 0x7fffffff; }
    if (lane == j) { my_pick = ib; my_logit = wv; }
  }

  int forced = -1;
  float g0 = 0.f, g1 = 0.f;
  if (lane == 0) {
    forced = forced_word(a, verb, x, mx, lsum);
    // gate head: log_softmax([stay, shift]) (:187-188), or [-1e3, 0] on a verb slot (:295)
    if (forced >= 0) { g0 = -1e3f; g1 = 0.f; }
    else {
      const float gm = fmaxf(stay, shift_logit);
      const float ls = logf(expf(stay - gm) + expf(shift_logit - gm));
      g0 = (stay - gm) - ls; g1 = (shift_logit - gm) - ls;
    }
  }
  forced = __shfl_sync(0xffffffffu, forced, 0);
  g0 = __shfl_sync(0xffffffffu, g0, 0);
  g1 = __shfl_sync(0xffffffffu, g1, 0);
  if (forced >= 0 && lane < topk) {
    // forced word first, then the lowest other indices (all tied at -1e6)
    int w = forced;
    if (lane > 0) { w = lane - 1; if (w >= forced) ++w; w = min(w, V - 1); }
    my_pick = w;
  }
  out.mx = mx; out.lsum = lsum; out.forced = forced; out.g0 = g0; out.g1 = g1; out.pick = my_pick; out.pick_logit = my_logit;
}

}  // namespace
}  // namespace vsr
